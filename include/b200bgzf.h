/*
 * b200bgzf.h — C ABI of the B200-native BGZF codec (lib7bgzf_b200.so / 7bgzf.so).
 *
 * This is the drop-in boundary for the one hot path of cielavenir/7bgzf: per-64 KiB-block BGZF compress
 * (libdeflate level class 1..12) and BGZF inflate.  Plain pointers and sizes only; every entry point states
 * the reference interface it stands in for (paths relative to the reference tree).
 *
 * There is NO CPU fallback: every compress/inflate call runs the sm_100a kernels and fails with
 * B200BGZF_E_CUDA when no usable GPU (or the CUDA runtime) is present.
 */
#ifndef B200BGZF_H
#define B200BGZF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200BGZF_BLOCK_SIZE 0xff00u      /* htslib BGZF_BLOCK_SIZE; applet/7bgzf.c:146-147 */
#define B200BGZF_MAX_BLOCK_SIZE 0x10000u /* htslib BGZF_MAX_BLOCK_SIZE = largest member and largest payload */
#define B200BGZF_EOF_BYTES 28u           /* bgzf_compress.c:43-49 */

/* return codes.  0 and 1 and -1 keep the meaning they have in bgzf_compress.c:39-198 */
#define B200BGZF_OK 0
#define B200BGZF_E_NOFIT 1      /* a member would not fit its capacity (reference: "libdeflate_deflate 1", returns 1) */
#define B200BGZF_E_ARG (-1)     /* bad argument / capacity below the fixed minimum (reference returns -1) */
#define B200BGZF_E_CUDA (-2)    /* no device, out of device memory, launch failure */
#define B200BGZF_E_FORMAT (-3)  /* input is not BGZF / corrupt DEFLATE data */
#define B200BGZF_E_NOSPACE (-4) /* output buffer too small */
#define B200BGZF_E_CRC (-5)     /* CRC32 or ISIZE mismatch (only with B200BGZF_VERIFY) */

#define B200BGZF_APPEND_EOF 1u  /* compress: finish the stream with the 28-byte EOF member (applet/7bgzf.c:283-289) */
#define B200BGZF_VERIFY 2u      /* inflate: check CRC32 and ISIZE of every member (the reference does not: 7bgzf.c:350-354) */
#define B200BGZF_FRAME_MIGZ 4u  /* compress: MiGz members instead of BGZF ones — the same DEFLATE data behind the gzip subfield "MZ" with the
                                   compressed size as u32 (applet/7migz.c:133-243; SURVEY 8f rank 3).  No EOF marker exists in that
                                   container (B200BGZF_APPEND_EOF is ignored); block_size <= 64512 keeps every member inside its slot. */

typedef struct b200bgzf_ctx b200bgzf_ctx;

/* One context = one GPU, its streams, pinned staging and device workspaces.  device < 0: current device.
 * Replaces the per-call libdeflate_alloc_compressor/free of lib/zlibutil.c:186-188 with process-lifetime pools. */
int b200bgzf_create(b200bgzf_ctx **ctx, int device);
void b200bgzf_destroy(b200bgzf_ctx *ctx);
const char *b200bgzf_strerror(int code);
/* last CUDA error text seen by this context (empty string if none) */
const char *b200bgzf_last_error(const b200bgzf_ctx *ctx);

/* Worst-case size of the BGZF stream for in_bytes of payload cut into block_size blocks (+EOF). */
size_t b200bgzf_compress_bound(size_t in_bytes, uint32_t block_size);

/*
 * Compress a contiguous buffer into a contiguous BGZF stream; block b carries payload bytes
 * [b*block_size, min((b+1)*block_size, in_bytes)).  This is the applet's _compress() loop
 * (applet/7bgzf.c:133-293: read block, libdeflate_deflate, frame, write in order) as one batched call.
 *   *_device: d_in/d_out are device pointers (d_in 16-byte aligned for the TMA path), `stream` is a
 *             cudaStream_t passed as void* (NULL: the context's stream).  Synchronises before returning.
 *   *_host:   host pointers (pinned memory copies fastest); pipelined H2D / kernels / D2H.
 * level: 1..12 (libdeflate classes, lib/libdeflate/deflate_compress.c:3921-4007).
 */
int b200bgzf_compress_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, uint32_t block_size, int level,
                             void *d_out, size_t out_cap, size_t *out_bytes, unsigned flags, void *stream);
int b200bgzf_compress_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level, void *out,
                           size_t out_cap, size_t *out_bytes, unsigned flags);

/*
 * SURVEY §8(f) rank 2 — the index side-product.  Same as b200bgzf_compress_host, and also reports where every member
 * starts: member_off[b] = byte offset in `out` of the member that carries block b (member_cap >= number of blocks;
 * the EOF marker is not listed).  These are the offsets the device scan computes for the compaction anyway, copied
 * back with each batch.  Together with b*block_size they are the (compressed, uncompressed) address pairs of
 * htslib's .gzi index and the upper 48 bits of BAM virtual offsets.  The reference has no counterpart (its applet
 * writes no index: applet/7bgzf.c:133-293); the .gzi layout follows htslib's bgzf_index_dump (not in the reference
 * tree, so parity with htslib is unpinned — tests check the index against a header walk of the stream).
 */
int b200bgzf_compress_host_index(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level, void *out,
                                 size_t out_cap, size_t *out_bytes, unsigned flags, uint64_t *member_off, size_t member_cap);
/* Serialise a .gzi: u64 entry count, then (caddr, uaddr) for every member except the first (which is 0,0 by
 * definition), little endian.  Needs 8 + 16*(nmembers-1) bytes; returns the bytes written or 0 if cap is too small. */
size_t b200bgzf_gzi_format(const uint64_t *caddr, const uint64_t *uaddr, size_t nmembers, void *dst, size_t cap);

/*
 * Compress nblocks independent payloads (src[i], slen[i] <= 65536) into dst[i]; dlen[i] holds the capacity on
 * entry and the member size on return; status[i] gets the per-block code of bgzf_compress().  This is the
 * batch form of bgzf_compress.c:39-198.  nblocks == 1 is what the LD_PRELOAD hook calls for every htslib block:
 * that case takes a dedicated low-latency path (one copy in, one kernel, one copy out, one synchronisation) on
 * one of 128 independent lanes, so concurrent callers each drive their own stream; while few callers are in
 * flight the kernel of a call runs on a thread-block cluster of 8 (or 4) SMs that share the block's match search
 * (same output bytes, less than half the latency); callers beyond the host's core count wait by sleeping, not
 * spinning.
 */
int b200bgzf_compress_blocks_host(b200bgzf_ctx *ctx, const void *const *src, const uint32_t *slen, void *const *dst,
                                  size_t *dlen, int *status, uint32_t nblocks, int level);

/*
 * Inflate a BGZF stream (any sequence of BGZF members, EOF markers included) — the applet's _decompress()
 * (applet/7bgzf.c:295-365) with zlibutil_auto_inflate (lib/zlibutil.c:82-93) as the per-member decoder.
 * The *_size helper walks the member headers on the host (7bgzf.c:81-131) and returns the member count and the
 * total ISIZE so the caller can size the output.
 */
int b200bgzf_inflate_size_host(const void *in, size_t in_bytes, size_t *out_bytes, size_t *nmembers);
/* The member header parser of that loop (_read_gz_header, applet/7bgzf.c:81-131), every flavour it accepts: BGZF ("BC"),
 * MiGz ("MZ"), mgzip v1/v2 ("IG"), jerodsanto's mgzip; optional name / comment / header-CRC fields are skipped.  Returns
 * the header length (offset of the DEFLATE data) and stores the whole member size, or returns 0 if `p` does not start
 * such a member (or it is cut short by `avail`).  The *_host inflate entry points accept all of these; the
 * device-resident one, which finds members by their signature on the device, takes BGZF only. */
uint32_t b200bgzf_member_header(const void *p, size_t avail, uint64_t *member_bytes);
int b200bgzf_inflate_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, void *d_out, size_t out_cap,
                            size_t *out_bytes, unsigned flags, void *stream);
int b200bgzf_inflate_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, void *out, size_t out_cap, size_t *out_bytes,
                          unsigned flags);

/*
 * Random access (SURVEY §8(f) rank 2, the reading half of the index above): decode only the members that a list of byte
 * ranges needs.  No GPU involved in the two index helpers.
 *
 * b200bgzf_index_host walks the member headers (any flavour b200bgzf_member_header accepts) and lists the start of every
 * member, the EOF marker and other empty members included, as (compressed offset, uncompressed offset) pairs.
 * b200bgzf_gzi_parse reads a .gzi (the inverse of b200bgzf_gzi_format) and puts back the implicit (0, 0) first entry; it
 * refuses a file whose size does not match its entry count and entries that are not ascending (compressed offsets
 * strictly, uncompressed offsets never going down).  Both store min(count, cap) pairs and set *nmembers to the count;
 * with cap below the count (caddr / uaddr may then be NULL) they return B200BGZF_E_NOSPACE.
 */
#define B200BGZF_RANGE_VOFFSET 8u   /* ranges are [vbeg, vend) BGZF virtual offsets (coffset << 16 | uoffset), not uncompressed offsets */
typedef struct b200bgzf_range {
    uint64_t beg, end;
} b200bgzf_range;
int b200bgzf_index_host(const void *in, size_t in_bytes, uint64_t *caddr, uint64_t *uaddr, size_t cap, size_t *nmembers);
int b200bgzf_gzi_parse(const void *gzi, size_t gzi_bytes, uint64_t *caddr, uint64_t *uaddr, size_t cap, size_t *nmembers);

/*
 * Decode byte ranges of a stream.
 *   Output     the ranges' bytes back to back in the caller's order; range_off[i] (optional, nranges entries) = where range i
 *              starts in `out`, *out_bytes = the total.  out_cap too small (or out NULL with a non-empty result): returns
 *              B200BGZF_E_NOSPACE with *out_bytes = the size needed, before any member is decoded.
 *   Ranges     any order, may overlap, may be empty.  A member that several ranges touch is decoded once per call (the host
 *              variant cuts the call into groups of consecutive ranges of at most 256 MiB of decoded members + output each;
 *              a member shared by two groups is decoded by both).
 *   Offsets    uncompressed: beg <= end <= total decoded size, else B200BGZF_E_ARG.  B200BGZF_RANGE_VOFFSET: [vbeg, vend)
 *              virtual offsets as a .bai / .csi query returns its chunks; vbeg <= vend, coffset a member start (listed in
 *              the index when one is given) or in_bytes with uoffset 0 (the end), uoffset <= that member's ISIZE, else
 *              B200BGZF_E_ARG.  An empty member (the EOF marker) never starts a range.
 *   Index      host variant: caddr / uaddr (nindex entries, as b200bgzf_index_host or b200bgzf_gzi_parse give them) or NULL,
 *              and the index is then built by a header walk.  With an index, the call reads only the compressed bytes of
 *              the members it touches and the header and trailer of the last listed member (for the total size).
 *   Verify     B200BGZF_VERIFY checks the CRC-32 of every decoded member (B200BGZF_E_CRC).  A corrupt member that is
 *              touched gives B200BGZF_E_FORMAT; one that is not touched is never read.
 *   Formats    host: what b200bgzf_inflate_host accepts.  Device: BGZF only (like b200bgzf_inflate_device, whose device
 *              index it builds); the ranges and range_off are host arrays, d_in / d_out device memory, and the decoded
 *              members go through a scratch buffer of at most 1 GiB in the context (more touched members: several
 *              passes).  Synchronises before returning.
 * One member decodes on one warp in 4-5 ms; these calls are built for batches of ranges (thousands of members side by
 * side), not for the latency of one small query.
 */
int b200bgzf_inflate_ranges_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, const uint64_t *caddr, const uint64_t *uaddr,
                                 size_t nindex, const b200bgzf_range *ranges, size_t nranges, void *out, size_t out_cap,
                                 size_t *out_bytes, uint64_t *range_off, unsigned flags);
int b200bgzf_inflate_ranges_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, const b200bgzf_range *ranges, size_t nranges,
                                   void *d_out, size_t out_cap, size_t *out_bytes, uint64_t *range_off, unsigned flags, void *stream);

/*
 * Inflate a list of units found by the caller — what the readers of the indexed containers need (dictzip's chunk table,
 * RAZF's block index, GZinga's member index: applet/7dictzip.c:320-400, 7razf.c:293-384, 7gzinga.c:218-307).  A unit is either
 * a gzip member (piece = 0: hdr_len bytes of header, DEFLATE data, CRC32 + ISIZE; out_len is ignored, ISIZE counts) or a raw
 * DEFLATE piece (piece = 1: in_len bytes after hdr_len skipped bytes, no trailer) that is complete once it has produced
 * out_len bytes at a block boundary.  Units are listed in ascending input order; their outputs follow one another in `out`.
 * One warp decodes one unit, as for BGZF members.  B200BGZF_VERIFY checks the members against their trailers (members of
 * any size); unit_crc (optional, nunits entries) receives the CRC-32 of every unit's output — a piece carries none of its
 * own: the caller combines them (b200bgzf_crc32_combine) and compares with its container's member trailer.
 */
typedef struct b200bgzf_unit {
    uint64_t in_off;
    uint32_t in_len;
    uint32_t hdr_len;
    uint32_t out_len;
    uint32_t piece;
} b200bgzf_unit;
int b200bgzf_inflate_units_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, const b200bgzf_unit *units, size_t nunits,
                                void *out, size_t out_cap, size_t *out_bytes, unsigned flags, uint32_t *unit_crc);

/*
 * Several GPUs behind one call (SURVEY 8e; the reference's fan-out over blocks: applet/7bgzf.c:159-227).  GPU g of G takes
 * the contiguous block range [B*g/G, B*(g+1)/G) of the input (b200bgzf_shard_blocks), runs its own pipelined host-buffer
 * call on its own context and host thread, and the shard outputs are joined at host-known offsets: no collective, and the
 * stream is byte-identical for every G.  devices == NULL: ordinals 0..ndevices-1 (an ordinal may repeat: two contexts on
 * one GPU).  The output buffer must hold b200bgzf_multi_compress_bound() bytes (28 more per extra shard than the
 * single-GPU bound: every shard is placed behind the worst case of the ones before it, then moved down).
 */
typedef struct b200bgzf_multi b200bgzf_multi;
int b200bgzf_multi_create(b200bgzf_multi **m, const int *devices, int ndevices);
void b200bgzf_multi_destroy(b200bgzf_multi *m);
int b200bgzf_multi_count(const b200bgzf_multi *m);
b200bgzf_ctx *b200bgzf_multi_ctx(b200bgzf_multi *m, int i);
void b200bgzf_shard_blocks(uint64_t nblocks, int shard, int nshards, uint64_t *first, uint64_t *last);
size_t b200bgzf_multi_compress_bound(const b200bgzf_multi *m, size_t in_bytes, uint32_t block_size);
int b200bgzf_multi_compress_host(b200bgzf_multi *m, const void *in, size_t in_bytes, uint32_t block_size, int level, void *out,
                                 size_t out_cap, size_t *out_bytes, unsigned flags);
int b200bgzf_multi_inflate_host(b200bgzf_multi *m, const void *in, size_t in_bytes, void *out, size_t out_cap, size_t *out_bytes,
                                unsigned flags);

/*
 * SURVEY §8(f) ranks 3 and 4 — the other block-gzip containers and whole-stream gzip on the same kernel.
 *
 * Piece mode: block b of the input becomes a raw DEFLATE *piece* (no gzip framing).  Members are runs of
 * spec->member_blocks pieces; a member's last piece is the final DEFLATE block, every other piece has BFINAL = 0 and ends
 * with an empty stored block that pads to the byte — the "full flush" the reference applies to every dictzip / RAZF chunk
 * (applet/7dictzip.c:92-126, applet/7razf.c:124-160) — so the pieces of a member concatenate bytewise into one DEFLATE
 * stream, and each piece also decodes on its own.  head_gap / tail_gap zero bytes are left before a member's first and
 * after its last piece for the container's header and trailer.  Returns the pieces (with their gaps) back to back in
 * `out`, piece_off[b] = where piece b (or its head gap) starts, piece_crc[b] = CRC-32 of block b's input (combine them
 * with b200bgzf_crc32_combine).  With block_size + 5 + head_gap + tail_gap <= 65536 every piece fits its 64 KiB slot whatever
 * the data; beyond that (up to block_size 65536) a piece that does not compress makes the call return B200BGZF_E_NOFIT.
 */
#define B200BGZF_MAX_GAP 64u
#define B200BGZF_MAX_HISTORY 32640u
typedef struct b200bgzf_piece_spec {
    uint32_t member_blocks;   /* pieces per member, >= 1 (0xffffffff: one member) */
    uint32_t head_gap;        /* <= B200BGZF_MAX_GAP */
    uint32_t tail_gap;        /* <= B200BGZF_MAX_GAP */
    uint32_t no_final;        /* 1: no piece is final (dictzip closes its member with an empty block of its own) */
    uint64_t piece_base;      /* the call's input is a slice of a longer stream of pieces: index of its first piece, and the */
    uint64_t piece_total;     /* number of pieces of the whole stream (0: the input is the whole stream) — for sharding over GPUs */
    uint32_t history;         /* dictionary priming, as pigz does between its chunks: matches of a piece may reach up to this many
                                 bytes back into the input before it, inside its member (0: independent pieces; else a multiple
                                 of 272, at most B200BGZF_MAX_HISTORY, and block_size + history <= 65536).  Such pieces still end
                                 on a byte but no longer decode on their own.  With piece_base > 0 the `history` bytes before
                                 `in` must be readable: they are the end of the previous slice. */
    uint32_t reserved;
} b200bgzf_piece_spec;
size_t b200bgzf_pieces_gap_bytes(size_t in_bytes, uint32_t block_size, const b200bgzf_piece_spec *spec);
int b200bgzf_compress_pieces_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level,
                                  const b200bgzf_piece_spec *spec, void *out, size_t out_cap, size_t *out_bytes,
                                  uint64_t *piece_off, uint32_t *piece_crc, size_t piece_cap);
/* CRC-32 of A||B from CRC-32(A), CRC-32(B) and len(B) (zlib's crc32_combine, lib/zlib/crc32.c:1021-1026) */
uint32_t b200bgzf_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b);

/*
 * The containers (host code in 7bgzf_b200/host/containers.c; `param` = 0 for the reference's default):
 *   GZIP     one gzip member (applet/7gzip.c + zlibrawstdio_compress.h:259-300 hand the whole file to one
 *            libdeflate_deflate call; here: 48 KiB pieces primed with the 16 KiB before them, as pigz primes its chunks, or with
 *            B200BGZF_PARAM_INDEPENDENT independent 65280-byte pieces, as pigz -i does)
 *   MIGZ     applet/7migz.c:133-243 — members of `param` KiB (default 512), subfield "MZ" = DEFLATE size
 *   GZINGA   applet/7gzinga.c:78-216 — 100 KiB members with an empty comment, then an index member whose comment lists
 *            "n:end-offset;" of every member
 *   DICTZIP  applet/7dictzip.c:177-318 — chunks of `param` bytes (default 58315), subfield "RA" with every chunk's size,
 *            members of at most 32762 chunks, each closed by an empty static block
 *   RAZF     applet/7razf.c:160-290 — 32768-byte blocks, subfield "RAZF", block index (big endian) after the trailer;
 *            inputs below 4 GiB
 * b200bgzf_container_compress_host = plan + b200bgzf_compress_pieces_host + b200bgzf_container_frame.
 */
#define B200BGZF_PARAM_SAFE 0x80000000u   /* MiGz: or-ed into param: pieces of at most 65280 bytes (see b200bgzf_container_plan) */
#define B200BGZF_PARAM_PRIMED 0x40000000u      /* MiGz: 32 KiB pieces with dictionary priming inside every member (gzip: the default) */
#define B200BGZF_PARAM_INDEPENDENT 0x20000000u /* gzip: independent 65280-byte pieces, as pigz -i (twice the throughput, +1.6 ... 2.8 % size) */
#define B200BGZF_CONTAINER_GZIP 1
#define B200BGZF_CONTAINER_MIGZ 2
#define B200BGZF_CONTAINER_GZINGA 3
#define B200BGZF_CONTAINER_DICTZIP 4
#define B200BGZF_CONTAINER_RAZF 5
/* block size and piece layout of a container (dictzip: for a member of `npieces` chunks); 0 or B200BGZF_E_ARG */
int b200bgzf_container_plan(int kind, uint32_t param, uint32_t *block_size, b200bgzf_piece_spec *spec);
/* bytes of container header that precede the piece stream of a member and do not live in a gap (dictzip's chunk table) */
size_t b200bgzf_container_head(int kind, size_t npieces);
size_t b200bgzf_container_bound(int kind, uint32_t param, size_t in_bytes);
/* Writes the framing around a piece stream: `member` is where the container (dictzip: this member) starts, the stream of
 * `stream_bytes` bytes made with the plan above lies at member + b200bgzf_container_head().  No GPU involved.  Returns the
 * size of the finished container (member), 0 if `cap` is too small or an argument is off. */
size_t b200bgzf_container_frame(int kind, uint32_t param, void *member, size_t cap, size_t stream_bytes, const uint64_t *piece_off,
                                const uint32_t *piece_crc, size_t npieces, size_t in_bytes);
int b200bgzf_container_compress_host(b200bgzf_ctx *ctx, int kind, uint32_t param, const void *in, size_t in_bytes, int level,
                                     void *out, size_t out_cap, size_t *out_bytes);
/* The same over several GPUs (SURVEY 8e): pieces are independent, so GPU g takes a contiguous range of them (whole members
 * where a container has several), the shard streams are joined at host-known offsets and framed once; byte-identical to
 * the single-GPU container for every number of GPUs.  The output buffer must hold b200bgzf_multi_container_bound() bytes. */
size_t b200bgzf_multi_container_bound(const b200bgzf_multi *m, int kind, uint32_t param, size_t in_bytes);
int b200bgzf_multi_container_compress_host(b200bgzf_multi *m, int kind, uint32_t param, const void *in, size_t in_bytes, int level,
                                           void *out, size_t out_cap, size_t *out_bytes);

/* The readers: the unit list of a dictzip / RAZF / GZinga file from its own index (a plain gzip member without an index is
 * one unit: one warp decodes it), to be released with b200bgzf_units_free; out_bytes = the decoded size.  No GPU involved.
 * b200bgzf_container_inflate_host = that list + b200bgzf_inflate_units_host (MiGz: b200bgzf_inflate_host, whose header
 * walk knows the "MZ" subfield). */
int b200bgzf_container_units(int kind, const void *in, size_t in_bytes, b200bgzf_unit **units, size_t *nunits, size_t *out_bytes);
void b200bgzf_units_free(b200bgzf_unit *units);
int b200bgzf_container_inflate_host(b200bgzf_ctx *ctx, int kind, const void *in, size_t in_bytes, void *out, size_t out_cap,
                                    size_t *out_bytes, unsigned flags);   /* flags: 0 or B200BGZF_VERIFY (CRC-32 of every member) */
/* decoded size (and number of units) of a container, to size the output: MiGz — and gzip input that turns out to be a
 * stream of members carrying their own size (BGZF, MiGz, mgzip) — by the header walk, the others by their index */
int b200bgzf_container_inflate_size(int kind, const void *in, size_t in_bytes, size_t *out_bytes, size_t *nunits);

/* Page-locked host memory for the *_host entry points (pageable buffers work too, but are copied at a fraction of
 * the PCIe rate).  The applet reads stdin straight into such buffers. */
void *b200bgzf_host_alloc(size_t bytes);
void b200bgzf_host_free(void *p);

/* Per-phase cycle counters of the compress kernel (development aid; n <= 288: 32 phase counters, then per-tile
 * timings of the chain build, see tools/link_split.py). Resets them when reset != 0. */
int b200bgzf_profile(b200bgzf_ctx *ctx, int enable, unsigned long long *cycles, int n, int reset);
/* number of kernel launches issued by this context so far */
unsigned long long b200bgzf_launch_count(const b200bgzf_ctx *ctx);

/*
 * The htslib hook (exported from 7bgzf.so only).  Same signature and return conventions as the reference's
 * bgzf_compress.c:39: 0 ok; -1 if *dlen < 28 for slen == 0 or *dlen < 26; 1 (+ "libdeflate_deflate 1" on
 * stderr) when the member does not fit; `level` is ignored, BGZF_METHOD=<name><digits> selects the level.
 */
int bgzf_compress(void *dst, size_t *dlen, const void *src, size_t slen, int level);

/* BGZF_METHOD parser used by the hook (bgzf_compress.c:53-113).  Returns 0 and the level (1..12) to use,
 * or -1 if the digits are out of range.  Every method name maps onto this codec; unset/zlib -> 6. */
int b200bgzf_parse_method(const char *spec, int *level, char *method_name, size_t method_cap);

#ifdef __cplusplus
}
#endif
#endif
