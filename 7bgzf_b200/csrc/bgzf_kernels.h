/* bgzf_kernels.h — internal launch interface between the C-ABI shim (b200bgzf_api.cu) and the kernels. */
#ifndef BGZF_KERNELS_H
#define BGZF_KERNELS_H
#include <cuda_runtime.h>
#include <stdint.h>

#include "bgzf_block.h"

#define BGZF_SCRATCH_WORDS (65536u + 32u + 16384u + 32u)   /* per-CTA scratch: u32 match per position + u8 build notes */
#define BGZF_SPLIT_EXTRA_WORDS 32768u                       /* split launch: the chain links of every tile, exchanged between the CTAs */
#define BGZF_SPLIT_MAX 8                                    /* largest cluster bgzf_launch_compress_split takes */
#define BGZF_PROF_SLOTS 288                                 /* 32 phase counters, then per tile of the chain build: relay turn, ready flag */
#define BGZF_PROF_TURN 32
#define BGZF_PROF_READY 160

struct BgzfCompressArgs {
    const uint8_t *in;         /* device: payload bytes */
    const uint64_t *in_off;    /* device: per-block byte offset into `in`, or NULL for fixed-size blocks */
    const uint32_t *in_len;    /* device: per-block length (with in_off) */
    uint64_t in_bytes;         /* fixed-size mode: total bytes */
    uint32_t block_size;       /* fixed-size mode: payload bytes per block (<= 65536) */
    uint32_t nblocks;
    uint32_t hdr_bytes;        /* 0 or 18: BGZF members; 20: MiGz members (same DEFLATE data, other gzip subfield) */
    BgParams prm;              /* search effort, from bg_level_params(level) on the host */
    uint8_t *slots;            /* device: nblocks * 65536 (+16) bytes */
    uint32_t *out_len;         /* device: member size per block (0 on failure) */
    uint32_t *status;          /* device: 0 ok, 1 member would exceed 65536 bytes */
    uint32_t *err_flag;        /* device: OR of all per-block status words */
    uint32_t *scratch;         /* device: grid * BGZF_SCRATCH_WORDS */
    uint32_t *cand;            /* device: grid * 4 * 65536 words (near-optimal levels), else NULL */
    const uint32_t *crctab;    /* device u32[256] */
    const uint32_t *crcpow;    /* device u32[1024] */
    unsigned long long *prof;  /* device u64[BGZF_PROF_SLOTS] cycle counters, or NULL */
    /* fused compaction (host-buffer batches): the last CTA to finish scans the member sizes and gathers the slots into one
     * stream itself, so that no small kernel has to find room among the resident compress CTAs */
    uint8_t *gather_out;       /* device: the batch's contiguous stream, or NULL (compaction by bgzf_launch_compact) */
    uint64_t *gather_off;      /* device u64[nblocks]: out: where every member starts in gather_out */
    uint64_t *gather_total;    /* device: in: bytes already in gather_out; out: bytes after this batch */
    uint32_t *done_count;      /* device: zero before the launch */
    /* piece mode (BgCtx.piece in bgzf_block.h): raw DEFLATE pieces for containers whose members span several blocks */
    uint32_t piece_mode;       /* 0: BGZF / MiGz members */
    uint32_t member_blocks;    /* pieces per member (>= 1); a member's last piece is the final DEFLATE block unless no_final */
    uint64_t piece_base;       /* index, in the whole stream, of this call's first piece */
    uint64_t piece_total;      /* pieces in the whole stream (its last piece ends a member whatever its index) */
    uint32_t head_gap;         /* free bytes before a member's first piece */
    uint32_t tail_gap;         /* free bytes after a member's last piece */
    uint32_t no_final;         /* 1: no piece is final (dictzip closes the member with an empty block of its own) */
    uint32_t *crc_out;         /* device u32[nblocks], optional: CRC-32 of every block's input */
    uint32_t history;          /* piece mode, fixed-size blocks: up to this many bytes (a multiple of 272, <= 32640; block_size + history
                                  <= 65536) right before a piece are loaded with it as match history (dictionary priming); a member's
                                  first piece has none */
    uint32_t lead;             /* bytes of the stream present in the device buffer before `in` (history of this launch's first blocks) */
};

struct BgzfInflateArgs {
    const uint8_t *in;         /* device: BGZF stream */
    const uint64_t *in_off;    /* device: byte offset of each member */
    const uint64_t *out_off;   /* device: byte offset of each member's payload in `out` */
    const uint32_t *hdr_len;   /* device, optional: offset of the DEFLATE data inside each member, as found by the host's header
                                  parser (any flavour of applet/7bgzf.c:81-131); NULL: strict BGZF headers, parsed by the kernel */
    const uint32_t *msize;     /* device, with hdr_len: whole member size */
    const uint32_t *unit_isize; /* device, optional (with hdr_len): 0xffffffff = a member (ISIZE from its trailer); anything else = a raw
                                  DEFLATE piece of msize bytes (hdr_len bytes skipped, no trailer) that yields this many bytes */
    uint32_t *unit_crc;        /* device, optional (verify_crc): out: CRC-32 of every unit's output (a piece has no trailer to check it against) */
    uint32_t nblocks;
    uint8_t *out;              /* device */
    uint32_t *status;          /* device: 0 ok, else error code per member */
    uint32_t *err_flag;        /* device: set to non-zero when any member fails */
    int verify_crc;            /* also run bgzf_verify_kernel: CRC-32 of every member's output against its trailer */
    const uint32_t *crctab;
    const uint32_t *crcpow;    /* device u32[1024] (verify) */
};

/* workspaces of the device-side member index (all device memory) */
struct BgzfIndexWork {
    uint32_t max_blocks;       /* capacity of the per-candidate / per-member arrays below */
    uint32_t *tile_count;      /* [tiles] signature hits per 32 KiB tile */
    uint64_t *tile_off;        /* [tiles] their exclusive scan */
    uint64_t *cand_off;        /* [max_blocks] offsets of all signature hits, ascending */
    uint32_t *jump, *jump2;    /* [max_blocks + 2] successor links of the candidates, squared in place (pointer doubling) */
    uint32_t *reach;           /* [max_blocks + 2] 1 = on the BSIZE chain from offset 0 */
    uint64_t *pick_idx;        /* [max_blocks] exclusive scan of reach[] */
    uint64_t *in_off;          /* [max_blocks] out: offset of every member */
    uint64_t *out_off;         /* [max_blocks] out: offset of every member's payload in the output */
    uint32_t *isize;           /* [max_blocks] out: ISIZE of every member */
    uint64_t *ncand, *nmembers, *out_bytes;   /* three consecutive u64 */
    uint32_t *status;          /* bit 0: not a BGZF stream, bit 1: more candidates than max_blocks */
};

/* random access (bgzf_ranges.cu): requested ranges -> touched members -> scratch -> caller's output */
#define BGZF_GATHER_TILE 32768u      /* bytes of one range copied by one gather CTA */

struct BgzfRangePlanArgs {
    const uint64_t *ranges;    /* device: [2 * nranges] beg, end (uncompressed offsets, or BGZF virtual offsets) */
    uint32_t nranges;
    int voffsets;
    uint64_t in_bytes;         /* stream size: a virtual offset may name it (uoffset 0) as the end */
    const uint64_t *in_off, *out_off;   /* device: the member index (bgzf_launch_index) */
    const uint32_t *isize;
    const uint64_t *nmembers, *total;   /* device: member count and decoded size */
    int32_t *diff;             /* device [nmembers + 1], zeroed: +1 at a range's first member, -1 after its last */
    uint32_t *first;           /* device [nranges] out: first member of every range */
    uint64_t *delta, *len;     /* device [nranges] out: offset of the range in its first member, length */
    uint32_t *status;          /* device: bit 0 set by a range that is out of bounds or names no member start */
};

struct BgzfRangeTouchArgs {
    uint32_t nmembers, nranges;
    const int32_t *diff;
    const uint64_t *in_off;    /* device [nmembers] */
    const uint32_t *isize;     /* device [nmembers] */
    uint64_t *t_in_off, *t_soff;   /* device [nmembers] out: the touched members' input offsets and scratch offsets, in order */
    uint64_t *m_soff;          /* device [nmembers] out: scratch offset of every touched member (by member number) */
    const uint32_t *first;
    const uint64_t *delta, *len;
    uint64_t *src, *range_off, *tile_off;   /* device [nranges] out: where a range starts in scratch / in the output; its first tile */
    uint64_t *counts;          /* device [4] out: touched members, scratch bytes, output bytes, gather tiles */
};

struct BgzfRangeGatherArgs {
    const uint8_t *scratch;    /* device: decoded bytes [win_lo, win_hi) of the scratch coordinates (+ 64 bytes of pad) */
    uint64_t win_lo, win_hi;
    uint8_t *out;              /* device */
    const uint64_t *src, *range_off, *len, *tile_off;   /* device [nranges] */
    uint32_t nranges;
};

/* whole-stream gzip (bgzf_gzip.cu): one member inflated in chunks cut at its byte-aligned flush points (all device memory) */
#define GZ_END_FLUSH 0u   /* ended right after a non-final empty stored block (searched route: at a block boundary at or after its stop) */
#define GZ_END_FINAL 1u   /* ended with the final block */
#define GZ_FAIL 2u        /* not a chunk a sequential decoder could produce without an error (or over the caps) */
struct BgzfGzipArgs {
    const uint8_t *data;       /* the member's DEFLATE data (after the header) */
    uint64_t data_len;         /* its bytes up to the 8-byte trailer */
    uint64_t max_in;           /* compressed bytes one chunk may span (a longer one ends the parallel attempt) */
    uint32_t *tile_count;      /* [tiles] candidates per 32 KiB tile */
    uint64_t *tile_off;        /* [tiles] their exclusive scan */
    uint64_t *counts;          /* [4]: candidates found by the scan, candidates (+ the data start), chained chunks, output bytes */
    const uint64_t *ncand, *nchunks;   /* counts + 1, counts + 2 */
    uint64_t *total;           /* counts + 3 */
    uint64_t *cand;            /* [ncand] candidate offsets in the DEFLATE data, ascending; cand[0] = 0 */
    uint64_t *end;             /* [ncand] where each candidate's chunk ends */
    uint32_t *olen, *status;   /* [ncand] its output bytes, how it ended */
    uint32_t *jump, *jump2, *reach;   /* [ncand + 2] successor links (pointer doubling) and the chain from candidate 0 */
    uint64_t *pick;            /* [ncand] exclusive scan of reach[] */
    uint32_t *chain_status;    /* bit 0: the chain from candidate 0 does not reach the end of the data */
    uint64_t *c_start;         /* [nchunks] the chained chunks: start in the DEFLATE data */
    uint32_t *c_len;           /* [nchunks] output bytes */
    uint64_t *c_off;           /* [nchunks] output offset in the member */
    uint32_t *lastm, *anchor;  /* [nchunks] one past the last marker a chunk wrote; 1 = its preceding 32 KiB hold no marker */
    uint16_t *scratch;         /* 32 KiB before the batch + the batch's output, one u16 per byte */
    uint8_t *out;              /* the member's output */
    uint32_t *err;             /* bit 0: a back-reference before the member start, bit 1: a chunk decoded differently */
};

/* random access through a gzip checkpoint index (bgzf_launch_gzip_runs): the batch's chunks lie in runs, each behind its window */
struct BgzfGzipRunArgs {
    uint32_t nchunks;          /* chunks of the batch (c_start, c_off, c_len of BgzfGzipArgs, from index 0) */
    const uint64_t *m_off;     /* [nchunks] each chunk's output offset in the member */
    uint32_t nwin;             /* windows to place */
    const uint8_t *win;        /* their bytes */
    const uint64_t *win_src;   /* [nwin] where window r starts in win */
    const uint32_t *win_len;   /* [nwin] its length (<= 32 KiB) */
    const uint64_t *win_dst;   /* [nwin] scratch offset of its 32 KiB slot (it is right-aligned there) */
};

#ifdef __cplusplus
extern "C" {
#endif
cudaError_t bgzf_launch_range_plan(const BgzfRangePlanArgs *a, cudaStream_t stream);
cudaError_t bgzf_launch_range_touch(const BgzfRangeTouchArgs *a, cudaStream_t stream);
cudaError_t bgzf_launch_range_gather(const BgzfRangeGatherArgs *a, uint64_t ntiles, cudaStream_t stream);
size_t bgzf_compress_smem_bytes(void);
cudaError_t bgzf_launch_compress(const BgzfCompressArgs *a, int grid, cudaStream_t stream);
cudaError_t bgzf_launch_compress_split(const BgzfCompressArgs *a, int csize, cudaStream_t stream);
cudaError_t bgzf_launch_scan(const uint32_t *len, uint64_t *off, uint32_t nmax, const uint64_t *count_dev,
                             const uint64_t *base_dev, uint64_t *total_out, cudaStream_t stream);
cudaError_t bgzf_launch_compact(const uint8_t *slots, const uint32_t *len, uint64_t *off, uint32_t nblocks, uint8_t *out,
                                uint64_t *total, int append_eof, cudaStream_t stream);
cudaError_t bgzf_launch_deliver(const uint8_t *slots, const uint32_t *len, const uint64_t *out_off, uint8_t *host_out, uint32_t n,
                                cudaStream_t stream);
size_t bgzf_index_tiles(uint64_t in_bytes);
size_t bgzf_gzip_tiles(uint64_t data_len);
size_t bgzf_gzip_window(void);
cudaError_t bgzf_launch_gzip_count(const BgzfGzipArgs *a, cudaStream_t stream);    /* counts[0] = flush points found */
cudaError_t bgzf_launch_gzip_chain(const BgzfGzipArgs *a, uint32_t ncand, cudaStream_t stream);
/* bit_end: NULL for flush-point chunks (c_start in bytes); else c_start and bit_end[j] are the bit offsets of the searched route */
cudaError_t bgzf_launch_gzip_batch(const BgzfGzipArgs *a, uint32_t j0, uint32_t j1, uint64_t base, uint64_t bytes,
                                   const uint64_t *bit_end, cudaStream_t stream);
/* members without flush points (DESIGN §6g): region size of the search (bytes); found[r - 1] = the proposed chunk start of
 * region r in bits (~0: none), r = 1 .. nreg - 1; the boundary pass over cand[0, n) (bits), each up to the first block
 * boundary at or after stop[k], into end (bits), olen and status */
size_t bgzf_gzip_region(void);
cudaError_t bgzf_launch_gzip_search(const BgzfGzipArgs *a, uint32_t nreg, uint64_t *found, cudaStream_t stream);
cudaError_t bgzf_launch_gzip_bit_bound(const BgzfGzipArgs *a, const uint64_t *stop, uint32_t n, cudaStream_t stream);
cudaError_t bgzf_launch_gzip_runs(const BgzfGzipArgs *a, const BgzfGzipRunArgs *r, uint64_t bytes, cudaStream_t stream);
#define BGZF_GZIP_CHAIN_LAUNCHES 8
#define BGZF_GZIP_BATCH_LAUNCHES 5
#define BGZF_INDEX_LAUNCHES 8
cudaError_t bgzf_launch_index(const uint8_t *in, uint64_t in_bytes, const BgzfIndexWork *w, cudaStream_t stream);
cudaError_t bgzf_launch_inflate(const BgzfInflateArgs *a, cudaStream_t stream);
cudaError_t bgzf_launch_verify(const BgzfInflateArgs *a, cudaStream_t stream);   /* bgzf_verify_kernel alone */
/* pointer doubling over successor links (bgzf_index_chain_kernel): reach[k] = 1 for every candidate on the chain from
 * candidate 0 (which must lie at offset 0); status bit 0 = the chain does not end at node `count` ("the end") */
cudaError_t bgzf_launch_chain(const uint64_t *cand_off, const uint64_t *count, uint32_t max_blocks, uint32_t *jump,
                              uint32_t *jump2, uint32_t *reach, uint32_t *status, cudaStream_t stream);
#ifdef __cplusplus
}
#endif
#endif
