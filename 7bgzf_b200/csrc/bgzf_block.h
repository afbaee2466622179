/*
 * bgzf_block.h — the per-BGZF-block DEFLATE encoder, written as per-thread *phase* functions.
 *
 * One CTA of BG_THREADS threads owns one BGZF block (<= 64 KiB) that sits in shared memory.  Every phase
 * below is a function of (context, thread index t, thread count T); the CUDA kernel (bgzf_compress.cu) calls
 * the phases with t = threadIdx.x and a __syncthreads() between them, and the development emulator
 * (tests/model/emul.cpp) calls the very same functions in a loop over t — in forward, reverse and shuffled
 * order, which doubles as a race detector: a phase may only read what an earlier phase wrote.
 * Warp-collective pieces (chain build, litlen key ranking, block scan, TMA load) live in the
 * .cu file and have plain sequential twins in the emulator; their results are order-independent by
 * construction, so GPU output == emulator output, byte for byte.
 *
 * What it replaces in the reference (the CPU hot path, re-designed, not translated):
 *   libdeflate_deflate_compress  lib/libdeflate/deflate_compress.c:4024-4066  (dispatcher, passthrough rule :4035)
 *   deflate_compress_lazy_generic :2605-2809 + hc_matchfinder.h:182-399  -> all-position chain search + local lazy rule
 *   choose_min_match_len :2295-2379                                      -> bg_min_match_len()
 *   deflate_make_huffman_code :1318-1396                                 -> bg_huff_lengths()/bg_huff_codes()
 *   deflate_precompute_huffman_header :1570-1631, compute_precode_items :1482-1557 -> bg_header_items()
 *   deflate_flush_block :1706-2038                                       -> bg_decide()/emit phases
 *   crc32 (hook) lib/zlib/crc32.c:1015, combine :155-186,1021-1026       -> bg_crc_* (per-thread slices + x^n combine)
 *   framing bgzf_compress.c:191-196                                      -> bg_emit_frame()
 *
 * The compressed bytes are NOT meant to equal libdeflate's (the search is all-position parallel, one dynamic
 * block per BGZF block); they must decode everywhere, CRC32/ISIZE must be exact and the size must stay
 * within 3 % of the reference at the matching level.
 */
#ifndef BGZF_BLOCK_H
#define BGZF_BLOCK_H

#include <stdint.h>
#include <stdio.h>

#if defined(__CUDACC__)
#define BG_HD __host__ __device__ __forceinline__
#else
#define BG_HD static inline
#endif
/* Bounds asserts of the checked build (`make checked`: -DBG_CHECK, build/checked/lib7bgzf_b200.so).  compute-sanitizer is not
 * available on the GPU pool, so the indices this round's code computes (bitmaps, queues, rings, scratch words, chunk order,
 * compaction offsets) are asserted in a separate build that the GPU tests can be pointed at (B200BGZF_LIB_PATH).  A failed
 * assert traps: the launch fails and the test with it. */
#if defined(BG_CHECK) && defined(__CUDA_ARCH__)
#define BG_ASSERT(cond) do { if (!(cond)) { printf("BG_ASSERT failed: %s (%s:%d) block %d thread %d\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, (int)threadIdx.x); __trap(); } } while (0)
#else
#define BG_ASSERT(cond) do { } while (0)
#endif


#define BG_MAX_BLOCK 65536u   /* largest payload a block may carry (applet -@1 uses 0x10000, htslib 0xff00) */
#define BG_DATA_BYTES (BG_MAX_BLOCK + 32u)
#define BG_HASH_BITS 14
#define BG_HASH_SIZE (1u << BG_HASH_BITS)
#define BG_NOPOS 0xFFFFu
#define BG_CHUNK 68u          /* parse/emit granule: one thread per chunk; 17 words => conflict-free lane stride */
#define BG_THREADS 1024u
#define BG_MAX_CHUNKS 1024u    /* array size; ceil(65536/68) = 964 chunks are ever live */
#define BG_SUPER 32u           /* chunks per super-chunk in the hierarchical walk */
#define BG_SUPER_POS (BG_SUPER * BG_CHUNK)
#define BG_MAX_TOKEN 258u
#define BG_SLOT_BYTES 65536u  /* one output slot = the largest legal BGZF member */
#define BG_HISTORY_STEP 272u  /* history comes in multiples of 4 chunks = 17 x 16 bytes: chunk-aligned for the token passes, 16-byte aligned for the bulk load */
#define BG_MAX_HISTORY 32640u /* 480 chunks: the most history a primed piece carries (the DEFLATE window is 32768) */
#define BG_CRC_WORDS 17u      /* CRC slice per thread, in 32-bit words (odd => conflict-free smem striding) */
#define BG_MIN_LOOKUP 3       /* shortest match the chain search can return (3 only where the hash window is 3 bytes: see bg_phase_settle) */

/* ---- region B overlay (32 KiB): the hash heads during the build, then everything Huffman ---- */
#define BG_B_LFREQ 0        /* u32[288] */
#define BG_B_DFREQ 1152     /* u32[32]  */
#define BG_B_PFREQ 1280     /* u32[20]  */
#define BG_B_LLEN 1360      /* u8[288]  */
#define BG_B_DLEN 1648      /* u8[32]   */
#define BG_B_PLEN 1680      /* u8[32]   */
#define BG_B_LCODE 1712     /* u16[288] */
#define BG_B_DCODE 2288     /* u16[32]  */
#define BG_B_PCODE 2352     /* u16[24]  */
#define BG_B_KEYS 2400      /* u32[512]  sort keys (freq<<9 | sym) */
#define BG_B_TREEW 4448     /* u32[640]  node weights, then depths */
#define BG_B_TREEP 7008     /* u16[640]  parent links */
#define BG_B_ENTRY 8288     /* u16[1024] first token start inside each chunk, chunk-relative (BG_NOPOS: none) */
#define BG_B_CBITS 10336    /* u32[1024] token bits per chunk, then exclusive prefix */
#define BG_B_ITEMS 14432    /* u16[320]  precode items: sym | extra<<5 */
#define BG_B_SCRATCH 15072  /* u32[64]   small-array scratch for the sequential Huffman code */
#define BG_B_DKEYS 15328    /* u32[32]   dist sort keys */
#define BG_B_PKEYS 15456    /* u32[32]   precode sort keys */
#define BG_B_DTREEW 15584   /* u32[64]   */
#define BG_B_DTREEP 15840   /* u16[64]   */
#define BG_B_END 15968
#define BG_B_SENTRY 16000     /* u32[32]   where the parse enters each super-chunk */
#define BG_B_XTAB 16384       /* u16[31*258] super-chunk exit offset for every possible entry offset */
#define BG_B_PERM 20480       /* u16[1024]   chunk order of the token passes (the walk tables are dead by then; IOFF ends at 20480) */
#define BG_B_CLASSCNT 4448    /* u32[8*32]   chunks per (class, warp), then their exclusive scan (tree space: written between the walk list's last use and the tally) */

/* scalars kept in the always-live misc area (u32 each) */
enum {
    BG_S_NUSED = 0, BG_S_MINLEN, BG_S_HBYTES, BG_S_CRC, BG_S_NITEMS, BG_S_NL, BG_S_ND, BG_S_NP,
    BG_S_BTYPE, BG_S_HDRBITS, BG_S_TOKBITS, BG_S_PAYLOAD, BG_S_STATUS, BG_S_DYNSYMS, BG_S_STASYMS, BG_S_WALKEND,
    BG_S_EXTRA, BG_S_DYNHDR, BG_S_WLIST, BG_S_HM, BG_S_HOVF, BG_S_DM, BG_S_PM, BG_S_DEPTH,
    BG_S_COUNT = 32
};

struct BgParams {
    int depth;        /* chain nodes visited per position */
    int nice;         /* stop searching at this length */
    int lazy;         /* 0 greedy, 1 one-ahead, 2 two-ahead */
    int passthrough;  /* inputs this short are stored (reference: 55 - 4*level) */
    int hlong;        /* hash window (bytes) when short matches do not pay (few distinct literals): 8 or 5 */
    int opt_passes;   /* > 0: near-optimal class (levels 10-12): that many min-cost-path passes after the lazy parse */
};

/* level 1..12 -> search effort; the classes follow libdeflate_alloc_compressor_ex (deflate_compress.c:3921-4007):
 * 1-4 greedy, 5-7 lazy, 8-9 lazy2, 10-12 near-optimal (lazy2 first, then min-cost-path passes over up to four
 * matches per position, the role of deflate_compress_near_optimal :3593-3850 / deflate_find_min_cost_path :3328-3400).  The numbers are this codec's own: on low-entropy text (FASTQ/SAM) an 8-byte
 * hash with a shallow chain reaches the reference's level-6 size (+1 %) at a fraction of the candidate visits.  Levels 8 and 9
 * walk 32 and 64 chain nodes (the reference: 300 and 600): +1.3 ... +2.0 % of the reference's size on FASTQ / SAM / BAM-like
 * data at the same level, for twice the throughput of the 64 / 128 this codec used before (+0.6 ... +1.2 %). */
BG_HD BgParams bg_level_params(int level)
{
    BgParams p;
    if (level < 1) level = 1;
    if (level > 12) level = 12;
    p.depth = level <= 4 ? level : level == 5 ? 6 : level == 6 ? 8 : level == 7 ? 16 : level == 8 ? 32 : level == 9 ? 64
            : level == 10 ? 128 : level == 11 ? 256 : 512;
    p.nice = level <= 2 ? 32 : level == 3 ? 48 : level <= 5 ? 64 : level == 6 ? 65 : level == 7 ? 130 : 258;
    p.lazy = level <= 4 ? 0 : level <= 7 ? 1 : 2;
    p.passthrough = 55 - 4 * level;
    p.hlong = level <= 7 ? 8 : level <= 9 ? 5 : 4;
    p.opt_passes = level <= 9 ? 0 : level <= 11 ? 3 : 4;
    return p;
}

struct BgCtx {
    uint32_t *dataw;    /* smem: the block, BG_DATA_BYTES */
    uint16_t *prev;     /* smem region A (128 KiB): hash, then chain links */
    uint8_t *stepcode;  /* region A[0..64K): 0 literal, 1..254 match len-2, 255 len >= 257 (see R) */
    uint8_t *jump8;     /* region A[64K..128K): exit offset past the chunk end, 255 = walk it */
    uint16_t *offarr;   /* region A[64K..128K) again, after the walk: match offset at [pos>>1] */
    uint16_t *head;     /* smem region B (32 KiB): hash heads, later the overlay above */
    uint8_t *regb;      /* region B as bytes */
    uint8_t *litflag;   /* smem u8[256] */
    uint32_t *crctab;   /* smem u32[256] */
    uint32_t *scal;     /* smem u32[BG_S_COUNT] */
    uint32_t *R;        /* global scratch u32[BG_MAX_BLOCK+8]: len<<16 | offset per position */
    uint32_t *cand;     /* global scratch u32[4*BG_MAX_BLOCK] or NULL: up to 4 matches per position (near-optimal class) */
    uint32_t *out;      /* global: this block's output slot, BG_SLOT_BYTES, 16-byte aligned */
    const uint32_t *crcpow; /* global u32[BG_THREADS]: x^(8*4*BG_CRC_WORDS*k) mod P */
    const uint16_t *perm;   /* smem u16[BG_MAX_CHUNKS] or NULL: which chunk thread i walks in the token passes (tally, sizes, emit).
                               Any permutation gives the same bytes; the kernel groups chunks of similar make-up into one warp. */
    uint32_t n;         /* payload bytes */
    /* framing of this block's slot, packed into one word (bg_frame): header bytes | trailer bytes << 8 | final << 16 | piece << 17.
     * Members: hdr = 18 BGZF ("BC" subfield, BSIZE) or 20 MiGz ("MZ" subfield, u32 compressed size: applet/7migz.c:224-228),
     * trl = 8 (CRC32, ISIZE), final = 1.
     * Piece mode (the other block-gzip containers and whole-stream gzip: a member is made of several 64 KiB pieces): the slot
     * holds `hdr` free bytes, the DEFLATE data of this block, `trl` free bytes; no gzip framing is written (the host fills the
     * gaps of a member's first and last piece).  A piece that is not `final` carries BFINAL = 0 and ends with an empty stored
     * block that pads to the byte ("full flush": what the reference makes of every dictzip / RAZF chunk by clearing the
     * final bit and appending 00 00 ff ff, applet/7dictzip.c:92-126, 7razf_testdecode.c:1023), so pieces concatenate bytewise. */
    uint32_t frame;             /* ... | history chunks << 18 (bg_f_hist) */
    BgParams prm;
};

BG_HD uint32_t bg_frame(uint32_t hdr, uint32_t trl, uint32_t final, uint32_t piece, uint32_t hist = 0) { return hdr | (trl << 8) | (final << 16) | (piece << 17) | ((hist / BG_CHUNK) << 18); }
/* history: the first bg_f_hist(c) bytes of the block buffer (a multiple of BG_HISTORY_STEP, at most BG_MAX_HISTORY) are the input
 * that precedes this piece: matches may reach into them (dictionary priming, as pigz does between its chunks), nothing is
 * emitted for them, and CRC-32 / sizes cover the payload behind them only */
BG_HD uint32_t bg_f_hist(const BgCtx &c) { return (c.frame >> 18) * BG_CHUNK; }
BG_HD uint32_t bg_f_hdr(const BgCtx &c) { return c.frame & 0xffu; }
BG_HD uint32_t bg_f_trl(const BgCtx &c) { return (c.frame >> 8) & 0xffu; }
BG_HD uint32_t bg_f_final(const BgCtx &c) { return (c.frame >> 16) & 1u; }
BG_HD bool bg_f_piece(const BgCtx &c) { return (c.frame >> 17) & 1u; }

/* ------------------------------------------------------------------------------------------------ */
/* small helpers                                                                                    */

BG_HD uint32_t bg_ld32(const uint32_t *w, uint32_t p)
{
    uint32_t i = p >> 2, s = (p & 3u) * 8u;
    uint32_t lo = w[i], hi = w[i + 1];
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, p << 3);      /* (the shift count is taken modulo 32: no need to mask it first) */
#else
    return s ? (lo >> s) | (hi << (32u - s)) : lo;
#endif
}

BG_HD uint32_t bg_ld8(const uint32_t *w, uint32_t p) { return ((const uint8_t *)w)[p]; }

BG_HD uint32_t bg_funnel(uint32_t lo, uint32_t hi, uint32_t s)
{
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, s);
#else
    return s ? (lo >> s) | (hi << (32u - s)) : lo;
#endif
}

BG_HD int bg_bsr(uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return 31 - __clz(v);
#else
    return 31 - __builtin_clz(v);
#endif
}

BG_HD int bg_ctz(uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return __ffs(v) - 1;
#else
    return __builtin_ctz(v);
#endif
}

BG_HD uint32_t bg_brev(uint32_t v, int nbits)
{
#if defined(__CUDA_ARCH__)
    return __brev(v) >> (32 - nbits);
#else
    uint32_t r = 0;
    for (int i = 0; i < nbits; i++)
        r |= ((v >> i) & 1u) << (nbits - 1 - i);
    return r;
#endif
}

BG_HD void bg_add32(uint32_t *a, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    atomicAdd(a, v);
#else
    *a += v;
#endif
}

BG_HD uint32_t bg_fetch_add32(uint32_t *a, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return atomicAdd(a, v);
#else
    uint32_t old = *a;
    *a += v;
    return old;
#endif
}

BG_HD void bg_or32(uint32_t *a, uint32_t v)
{
#if defined(__CUDA_ARCH__)
    atomicOr(a, v);
#else
    *a |= v;
#endif
}

/* DEFLATE length (3..258) -> slot 0..28, extra bit count and value (RFC 1951 3.2.5) computed, not tabled */
BG_HD uint32_t bg_len_slot(uint32_t len, uint32_t *nextra, uint32_t *extra)
{
    uint32_t l = len - 3;
    if (l < 8) { *nextra = 0; *extra = 0; return l; }
    if (len == 258) { *nextra = 0; *extra = 0; return 28; }
    uint32_t nb = (uint32_t)bg_bsr(l) - 2;
    *nextra = nb;
    *extra = l & ((1u << nb) - 1);
    return 8 + 4 * (nb - 1) + ((l >> nb) & 3);
}

/* offset (1..32768) -> slot 0..29 */
BG_HD uint32_t bg_off_slot(uint32_t off, uint32_t *nextra, uint32_t *extra)
{
    uint32_t d = off - 1;
    if (d < 4) { *nextra = 0; *extra = 0; return d; }
    uint32_t b = (uint32_t)bg_bsr(d);
    *nextra = b - 1;
    *extra = d & ((1u << (b - 1)) - 1);
    return 2 * b + ((d >> (b - 1)) & 1);
}

BG_HD uint32_t bg_len_slot_extra_bits(uint32_t slot) { return slot < 8 || slot == 28 ? 0 : (slot - 4) >> 2; }
BG_HD uint32_t bg_off_slot_extra_bits(uint32_t slot) { return slot < 4 ? 0 : (slot - 2) >> 1; }

/* static litlen code length (RFC 1951 3.2.6) */
BG_HD uint32_t bg_static_llen(uint32_t sym) { return sym < 144 ? 8 : sym < 256 ? 9 : sym < 280 ? 7 : 8; }

/* ---- CRC-32 (reflected 0xEDB88320) ------------------------------------------------------------- */

#define BG_CRC_POLY 0xEDB88320u

/* a(x)*b(x) mod P in the reflected representation (bit 31 = x^0); same algebra as zlib's multmodp */
BG_HD uint32_t bg_crc_mul(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (int i = 0; i < 32; i++) {
        p ^= b & (0u - ((a >> (31 - i)) & 1u));
        b = (b >> 1) ^ (BG_CRC_POLY & (0u - (b & 1u)));
    }
    return p;
}

BG_HD uint32_t bg_crc_byte(const uint32_t *tab, uint32_t r, uint32_t b) { return tab[(r ^ b) & 0xff] ^ (r >> 8); }

/* ---- match words (the per-position scratch R[]): len << 16 | (0xffff - offset).  The maximum of two such words is the
 * longer match and, among equals, the nearer one: candidates of one position can be merged with atomicMax in any order. */
BG_HD uint32_t bg_mw(uint32_t len, uint32_t off) { return (len << 16) | (0xffffu - off); }
BG_HD uint32_t bg_mw_off(uint32_t r) { return 0xffffu - (r & 0xffffu); }

/* ------------------------------------------------------------------------------------------------ */
/* phase 0: clear                                                                                   */

BG_HD void bg_phase_init(const BgCtx &c, uint32_t t, uint32_t T)
{
    for (uint32_t i = t; i < BG_HASH_SIZE; i += T)
        c.head[i] = BG_NOPOS;
    if (t < 256)
        c.litflag[t] = 0;
    if (t < 28)
        ((uint8_t *)c.dataw)[c.n + t] = 0;  /* zero tail so word reads past n are defined */
    if (t < BG_S_COUNT)
        c.scal[t] = 0;
}

/* phase 1a: which literals occur (benign same-value stores) */
BG_HD void bg_phase_census(const BgCtx &c, uint32_t t, uint32_t T)
{
    for (uint32_t p = t; p < c.n; p += T)
        c.litflag[bg_ld8(c.dataw, p)] = 1;
}

/* CRC over the first m = n/4 words of the payload (hw history words come first), cut into BG_THREADS slices of BG_CRC_WORDS
 * words, right-aligned: slice k ends k slices before word m, so its combine factor is the constant crcpow[k].  Thread u of
 * U takes slices u, u + U, u + 2U, ...: two at a time, as two independent lookup chains.  Each thread's share is XORed into
 * scal[BG_S_CRC], which must start at 0; bg_crc_finish() adds the ragged tail once every share is in. */
BG_HD void bg_crc_slices(const BgCtx &c, uint32_t u, uint32_t U)
{
    const uint32_t hw = bg_f_hist(c) >> 2;
    const uint32_t m = (c.n >> 2) - hw;
    const uint32_t *d = c.dataw + hw;
    uint32_t acc = 0;
    for (uint32_t k0 = u; k0 < BG_THREADS; k0 += 2 * U) {
        const uint32_t k1 = k0 + U;                                   /* (k1 >= BG_THREADS: an empty slice) */
        const uint32_t e0 = m >= BG_CRC_WORDS * k0 ? m - BG_CRC_WORDS * k0 : 0;
        const uint32_t e1 = k1 < BG_THREADS && m >= BG_CRC_WORDS * k1 ? m - BG_CRC_WORDS * k1 : 0;
        const uint32_t b0 = e0 >= BG_CRC_WORDS ? e0 - BG_CRC_WORDS : 0, b1 = e1 >= BG_CRC_WORDS ? e1 - BG_CRC_WORDS : 0;
        if (e0 == b0) break;                                          /* (slices further left are empty too) */
        uint32_t r0 = b0 == 0 ? 0xFFFFFFFFu : 0u, r1 = b1 == 0 ? 0xFFFFFFFFu : 0u;
        for (uint32_t i = 0; i < BG_CRC_WORDS; i++) {
            if (b0 + i < e0) {
                const uint32_t v = d[b0 + i];
                r0 = bg_crc_byte(c.crctab, r0, v & 0xff);
                r0 = bg_crc_byte(c.crctab, r0, (v >> 8) & 0xff);
                r0 = bg_crc_byte(c.crctab, r0, (v >> 16) & 0xff);
                r0 = bg_crc_byte(c.crctab, r0, v >> 24);
            }
            if (b1 + i < e1) {
                const uint32_t v = d[b1 + i];
                r1 = bg_crc_byte(c.crctab, r1, v & 0xff);
                r1 = bg_crc_byte(c.crctab, r1, (v >> 8) & 0xff);
                r1 = bg_crc_byte(c.crctab, r1, (v >> 16) & 0xff);
                r1 = bg_crc_byte(c.crctab, r1, v >> 24);
            }
        }
        acc ^= bg_crc_mul(r0, c.crcpow[k0]);
        if (e1 > b1) acc ^= bg_crc_mul(r1, c.crcpow[k1]);
    }
    /* XOR is order-independent: fold inside the warp, then one shared atomic per warp */
#if defined(__CUDA_ARCH__)
    for (int s = 16; s > 0; s >>= 1)
        acc ^= __shfl_xor_sync(0xffffffffu, acc, s);
    if ((u & 31u) == 0 && acc)
        atomicXor(&c.scal[BG_S_CRC], acc);
#else
    c.scal[BG_S_CRC] ^= acc;
#endif
}

/* phase 1: census and CRC slices, one slice per thread (the kernel runs the two apart: the census feeds the search, the
 * CRC is read only by the trailer) */
BG_HD void bg_phase_scan(const BgCtx &c, uint32_t t, uint32_t T)
{
    bg_phase_census(c, t, T);
    bg_crc_slices(c, t, T);
}

/* phase 2: distinct-literal count (t < 256) */
BG_HD void bg_phase_count(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    if (t < 256 && c.litflag[t])
        bg_add32(&c.scal[BG_S_NUSED], 1);
}

/* Minimum useful match length from the number of distinct literals: cheap literals (DNA, quality strings)
 * make short matches a loss for a lazy parser.  Same thresholds as the reference's heuristic table
 * (deflate_compress.c:2295-2327), expressed as ranges. */
BG_HD uint32_t bg_min_match_len(uint32_t nused, int depth, uint32_t n)
{
    uint32_t ml;
    if (n < 512) return 3;
    ml = nused < 6 ? 9 : nused < 8 ? 8 : nused < 10 ? 7 : nused < 16 ? 6 : nused < 45 ? 5 : nused < 80 ? 4 : 3;
    if (depth < 16) {
        uint32_t cap = depth < 5 ? 4 : depth < 10 ? 5 : 7;
        if (ml > cap) ml = cap;
    }
    return ml;
}

/* one thread, after every bg_crc_slices() share is in: the ragged tail bytes and the final complement */
BG_HD void bg_crc_finish(const BgCtx &c)
{
    const uint32_t n = c.n;
    uint32_t r = c.scal[BG_S_CRC];
    if (((n - bg_f_hist(c)) >> 2) == 0) r = 0xFFFFFFFFu;
    for (uint32_t p = n & ~3u; p < n; p++)
        r = bg_crc_byte(c.crctab, r, bg_ld8(c.dataw, p));
    c.scal[BG_S_CRC] = ~r;
}

/* phase 3a (thread 0): minlen, chain depth and hash width from the literal census */
BG_HD void bg_phase_settle_census(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    if (t != 0) return;
    const uint32_t n = c.n;
    c.scal[BG_S_MINLEN] = bg_min_match_len(c.scal[BG_S_NUSED], c.prm.depth, n);
    /* binary-looking blocks (BAM records, executables: 80+ distinct byte values) get half as much chain depth again:
     * their matches are spread over more candidates than those of text, and the fixed depth that reaches the
     * reference's size on FASTQ/SAM text is 1 % short of it there (DESIGN.md, ratio probe) */
    c.scal[BG_S_DEPTH] = c.scal[BG_S_NUSED] >= 80 && c.prm.opt_passes == 0 ? (uint32_t)c.prm.depth + ((uint32_t)c.prm.depth + 1) / 2 : (uint32_t)c.prm.depth;
    /* hash width follows the literal census alone (not the depth cap): cheap literals => only long matches pay */
    c.scal[BG_S_HBYTES] = bg_min_match_len(c.scal[BG_S_NUSED], 1000, n) >= 5 ? (uint32_t)c.prm.hlong : 4u;
    /* Binary-looking blocks (3-byte matches pay: 80+ distinct byte values) at levels 6 and up hash THREE bytes, so that the
     * chains also hold the 3-byte matches the reference finds with its hash3 table (hc_matchfinder.h:112-131,222-227).  Chain
     * nodes that share only those 3 bytes with the position do not count against the depth (BG_DEEP_SCAN): the walk still
     * reaches every node a 4-byte window would have chained.  Measured at level 6: an ELF binary -3.0 % (it was 4 % behind
     * the reference), BAM-like records +-0.0 %; shallower walks (levels 2-5) lose on BAM-like data (+0.7 % at level 3): not done there. */
    if (c.scal[BG_S_MINLEN] == 3 && c.prm.depth >= 8) c.scal[BG_S_HBYTES] = 3;
}

/* phase 3 (thread 0): finish the CRC, settle minlen/hash width */
BG_HD void bg_phase_settle(const BgCtx &c, uint32_t t, uint32_t T)
{
    if (t == 0) bg_crc_finish(c);
    bg_phase_settle_census(c, t, T);
}

/* phase 4: hash every position that has a full hash window into prev[] */
BG_HD uint32_t bg_hash(const uint32_t *dataw, uint32_t p, uint32_t hbytes)
{
    uint32_t v = bg_ld32(dataw, p);
    if (hbytes == 3) v &= 0xffffffu;        /* (callers in a loop pass a loop-invariant hbytes: the test is hoisted or predicated) */
    uint32_t h = v * 0x1E35A7BDu;
    if (hbytes == 5)
        h ^= bg_ld8(dataw, p + 4) * 0x9E3779B1u;
    else if (hbytes == 8)
        h ^= bg_ld32(dataw, p + 4) * 0x9E3779B1u;
    return h >> (32 - BG_HASH_BITS);
}

BG_HD void bg_phase_hash(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n, hb = c.scal[BG_S_HBYTES];
    for (uint32_t p = t; p < n; p += T)
        c.prev[p] = (p + hb <= n) ? (uint16_t)bg_hash(c.dataw, p, hb) : (uint16_t)BG_NOPOS;
}

/* phase 5 (sequential twin of the warp build in the .cu): prev[p] = nearest earlier position with my hash */
BG_HD void bg_build_sequential(const BgCtx &c)
{
    for (uint32_t p = 0; p < c.n; p++) {
        uint32_t h = c.prev[p];
        if (h == BG_NOPOS) continue;
        c.prev[p] = c.head[h];
        c.head[h] = (uint16_t)p;
    }
}

/* number of equal bytes of p.. and q.. starting at offset l (a multiple of 4), capped at maxl.  The two byte streams
 * are read as aligned words that slide along (one new word per stream and step) with fixed funnel-shift amounts. */
BG_HD uint32_t bg_match_len(const uint32_t *dw, uint32_t p, uint32_t q, uint32_t l, uint32_t maxl)
{
    if (l >= maxl) return maxl;
    const uint32_t sp = (p & 3u) * 8u, sq = (q & 3u) * 8u;
    const uint32_t *wp = dw + ((p + l) >> 2), *wq = dw + ((q + l) >> 2);
    uint32_t plo = wp[0], qlo = wq[0];
    /* eight bytes per turn: the four new words are requested together, so their shared-memory latencies overlap (the block is
     * followed by 32 zero bytes: reading two words past the last compared byte stays inside the buffer) */
    for (;;) {
        const uint32_t p1 = wp[1], q1 = wq[1], p2 = wp[2], q2 = wq[2];
        const uint32_t x1 = bg_funnel(plo, p1, sp) ^ bg_funnel(qlo, q1, sq);
        if (x1) { l += (uint32_t)bg_ctz(x1) >> 3; break; }
        const uint32_t x2 = bg_funnel(p1, p2, sp) ^ bg_funnel(q1, q2, sq);
        if (x2) { l += 4u + ((uint32_t)bg_ctz(x2) >> 3); break; }
        l += 8;
        if (l >= maxl) break;
        plo = p2;
        qlo = q2;
        wp += 2;
        wq += 2;
    }
    return l > maxl ? maxl : l;
}

/* is q a candidate for p: an earlier position at most 32768 back?  One unsigned compare covers "no link" as well:
 * BG_NOPOS is 65535 >= p, so p - q - 1 wraps around for it (as it does for q == p). */
BG_HD bool bg_in_window(uint32_t p, uint32_t q) { return p - q - 1u < 32768u; }

/* phase 6: all-position search.
 * For position p: follow the chain of earlier positions with the same hash (nearest first, at most `depth`
 * of them, offsets <= 32768), keep the longest match (first found wins ties, i.e. the nearest), stop at
 * `nice` or at the end of the block.  A candidate is examined only if the 4 bytes ending just past the best
 * length so far agree (they must, for it to be longer).
 * (A per-lane step machine — one 4-byte comparison per call, lanes refilling themselves — and a per-lane parse of
 * ranges with match remainders were both built and measured this round; in lock-step they cost more than these
 * nested loops save: DESIGN.md section 3, branch exp/range-parse.) */

/* ---- greedy / lazy classes (levels 1-9): the search in three passes ---------------------------------------------
 * The reference searches only where its parse stands (13-23 % of the positions at level 6, SURVEY section 6); an
 * all-position search pays the full chain walk and the long extensions inside every match as well.  Here:
 *   pass 1  every position: the match with its NEAREST candidate only (uniform work).  A greedy step from p lands on
 *           p + len (or p + 1): that landing position is marked; a position also notes whether a deeper look could pay
 *           at all (it has a second candidate in the window and the nearest match is short of `nice`)
 *   todo    positions worth a deep search = marked ones (any parse that steps through nearest matches stands only on
 *           those), plus the one or two after them that the lazy rule looks at, if they are eligible
 *   pass 2  deep search of the todo positions only: walk the rest of the chain; a candidate that agrees with p on the
 *           4 bytes ending just past the nearest match's length may be longer and is put on a queue
 *   pass 3  the queue is drained 32 candidates at a time — one candidate per lane, all lanes busy — and merged into
 *           R[p] with atomicMax on the match word (longest, nearest among equals)
 * A parse that leaves the marked set (a deep match ends elsewhere) continues on nearest-candidate matches until its next
 * step, which lands on a marked position again.  Measured (8 MiB, level 6): 43 % (FASTQ-like) / 21 % (SAM-like) of the
 * positions get a deep search instead of 76 %, for +0.09 % / +0.09 % compressed size.
 * Region B during the search (the hash heads are dead): */
#define BG_B_TODO 0u          /* u32[2048]  pass 1: eligible bits; then the todo bits */
#define BG_B_MARK 8192u       /* u32[2064]  landing positions of the greedy steps (dead once the todo bits are made) */
#define BG_B_QUEUE 8192u      /* u32[32][160] (shallow chains) or u32[32][96] (deep): per warp, (p << 16 | q) candidates waiting for their extension */
#define BG_B_RINGR 20480u     /* u32[32][64]   deep chains, per warp: the nearest-match words of the todo positions in the ring (fetched ahead, cp.async) */
#define BG_B_RING 28672u      /* u16[32][64]   per warp: ring of todo positions waiting for a free lane */
#define BG_QUEUE_WORDS 96u    /* deep chains: a look at the queue every 2 chain steps: 31 + 32 * 2 entries fit */
#define BG_SCAN_CHUNK 2u
#define BG_QUEUE_WORDS_SHALLOW 160u   /* shallow chains (32 positions side by side): every 4 steps, 31 + 32 * 4 */
#define BG_SCAN_CHUNK_SHALLOW 4u

BG_HD bool bg_match_ok(uint32_t r, uint32_t minlen);

/* pass 1 for one position: match word of the nearest candidate (0: none of length >= 4); *deep: a deep search may
 * improve on it; *target: where a greedy step from p lands */
struct BgSearchPrm {      /* the block's search scalars, read once per phase (not once per position) */
    uint32_t depth, nice, minlen;
    bool h3;              /* 3-byte hash window (binary-looking block, level 6 and up) */
};
BG_HD BgSearchPrm bg_search_prm(const BgCtx &c)
{
    BgSearchPrm s;
    s.depth = c.scal[BG_S_DEPTH];
    s.nice = (uint32_t)c.prm.nice;
    s.minlen = c.scal[BG_S_MINLEN];
    s.h3 = c.scal[BG_S_HBYTES] == 3;
    return s;
}

template <bool H3>
BG_HD uint32_t bg_nearest_t(const BgCtx &c, const BgSearchPrm &sp, uint32_t p, bool *deep, uint32_t *target)
{
    uint32_t maxl = c.n - p;
    if (maxl > 258) maxl = 258;
    *deep = false;
    *target = p + 1;
    if (maxl < (uint32_t)BG_MIN_LOOKUP) return 0;
    const uint32_t q = c.prev[p];
    if (!bg_in_window(p, q)) return 0;
    const uint32_t *dw = c.dataw;
    uint32_t len = 3;
    if (H3) {
        len = 2;
        if (((bg_ld32(dw, q) ^ bg_ld32(dw, p)) & 0xffffffu) == 0) len = bg_match_len(dw, p, q, 0, maxl);
    } else if (bg_ld32(dw, q) == bg_ld32(dw, p)) {
        len = bg_match_len(dw, p, q, 4, maxl);
    }
    *deep = sp.depth > 1 && len < sp.nice && len < maxl && bg_in_window(p, c.prev[q]);
    if (len <= (H3 ? 2u : 3u)) return 0;
    const uint32_t r = bg_mw(len, p - q);
    if (bg_match_ok(r, sp.minlen)) *target = p + len;
    return r;
}
BG_HD uint32_t bg_nearest(const BgCtx &c, const BgSearchPrm &sp, uint32_t p, bool *deep, uint32_t *target)
{
    return sp.h3 ? bg_nearest_t<true>(c, sp, p, deep, target) : bg_nearest_t<false>(c, sp, p, deep, target);
}

/* ---- near-optimal class (levels 10-12): the same passes, over EVERY position that has a second candidate, and besides the
 * longest match (R[p], which seeds the first parse) the longest match of each of four offset ranges is kept (cand[4p + bin]:
 * match words merged with atomicMax like R[p]) — the candidates the min-cost-path passes choose from.  For a length l the
 * cheapest offset is that of the nearest range holding a match of at least l bytes; a longer, nearer match makes a farther,
 * shorter one irrelevant, so it does not matter whether such a dominated candidate was measured at all (the kernel stops
 * testing against the nearest match once longer ones are known: same decisions, fewer extensions).  This is the role of
 * bt_matchfinder_get_matches (bt_matchfinder.h:140-340: all matches of strictly increasing length and offset), capped at
 * one match per range. */
BG_HD uint32_t bg_off_bin(uint32_t off) { return off <= 32u ? 0u : off <= 512u ? 1u : off <= 8192u ? 2u : 3u; }

BG_HD void bg_cand_init(const BgCtx &c, uint32_t p, uint32_t r)
{
    uint32_t *cd = c.cand + 4u * p;
    const uint32_t k = r ? bg_off_bin(bg_mw_off(r)) : 4u;
    cd[0] = k == 0 ? r : 0u; cd[1] = k == 1 ? r : 0u; cd[2] = k == 2 ? r : 0u; cd[3] = k == 3 ? r : 0u;
}

BG_HD void bg_phase_search_clear(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint32_t *w = (uint32_t *)(c.regb + BG_B_TODO);
    for (uint32_t i = t; i < (BG_B_MARK + 8256u) / 4u; i += T) w[i] = 0;
}

/* (the kernel's pass 1 sets the same bits with one ballot per 32 positions: bgzf_compress.cu) */
BG_HD void bg_phase_search1(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint32_t *elig = (uint32_t *)(c.regb + BG_B_TODO), *mark = (uint32_t *)(c.regb + BG_B_MARK);
    const uint32_t hist = bg_f_hist(c);
    if (t == 0) bg_or32(&mark[hist >> 5], 1u << (hist & 31u));      /* the parse starts behind the history */
    const BgSearchPrm sp = bg_search_prm(c);
    for (uint32_t p = t; p < c.n; p += T) {
        bool deep;
        uint32_t target;
        if (p < hist) {                                             /* history: never a token, never searched */
            c.R[p] = 0;
            if (c.prm.opt_passes > 0) bg_cand_init(c, p, 0);
            continue;
        }
        c.R[p] = bg_nearest(c, sp, p, &deep, &target);
        if (c.prm.opt_passes > 0) bg_cand_init(c, p, c.R[p]);
        if (deep) bg_or32(&elig[p >> 5], 1u << (p & 31u));
        bg_or32(&mark[target >> 5], 1u << (target & 31u));
    }
}

/* todo = (marked, and the `lazy` positions after a marked one) & eligible; `own`/`parts`: a cluster's CTA keeps every
 * parts-th word (32 positions) only */
BG_HD void bg_phase_search_todo(const BgCtx &c, uint32_t t, uint32_t T, uint32_t own, uint32_t parts)
{
    uint32_t *todo = (uint32_t *)(c.regb + BG_B_TODO);
    const uint32_t *mark = (const uint32_t *)(c.regb + BG_B_MARK);
    for (uint32_t i = t; i < 2048u; i += T) {
        const uint32_t m = mark[i], pm = i ? mark[i - 1] : 0u;
        uint32_t w = m;
        if (c.prm.lazy >= 1) w |= (m << 1) | (pm >> 31);
        if (c.prm.lazy >= 2) w |= (m << 2) | (pm >> 30);
        if (c.prm.opt_passes > 0) w = 0xffffffffu;                  /* near-optimal class: the optimiser may stand anywhere */
        w &= todo[i];
        if (i % parts != own) w = 0;
        todo[i] = w;
    }
}

/* which of the 4 bytes ending just past the match to beat a candidate must share: all of them; with a 3-byte hash window
 * and nothing to beat yet (no nearest match), the first three — a 3-byte match is a match there */
BG_HD uint32_t bg_tail_mask(bool h3, uint32_t r1) { return h3 && !r1 ? 0xffffffu : 0xffffffffu; }

/* pass 2 for one position: chain candidates beyond the nearest that may beat it.  Calls push(q) for each. */
#define BG_DEEP_SCAN(c, p, PUSH)                                                                     \
    do {                                                                                             \
        const uint32_t r1_ = (c).R[p];                                                               \
        const uint32_t b1_ = r1_ ? r1_ >> 16 : 3u;                                                   \
        const bool h3_ = (c).scal[BG_S_HBYTES] == 3;                                                 \
        const uint32_t tmask_ = bg_tail_mask(h3_, r1_);                                              \
        const uint32_t tail_ = bg_ld32((c).dataw, (p) + b1_ - 3u) & tmask_;                          \
        uint32_t q_ = (c).prev[(c).prev[p]];                                                         \
        int depth_ = (int)(c).scal[BG_S_DEPTH] - 1, cap_ = 4 * depth_;                               \
        const uint32_t f4_ = bg_ld32((c).dataw, (p));                                                \
        while (depth_ > 0 && cap_ > 0 && bg_in_window(p, q_)) {                                      \
            if ((bg_ld32((c).dataw, q_ + b1_ - 3u) & tmask_) == tail_) { PUSH(q_); }                 \
            /* 3-byte hash window: a node that shares only 3 bytes with p is looked at for free (up to 4x the depth in   \
             * all), so that the nodes a 4-byte window would have chained are still all visited */                    \
            if (!h3_ || bg_ld32((c).dataw, q_) == f4_) depth_--;                                     \
            cap_--;                                                                                  \
            q_ = (c).prev[q_];                                                                       \
        }                                                                                            \
    } while (0)

/* pass 3 for one queued candidate: its full length, merged into R[p] (the kernel: atomicMax) */
BG_HD uint32_t bg_deep_extend(const BgCtx &c, bool h3, uint32_t p, uint32_t q)
{
    uint32_t maxl = c.n - p;
    if (maxl > 258) maxl = 258;
    const uint32_t l = bg_match_len(c.dataw, p, q, 0, maxl);
    return l >= (h3 ? 3u : 4u) ? bg_mw(l, p - q) : 0u;
}

/* sequential twin of the kernel's passes 2 and 3 */
BG_HD void bg_phase_search2(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t *todo = (const uint32_t *)(c.regb + BG_B_TODO);
    for (uint32_t p = t; p < c.n; p += T) {
        if (!((todo[p >> 5] >> (p & 31u)) & 1u)) continue;
#define BG_PUSH_SEQ(q) do { const uint32_t v_ = bg_deep_extend(c, c.scal[BG_S_HBYTES] == 3, p, (q)); if (v_ > c.R[p]) c.R[p] = v_; \
                            if (v_ && c.prm.opt_passes > 0) { uint32_t *cd_ = c.cand + 4u * p + bg_off_bin(bg_mw_off(v_)); if (v_ > *cd_) *cd_ = v_; } } while (0)
        /* (the tail bytes compared are those of the NEAREST match for every candidate: R[p] is read once, before the walk) */
        BG_DEEP_SCAN(c, p, BG_PUSH_SEQ);
    }
}


/* ---- near-optimal class: minimum-cost path ------------------------------------------------------------------ */
#define BG_DP_OVERLAP 512u        /* a segment's backward pass starts this far past its end, from cost 0 */
#define BG_DP_RING 512u           /* cost-to-end of the next positions (power of two > 258) */
#define BG_B_LITCOST BG_B_KEYS            /* u8[256]  bits of literal b                      (sort keys are dead here) */
#define BG_B_LENCOST (BG_B_KEYS + 256)    /* u8[260]  bits of match length l (symbol + extra) */
#define BG_B_OFFCOST (BG_B_KEYS + 516)    /* u8[32]   bits of offset slot s (symbol + extra)  */

/* bit costs from the code lengths of the previous parse; unused symbols get a flat guess */
BG_HD void bg_phase_costs(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    uint8_t *rb = c.regb;
    const uint8_t *llen = rb + BG_B_LLEN, *dlen = rb + BG_B_DLEN;
    if (t < 256) rb[BG_B_LITCOST + t] = llen[t] ? llen[t] : 13;
    if (t >= 3 && t <= 258) {
        uint32_t nb, ex;
        const uint32_t sl = bg_len_slot(t, &nb, &ex);
        rb[BG_B_LENCOST + t] = (uint8_t)((llen[257 + sl] ? llen[257 + sl] : 13) + nb);
    }
    if (t < 30) rb[BG_B_OFFCOST + t] = (uint8_t)((dlen[t] ? dlen[t] : 10) + bg_off_slot_extra_bits(t));
}

/* packed choice: cost << 11 | length << 2 | candidate; the minimum of these picks the cheapest, then the shortest */
BG_HD uint32_t bg_dp_pack(uint32_t cost, uint32_t len, uint32_t cidx) { return (cost << 11) | (len << 2) | cidx; }

/* One backward step at position p of a segment ending (for this pass) at `e`: best way to code data[p..e).
 * ring[(q) & 511] holds the cost-to-end of position q for p < q <= p+258.  Sequential formulation. */
BG_HD uint32_t bg_dp_choose(const BgCtx &c, uint32_t p, uint32_t e, const uint32_t *ring)
{
    const uint8_t *rb = c.regb;
    uint32_t best = bg_dp_pack(rb[BG_B_LITCOST + bg_ld8(c.dataw, p)] + ring[(p + 1) & (BG_DP_RING - 1)], 1, 0);
    const uint32_t *cd = c.cand + 4u * p;
    uint32_t L[4], O[4], longest = 0;
    for (int k = 0; k < 4; k++) {
        L[k] = cd[k] >> 16;
        O[k] = cd[k] ? bg_mw_off(cd[k]) : 0u;
        if (L[k] > longest) longest = L[k];
    }
    uint32_t maxl = e - p;
    if (longest < maxl) maxl = longest;
    for (uint32_t l = 3; l <= maxl; l++) {
        const uint32_t k = l <= L[0] ? 0 : l <= L[1] ? 1 : l <= L[2] ? 2 : 3;      /* the nearest range that has a match this long */
        uint32_t nb, ex;
        const uint32_t cost = rb[BG_B_LENCOST + l] + rb[BG_B_OFFCOST + bg_off_slot(O[k], &nb, &ex)] + ring[(p + l) & (BG_DP_RING - 1)];
        const uint32_t v = bg_dp_pack(cost, l, k);
        if (v < best) best = v;
    }
    return best;
}

BG_HD void bg_dp_commit(const BgCtx &c, uint32_t p, uint32_t choice)
{
    const uint32_t l = (choice >> 2) & 511u, k = choice & 3u;
    if (l == 1) {
        c.stepcode[p] = 0;
    } else {
        c.stepcode[p] = (uint8_t)(l <= 256 ? l - 2 : 255);
        c.R[p] = bg_mw(l, bg_mw_off(c.cand[4u * p + k]));
    }
}

/* segment w of W (one warp each in the kernel): positions [w*S, (w+1)*S) get their decisions; the pass starts
 * BG_DP_OVERLAP positions later with cost 0 so that the relative costs have settled when it reaches the segment */
BG_HD void bg_dp_segment_bounds(uint32_t n, uint32_t w, uint32_t W, uint32_t *a, uint32_t *b, uint32_t *e)
{
    const uint32_t S = (n + W - 1) / W;
    *a = w * S < n ? w * S : n;
    *b = *a + S < n ? *a + S : n;
    *e = *b + BG_DP_OVERLAP < n ? *b + BG_DP_OVERLAP : n;
}

/* sequential twin of the kernel's warp-parallel pass (the emulator runs it with one "thread" per segment) */
BG_HD void bg_phase_dp(const BgCtx &c, uint32_t t, uint32_t T, uint32_t *rings)
{
    const uint32_t W = 32;
    if (t >= W || T < W) return;
    uint32_t a, b, e;
    bg_dp_segment_bounds(c.n, t, W, &a, &b, &e);
    if (a >= b) return;
    uint32_t *ring = rings + t * BG_DP_RING;
    ring[e & (BG_DP_RING - 1)] = 0;
    for (uint32_t p = e; p-- > a;) {
        const uint32_t choice = bg_dp_choose(c, p, e, ring);
        ring[p & (BG_DP_RING - 1)] = choice >> 11;
        if (p < b) bg_dp_commit(c, p, choice);
    }
}

/* phase 7: local accept + lazy rule -> stepcode (deflate_compress.c:2664-2670, 2723-2726, 2753-2756 restated
 * as a function of the matches at p, p+1, p+2 only, so that every position decides independently) */
BG_HD bool bg_match_ok(uint32_t r, uint32_t minlen)
{
    uint32_t len = r >> 16, off = bg_mw_off(r);
    return len >= minlen && len >= 3 && !(len == 3 && off > 8192);
}

BG_HD uint32_t bg_accept_code(uint32_t r0, uint32_t r1, uint32_t r2, uint32_t minlen, int lazy, uint32_t nice)
{
    if (!bg_match_ok(r0, minlen)) return 0;
    const uint32_t cl = r0 >> 16, co = bg_mw_off(r0);
    if (lazy >= 1 && cl < nice) {
        if (bg_match_ok(r1, minlen)) {
            const int nl = (int)(r1 >> 16);
            if (nl >= (int)cl && 4 * (nl - (int)cl) + (bg_bsr(co) - bg_bsr(bg_mw_off(r1))) > 2) return 0;
        }
        if (lazy >= 2 && bg_match_ok(r2, minlen)) {
            const int nl = (int)(r2 >> 16);
            if (nl >= (int)cl && 4 * (nl - (int)cl) + (bg_bsr(co) - bg_bsr(bg_mw_off(r2))) > 6) return 0;
        }
    }
    return cl <= 256 ? cl - 2 : 255;
}

/* Four consecutive positions per thread and step: their six match words come with two vector loads from the
 * L2-resident scratch, the four step codes leave as one shared-memory word. */
BG_HD void bg_phase_accept(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n, minlen = c.scal[BG_S_MINLEN];
    const int lazy = c.prm.lazy;
    const uint32_t nice = (uint32_t)c.prm.nice;
#if defined(__CUDA_ARCH__)
    /* the next step's loads are in flight while this step decides (the scratch is an L2 round trip away) */
    uint4 na = make_uint4(0, 0, 0, 0);
    uint2 nb = make_uint2(0, 0);
    if (4 * t < n) { na = __ldcg((const uint4 *)(c.R + 4 * t)); nb = __ldcg((const uint2 *)(c.R + 4 * t + 4)); }
#endif
    for (uint32_t p = 4 * t; p < n; p += 4 * T) {
        uint32_t r[6];
#if defined(__CUDA_ARCH__)
        const uint4 a = na;
        const uint2 b = nb;
        if (p + 4 * T < n) { na = __ldcg((const uint4 *)(c.R + p + 4 * T)); nb = __ldcg((const uint2 *)(c.R + p + 4 * T + 4)); }
        r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w; r[4] = b.x; r[5] = b.y;
#else
        for (uint32_t j = 0; j < 6; j++) r[j] = p + j < n ? c.R[p + j] : 0;
#endif
        uint32_t codes = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (uint32_t j = 0; j < 4; j++) {
            /* (what lies past the end of the block is no match) */
            const uint32_t r0 = p + j < n ? r[j] : 0, r1 = p + j + 1 < n ? r[j + 1] : 0, r2 = p + j + 2 < n ? r[j + 2] : 0;
            codes |= bg_accept_code(r0, r1, r2, minlen, lazy, nice) << (8 * j);
        }
        *(uint32_t *)(c.stepcode + p) = codes;
    }
}

/* history positions step one byte at a time, whatever the parse decided there: the walk then enters the payload exactly
 * at its first byte (run after bg_phase_accept / the min-cost passes; hist is a multiple of 4) */
BG_HD void bg_phase_history_steps(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t hw = bg_f_hist(c) >> 2;
    for (uint32_t i = t; i < hw; i += T) ((uint32_t *)c.stepcode)[i] = 0;
}

BG_HD uint32_t bg_step(const BgCtx &c, uint32_t p)
{
    uint32_t sc = c.stepcode[p];
    if (sc == 0) return 1;
    if (sc == 255) return c.R[p] >> 16;
    return sc + 2;
}

/* phase 8: per chunk, from the back: where does a parse entering at p leave the chunk? */
BG_HD void bg_phase_jump(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n;
    for (uint32_t ch = t; ch * BG_CHUNK < n; ch += T) {
        uint32_t s = ch * BG_CHUNK, e = s + BG_CHUNK;
        if (e > n) e = n;
        for (uint32_t p = e; p-- > s;) {
            uint32_t nx = p + bg_step(c, p);
            uint32_t j;
            if (nx >= e) { j = nx - e; if (j > 255) j = 255; }
            else j = c.jump8[nx];
            c.jump8[p] = (uint8_t)j;
        }
    }
}

/* phase 9: where does the parse enter each chunk?  Done in three short phases instead of one 1000-step walk:
 *   9a (all threads)  for every super-chunk (32 chunks) and every offset 0..257 at which a parse can enter it,
 *                     where does that parse leave it                                     -> xtab
 *   9b (thread 0)     chain the <= 31 super-chunks from position 0                        -> sentry
 *   9c (one thread per super-chunk) walk its 32 chunks from the true entry               -> entry */
BG_HD uint32_t bg_walk_chunks(const BgCtx &c, uint32_t e, uint32_t ch0, uint32_t ch1, uint16_t *entry)
{
    const uint32_t n = c.n;
    for (uint32_t ch = ch0; ch < ch1 && ch * BG_CHUNK < n; ch++) {
        uint32_t end = ch * BG_CHUNK + BG_CHUNK;
        if (end > n) end = n;
        if (e >= end) {
            if (entry) entry[ch] = BG_NOPOS;
            continue;
        }
        if (entry) entry[ch] = (uint16_t)(e - ch * BG_CHUNK);   /* chunk-relative: 65535 is a legal position */
        const uint32_t j = c.jump8[e];
        if (j == 255) {
            uint32_t q = e;
            while (q < end) q += bg_step(c, q);
            e = q;
        } else {
            e = end + j;
        }
    }
    return e;
}

/* 9-: which entry offsets can occur at all?  Offset k into super-chunk sc is possible only if some position in the
 * 258 before its start steps exactly onto it (or it is the very start of the block).  Typically a few dozen of the 258. */
BG_HD void bg_phase_walk_mark(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n;
    const uint32_t nsuper = (n + BG_SUPER_POS - 1) / BG_SUPER_POS;
    uint16_t *xtab = (uint16_t *)(c.regb + BG_B_XTAB);
    for (uint32_t w = t; w < nsuper * BG_MAX_TOKEN; w += T) {
        const uint32_t sc = w / BG_MAX_TOKEN, back = w - sc * BG_MAX_TOKEN + 1;    /* 1..258 positions before the start */
        const uint32_t start = sc * BG_SUPER_POS;
        if (sc == 0) {
            if (back == 1) xtab[0] = 0xFFFFu;
            continue;
        }
        const uint32_t q = start - back;           /* start >= 2176 > 258 */
        const uint32_t nx = q + bg_step(c, q);
        if (nx >= start && nx < start + BG_MAX_TOKEN) xtab[sc * BG_MAX_TOKEN + (nx - start)] = 0xFFFFu;   /* same value from all writers */
    }
}

BG_HD void bg_phase_walk_clear(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t nsuper = (c.n + BG_SUPER_POS - 1) / BG_SUPER_POS;
    uint16_t *xtab = (uint16_t *)(c.regb + BG_B_XTAB);
    for (uint32_t w = t; w < nsuper * BG_MAX_TOKEN; w += T) xtab[w] = 0;
    if (t == 0) c.scal[BG_S_WLIST] = 0;
}

/* possible entry w = (super-chunk, offset): where does a parse entering there leave the super-chunk */
BG_HD void bg_walk_entry(const BgCtx &c, uint32_t w)
{
    const uint32_t n = c.n;
    uint16_t *xtab = (uint16_t *)(c.regb + BG_B_XTAB);
    const uint32_t sc = w / BG_MAX_TOKEN, k = w - sc * BG_MAX_TOKEN;
    uint32_t send = (sc + 1) * BG_SUPER_POS;
    if (send > n) send = n;
    uint32_t e = sc * BG_SUPER_POS + k;
    if (e < send) e = bg_walk_chunks(c, e, sc * BG_SUPER, (sc + 1) * BG_SUPER, (uint16_t *)0);
    xtab[w] = (uint16_t)(e >= send ? e - send : 0);
}

/* 9a-: the possible entries (typically a thousand of the 8 000 table slots, in clusters) are gathered into a list so
 * that the walks of 9a spread evenly over the threads; what does not fit the list is walked on the spot */
#define BG_B_WLIST 1408u          /* u16[BG_WLIST_CAP], in histogram/Huffman space that is written only after the walk */
#define BG_WLIST_CAP 3400u
BG_HD void bg_phase_walk_list(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t nsuper = (c.n + BG_SUPER_POS - 1) / BG_SUPER_POS;
    const uint16_t *xtab = (const uint16_t *)(c.regb + BG_B_XTAB);
    uint16_t *list = (uint16_t *)(c.regb + BG_B_WLIST);
    for (uint32_t w = t; w < nsuper * BG_MAX_TOKEN; w += T) {
        if (xtab[w] != 0xFFFFu) continue;          /* not a possible entry */
        const uint32_t slot = bg_fetch_add32(&c.scal[BG_S_WLIST], 1);
        if (slot < BG_WLIST_CAP) list[slot] = (uint16_t)w;
        else bg_walk_entry(c, w);
    }
}

BG_HD void bg_phase_walk_a(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint16_t *list = (const uint16_t *)(c.regb + BG_B_WLIST);
    uint32_t m = c.scal[BG_S_WLIST];
    if (m > BG_WLIST_CAP) m = BG_WLIST_CAP;
    for (uint32_t i = t; i < m; i += T) bg_walk_entry(c, list[i]);
}

BG_HD void bg_phase_walk_b(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    if (t != 0) return;
    const uint32_t n = c.n;
    const uint32_t nsuper = (n + BG_SUPER_POS - 1) / BG_SUPER_POS;
    const uint16_t *xtab = (const uint16_t *)(c.regb + BG_B_XTAB);
    uint32_t *sentry = (uint32_t *)(c.regb + BG_B_SENTRY);
    uint32_t e = 0;
    for (uint32_t sc = 0; sc < nsuper; sc++) {
        uint32_t send = (sc + 1) * BG_SUPER_POS;
        if (send > n) send = n;
        sentry[sc] = e;
        if (e < send) e = send + xtab[sc * BG_MAX_TOKEN + (e - sc * BG_SUPER_POS)];
    }
    c.scal[BG_S_WALKEND] = e;   /* must equal n */
}

BG_HD void bg_phase_walk_c(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n;
    const uint32_t nsuper = (n + BG_SUPER_POS - 1) / BG_SUPER_POS;
    const uint32_t *sentry = (const uint32_t *)(c.regb + BG_B_SENTRY);
    uint16_t *entry = (uint16_t *)(c.regb + BG_B_ENTRY);
    /* spread the walkers over the warps: thread 32*sc of the block handles super-chunk sc */
    for (uint32_t sc = t / 32; sc < nsuper; sc += (T + 31) / 32)
        if ((t & 31u) == 0 || T < 32)
            bg_walk_chunks(c, sentry[sc], sc * BG_SUPER, (sc + 1) * BG_SUPER, entry);
}

/* phase 10: clear histograms (region B is free now) */
BG_HD void bg_phase_clear_freq(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint32_t *f = (uint32_t *)(c.regb + BG_B_LFREQ);
    for (uint32_t i = t; i < (BG_B_LLEN - BG_B_LFREQ) / 4; i += T)
        f[i] = 0;
    if (t == 0) { c.scal[BG_S_HM] = 0; c.scal[BG_S_DM] = 0; }
}

/* phase 11: tally symbols along the parse; remember match offsets in smem */
BG_HD void bg_phase_tally(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n;
    uint32_t *lfreq = (uint32_t *)(c.regb + BG_B_LFREQ);
    uint32_t *dfreq = (uint32_t *)(c.regb + BG_B_DFREQ);
    const uint16_t *entry = (const uint16_t *)(c.regb + BG_B_ENTRY);
    for (uint32_t i = t; i < BG_MAX_CHUNKS; i += T) {
        const uint32_t ch = c.perm ? c.perm[i] : i;
        if (ch * BG_CHUNK >= n || ch * BG_CHUNK < bg_f_hist(c)) continue;
        uint32_t p = entry[ch];
        if (p == BG_NOPOS) continue;
        p += ch * BG_CHUNK;
        uint32_t end = ch * BG_CHUNK + BG_CHUNK;
        if (end > n) end = n;
        while (p < end) {
            if ((p & 3u) == 0 && p + 4 <= end && *(const uint32_t *)(c.stepcode + p) == 0) {
                /* four literals in a row (sequence and quality text is full of them): one look at the step codes */
                const uint32_t d = c.dataw[p >> 2];
                bg_add32(&lfreq[d & 0xffu], 1);
                bg_add32(&lfreq[(d >> 8) & 0xffu], 1);
                bg_add32(&lfreq[(d >> 16) & 0xffu], 1);
                bg_add32(&lfreq[d >> 24], 1);
                p += 4;
            } else if (c.stepcode[p] == 0) {
                bg_add32(&lfreq[bg_ld8(c.dataw, p)], 1);
                p++;
            } else {
                uint32_t r = c.R[p], len = r >> 16, off = bg_mw_off(r), nb, ex;
                bg_add32(&lfreq[257 + bg_len_slot(len, &nb, &ex)], 1);
                bg_add32(&dfreq[bg_off_slot(off, &nb, &ex)], 1);
                c.offarr[p >> 1] = (uint16_t)(off - 1);
                p += len;
            }
        }
    }
    if (t == 0)
        bg_add32(&lfreq[256], 1);
}

/* phase 12: make sort keys for the litlen code (parallel) */
BG_HD void bg_phase_lkeys(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t *lfreq = (const uint32_t *)(c.regb + BG_B_LFREQ);
    uint32_t *keys = (uint32_t *)(c.regb + BG_B_KEYS);
    for (uint32_t i = t; i < 512; i += T) {
        const bool used = i < 288 && lfreq[i];
        keys[i] = used ? (lfreq[i] << 9) | i : 0xFFFFFFFFu;
        if (used) bg_add32(&c.scal[BG_S_HM], 1);       /* number of used litlen symbols (zeroed with the histograms) */
    }
}

/* ---- sequential Huffman pieces (one thread; arrays in shared memory) ---------------------------- */

/* Sort keys of the small alphabets (distance, precode), one thread per symbol: a used symbol's place is the number of used symbols with a smaller key
 * (keys are distinct: the symbol is part of the key).  Returns true for a used symbol (the caller counts them). */
BG_HD bool bg_rank_key(const uint32_t *freq, uint32_t nsym, uint32_t sym, uint32_t *keys)
{
    const uint32_t f = freq[sym];
    if (!f) return false;
    const uint32_t k = (f << 9) | sym;
    uint32_t rank = 0;
    for (uint32_t j = 0; j < nsym; j++) {
        const uint32_t fj = freq[j];
        rank += (fj != 0 && ((fj << 9) | j) < k) ? 1u : 0u;
    }
    keys[rank] = k;
    return true;
}

/* keys: ascending (freq<<9|sym) for the m used symbols.  lens[] must be zeroed by the caller.
 * Two-queue Huffman tree, depths clamped to maxbits with the classic overflow repair on the
 * per-length counts (the approach of zlib's gen_bitlen), longest codes to the rarest symbols. */
BG_HD void bg_huff_lengths(const uint32_t *keys, uint32_t m, uint32_t maxbits, uint32_t *w, uint16_t *par,
                           uint32_t *blc /* u32[16] scratch */, uint8_t *lens)
{
    if (m == 0) { lens[0] = 1; lens[1] = 1; return; }
    if (m == 1) {
        uint32_t s = keys[0] & 511u;
        lens[s] = 1;
        lens[s ? 0 : 1] = 1;
        return;
    }
    for (uint32_t i = 0; i < m; i++) w[i] = keys[i] >> 9;
    uint32_t a = 0, b = m, e = m;
    while (e < 2 * m - 1) {
        uint32_t x0, x1;
        if (a < m && (b >= e || w[a] <= w[b])) x0 = a++; else x0 = b++;
        if (a < m && (b >= e || w[a] <= w[b])) x1 = a++; else x1 = b++;
        w[e] = w[x0] + w[x1];
        par[x0] = (uint16_t)e;
        par[x1] = (uint16_t)e;
        e++;
    }
    for (uint32_t i = 0; i <= maxbits; i++) blc[i] = 0;
    int overflow = 0;
    w[e - 1] = 0;
    for (uint32_t i = e - 1; i-- > 0;) {
        uint32_t d = w[par[i]] + 1;
        if (d > maxbits) { d = maxbits; overflow++; }
        w[i] = d;
        if (i < m) blc[d]++;
    }
    while (overflow > 0) {
        uint32_t bits = maxbits - 1;
        while (blc[bits] == 0) bits--;
        blc[bits]--;
        blc[bits + 1] += 2;
        blc[maxbits]--;
        overflow -= 2;
    }
    uint32_t i = 0;
    for (uint32_t bits = maxbits; bits >= 1; bits--)
        for (uint32_t k = blc[bits]; k > 0; k--)
            lens[keys[i++] & 511u] = (uint8_t)bits;
}

/* canonical, bit-reversed codewords; scratch = u32[36] */
BG_HD void bg_huff_codes(const uint8_t *lens, uint32_t nsym, uint32_t maxbits, uint32_t *scratch, uint16_t *codes)
{
    uint32_t *count = scratch, *next = scratch + 18;
    for (uint32_t i = 0; i <= maxbits; i++) count[i] = 0;
    for (uint32_t s = 0; s < nsym; s++) count[lens[s]]++;
    count[0] = 0;
    uint32_t code = 0;
    for (uint32_t l = 1; l <= maxbits; l++) {
        code = (code + count[l - 1]) << 1;
        next[l] = code;
    }
    for (uint32_t s = 0; s < nsym; s++) {
        uint32_t l = lens[s];
        codes[s] = l ? (uint16_t)bg_brev(next[l]++, (int)l) : 0;
    }
}

/* run-length items over litlen+offset lengths (RFC 1951 3.2.7); returns item count, fills pfreq */
BG_HD uint32_t bg_header_items(const uint8_t *llen, uint32_t nl, const uint8_t *dlen, uint32_t nd, uint16_t *items,
                               uint32_t *pfreq)
{
    for (uint32_t i = 0; i < 19; i++) pfreq[i] = 0;
    const uint32_t total = nl + nd;
    uint32_t ni = 0, i = 0;
    while (i < total) {
        uint32_t v = i < nl ? llen[i] : dlen[i - nl];
        uint32_t j = i + 1;
        while (j < total && (j < nl ? llen[j] : dlen[j - nl]) == v) j++;
        uint32_t run = j - i;
        if (v == 0) {
            while (run >= 11) {
                uint32_t r = run > 138 ? 138 : run;
                items[ni++] = (uint16_t)(18 | ((r - 11) << 5));
                pfreq[18]++;
                run -= r;
            }
            if (run >= 3) {
                items[ni++] = (uint16_t)(17 | ((run - 3) << 5));
                pfreq[17]++;
                run = 0;
            }
        } else {
            items[ni++] = (uint16_t)v;
            pfreq[v]++;
            run--;
            while (run >= 3) {
                uint32_t r = run > 6 ? 6 : run;
                items[ni++] = (uint16_t)(16 | ((r - 3) << 5));
                pfreq[16]++;
                run -= r;
            }
        }
        while (run > 0) { items[ni++] = (uint16_t)v; pfreq[v]++; run--; }
        i = j;
    }
    return ni;
}

/* precode length order 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15 (RFC 1951 3.2.7), 5 bits each */
BG_HD uint32_t bg_precode_order(uint32_t i)
{
    const uint64_t lo = 16ull | 17ull << 5 | 18ull << 10 | 0ull << 15 | 8ull << 20 | 7ull << 25 | 9ull << 30 | 6ull << 35 |
                        10ull << 40 | 5ull << 45 | 11ull << 50 | 4ull << 55;
    const uint64_t hi = 12ull | 3ull << 5 | 13ull << 10 | 2ull << 15 | 14ull << 20 | 1ull << 25 | 15ull << 30;
    return (uint32_t)((i < 12 ? lo >> (5 * i) : hi >> (5 * (i - 12))) & 31u);
}

/* The two-queue merge of bg_huff_lengths() with the heads of both queues held in registers, so that picking the two
 * lightest nodes does not wait for shared memory (a node just made is often the very next one needed).  Same picks,
 * same ties (a leaf before an internal node of equal weight).  w[0..m) = leaf weights ascending; fills w[m..2m-1), par. */
BG_HD void bg_huff_merge(uint32_t m, uint32_t *w, uint16_t *par)
{
    const uint32_t none = 0xFFFFFFFFu;
    uint32_t a = 0, b = m, e = m;
    uint32_t wa = w[0], wb = none;
    while (e < 2 * m - 1) {
        uint32_t x0, x1, v0, v1;
        if (wa <= wb) { x0 = a; v0 = wa; a++; wa = a < m ? w[a] : none; }
        else { x0 = b; v0 = wb; b++; wb = b < e ? w[b] : none; }
        if (wa <= wb && wa != none) { x1 = a; v1 = wa; a++; wa = a < m ? w[a] : none; }
        else { x1 = b; v1 = wb; b++; wb = b < e ? w[b] : none; }
        const uint32_t v = v0 + v1;
        w[e] = v;
        par[x0] = (uint16_t)e;
        par[x1] = (uint16_t)e;
        if (b == e) wb = v;                     /* the internal queue had run empty: the new node is its head */
        e++;
    }
}

#define BG_B_BLC BG_B_SCRATCH           /* u32[16] litlen codewords per length */

/* phase 13a (parallel): leaf weights in sorted order, cleared lengths and counters */
BG_HD void bg_phase_huff_prep(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint8_t *rb = c.regb;
    const uint32_t *keys = (const uint32_t *)(rb + BG_B_KEYS);
    uint32_t *w = (uint32_t *)(rb + BG_B_TREEW);
    const uint32_t m = c.scal[BG_S_HM];
    for (uint32_t i = t; i < 288; i += T) {
        if (i < m) w[i] = keys[i] >> 9;
        rb[BG_B_LLEN + i] = 0;
    }
    if (t < 16) ((uint32_t *)(rb + BG_B_BLC))[t] = 0;
    if (t == 16 % T) c.scal[BG_S_HOVF] = 0;
    /* the distance alphabet's sort keys, one thread per symbol (BG_S_DM was zeroed with the histograms) */
    for (uint32_t sym = t; sym < 30; sym += T)
        if (bg_rank_key((const uint32_t *)(rb + BG_B_DFREQ), 30, sym, (uint32_t *)(rb + BG_B_DKEYS))) bg_add32(&c.scal[BG_S_DM], 1);
}

/* phase 13b: thread 0 merges the litlen tree, thread 32 builds the (small) distance code start to finish */
BG_HD void bg_phase_huff(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint8_t *rb = c.regb;
    if (t == 0) {
        const uint32_t *keys = (const uint32_t *)(rb + BG_B_KEYS);
        uint8_t *llen = rb + BG_B_LLEN;
        const uint32_t m = c.scal[BG_S_HM];
        if (m == 0) { llen[0] = 1; llen[1] = 1; }
        else if (m == 1) {
            const uint32_t s1 = keys[0] & 511u;
            llen[s1] = 1;
            llen[s1 ? 0 : 1] = 1;
        } else {
            bg_huff_merge(m, (uint32_t *)(rb + BG_B_TREEW), (uint16_t *)(rb + BG_B_TREEP));
        }
    }
    if (t == 32 % T) {
        uint32_t *dkeys = (uint32_t *)(rb + BG_B_DKEYS);
        uint8_t *dlen = rb + BG_B_DLEN;
        for (uint32_t i = 0; i < 32; i++) dlen[i] = 0;
        const uint32_t m = c.scal[BG_S_DM];
        bg_huff_lengths(dkeys, m, 15, (uint32_t *)(rb + BG_B_DTREEW), (uint16_t *)(rb + BG_B_DTREEP),
                        (uint32_t *)(rb + BG_B_SCRATCH) + 32, dlen);
    }
}

/* phase 13c (parallel): depth of every node by walking up to the root; leaves count into the per-length table, and
 * every node deeper than 15 counts as overflow — the sums the sequential pass of bg_huff_lengths() produces */
BG_HD void bg_phase_huff_depth(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint8_t *rb = c.regb;
    const uint32_t m = c.scal[BG_S_HM];
    if (m < 2) return;
    const uint16_t *par = (const uint16_t *)(rb + BG_B_TREEP);
    uint32_t *blc = (uint32_t *)(rb + BG_B_BLC);
    const uint32_t root = 2 * m - 2;
    for (uint32_t i = t; i < root; i += T) {
        uint32_t d = 0;
        for (uint32_t x = i; x != root && d < 2 * 288; x = par[x]) d++;     /* (the cap only matters if memory were corrupt) */
        if (d > 15) { d = 15; bg_add32(&c.scal[BG_S_HOVF], 1); }
        if (i < m) bg_add32(&blc[d], 1);
    }
}

/* phase 13d (thread 0): the overflow repair on the per-length counts (zlib's gen_bitlen) */
BG_HD void bg_phase_huff_fix(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    if (t != 0 || c.scal[BG_S_HM] < 2) return;
    uint32_t *blc = (uint32_t *)(c.regb + BG_B_BLC);
    int overflow = (int)c.scal[BG_S_HOVF];
    while (overflow > 0) {
        uint32_t bits = 14;
        while (bits > 1 && blc[bits] == 0) bits--;
        blc[bits]--;
        blc[bits + 1] += 2;
        blc[15]--;
        overflow -= 2;
    }
}

/* phase 13e (parallel): the i-th rarest symbol gets the i-th longest length */
BG_HD void bg_phase_huff_assign(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint8_t *rb = c.regb;
    const uint32_t m = c.scal[BG_S_HM];
    if (m < 2) return;
    const uint32_t *keys = (const uint32_t *)(rb + BG_B_KEYS);
    const uint32_t *blc = (const uint32_t *)(rb + BG_B_BLC);
    for (uint32_t i = t; i < m; i += T) {
        uint32_t bits = 15, cum = blc[15];
        while (cum <= i && bits > 1) cum += blc[--bits];
        rb[BG_B_LLEN + (keys[i] & 511u)] = (uint8_t)bits;
    }
}

/* phase 14: the dynamic header, in parallel.
 *   h1  trim trailing zero lengths (atomic max), symbol cost sums of the dynamic and the static code
 *   h2  one thread per code length: does a run start here?  (ballot words)
 *   h3  each run start measures its run and counts the run-length items it will emit  -> scan -> offsets
 *   h4  each run start writes its items and tallies the precode alphabet
 *   h5  thread 0: precode lengths, HCLEN, header bit count
 * The items are exactly those of the sequential rule in bg_header_items() (kept below as documentation and
 * for the emulator's cross-check). */
#define BG_B_RUNMASK BG_B_SCRATCH      /* u32[12] run-start ballots, one word per 32 code lengths */

BG_HD uint32_t bg_hdr_len_at(const BgCtx &c, uint32_t i, uint32_t nl)
{
    return i < nl ? c.regb[BG_B_LLEN + i] : c.regb[BG_B_DLEN + (i - nl)];
}

BG_HD void bg_phase_hdr1(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    uint8_t *rb = c.regb;
    const uint32_t *lfreq = (const uint32_t *)(rb + BG_B_LFREQ), *dfreq = (const uint32_t *)(rb + BG_B_DFREQ);
    const uint8_t *llen = rb + BG_B_LLEN, *dlen = rb + BG_B_DLEN;
    uint32_t dyn = 0, sta = 0, extra = 0;
    if (t < 286) {
        const uint32_t f = lfreq[t];
        dyn = f * llen[t];
        sta = f * bg_static_llen(t);
        if (t > 256) extra = f * bg_len_slot_extra_bits(t - 257);
        if (llen[t]) {
#if defined(__CUDA_ARCH__)
            atomicMax(&c.scal[BG_S_NL], t + 1);
#else
            if (c.scal[BG_S_NL] < t + 1) c.scal[BG_S_NL] = t + 1;
#endif
        }
    } else if (t < 316) {
        const uint32_t sym = t - 286, f = dfreq[sym];
        dyn = f * dlen[sym];
        sta = f * 5;
        extra = f * bg_off_slot_extra_bits(sym);
        if (dlen[sym]) {
#if defined(__CUDA_ARCH__)
            atomicMax(&c.scal[BG_S_ND], sym + 1);
#else
            if (c.scal[BG_S_ND] < sym + 1) c.scal[BG_S_ND] = sym + 1;
#endif
        }
    }
#if defined(__CUDA_ARCH__)
    dyn = __reduce_add_sync(0xffffffffu, dyn);
    sta = __reduce_add_sync(0xffffffffu, sta);
    extra = __reduce_add_sync(0xffffffffu, extra);
    if ((t & 31u) == 0 && t < 320) {
        atomicAdd(&c.scal[BG_S_DYNSYMS], dyn);
        atomicAdd(&c.scal[BG_S_STASYMS], sta);
        atomicAdd(&c.scal[BG_S_EXTRA], extra);
    }
#else
    c.scal[BG_S_DYNSYMS] += dyn;
    c.scal[BG_S_STASYMS] += sta;
    c.scal[BG_S_EXTRA] += extra;
#endif
    if (t < 20) ((uint32_t *)(rb + BG_B_PFREQ))[t] = 0;
    if (t == 20 % T) c.scal[BG_S_PM] = 0;
    if (t < 12) ((uint32_t *)(rb + BG_B_RUNMASK))[t] = 0;
}

BG_HD void bg_hdr_dims(const BgCtx &c, uint32_t *nl, uint32_t *nd)
{
    *nl = c.scal[BG_S_NL] < 257 ? 257 : c.scal[BG_S_NL];
    *nd = c.scal[BG_S_ND] < 1 ? 1 : c.scal[BG_S_ND];
}

BG_HD void bg_phase_hdr2(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    uint32_t nl, nd;
    bg_hdr_dims(c, &nl, &nd);
    const uint32_t total = nl + nd;
    bool start = false;
    if (t < total) start = t == 0 || bg_hdr_len_at(c, t, nl) != bg_hdr_len_at(c, t - 1, nl);
#if defined(__CUDA_ARCH__)
    const unsigned m = __ballot_sync(0xffffffffu, start);
    if ((t & 31u) == 0 && t < 352) ((uint32_t *)(c.regb + BG_B_RUNMASK))[t >> 5] = m;
#else
    if (start) ((uint32_t *)(c.regb + BG_B_RUNMASK))[t >> 5] |= 1u << (t & 31u);
#endif
}

/* run starting at i: its length, from the ballot words */
BG_HD uint32_t bg_hdr_run_len(const BgCtx &c, uint32_t i, uint32_t total)
{
    const uint32_t *mask = (const uint32_t *)(c.regb + BG_B_RUNMASK);
    uint32_t w = i >> 5;
    uint32_t m = mask[w] & ~((2u << (i & 31u)) - 1u);      /* starts above i in the same word */
    while (m == 0 && (w + 1) * 32 < total) m = mask[++w];
    const uint32_t next = m ? w * 32 + (uint32_t)bg_ctz(m) : total;
    return (next < total ? next : total) - i;
}

/* the sequential rule, as counts: how many items does a run (value v, length r) produce */
BG_HD uint32_t bg_hdr_run_items(uint32_t v, uint32_t r)
{
    if (v == 0) {
        const uint32_t full = r / 138, rem = r - full * 138;
        return full + (rem >= 3 ? 1 : rem);
    }
    const uint32_t r1 = r - 1, full = r1 / 6, rem = r1 - full * 6;
    return 1 + full + (rem >= 3 ? 1 : rem);
}

BG_HD void bg_phase_hdr3(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint32_t nl, nd;
    bg_hdr_dims(c, &nl, &nd);
    const uint32_t total = nl + nd;
    uint32_t *cnt = (uint32_t *)(c.regb + BG_B_CBITS);
    const uint32_t *mask = (const uint32_t *)(c.regb + BG_B_RUNMASK);
    for (uint32_t i = t; i < BG_MAX_CHUNKS; i += T) {
        uint32_t k = 0;
        if (i < total && ((mask[i >> 5] >> (i & 31u)) & 1u))
            k = bg_hdr_run_items(bg_hdr_len_at(c, i, nl), bg_hdr_run_len(c, i, total));
        cnt[i] = k;
    }
}

/* (the driver turns cnt[] into its exclusive prefix sum; the grand total is the item count) */

BG_HD void bg_phase_hdr4(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint32_t nl, nd;
    bg_hdr_dims(c, &nl, &nd);
    const uint32_t total = nl + nd;
    const uint32_t *off = (const uint32_t *)(c.regb + BG_B_CBITS);
    const uint32_t *mask = (const uint32_t *)(c.regb + BG_B_RUNMASK);
    uint16_t *items = (uint16_t *)(c.regb + BG_B_ITEMS);
    uint32_t *pfreq = (uint32_t *)(c.regb + BG_B_PFREQ);
    for (uint32_t i = t; i < total; i += T) {
        if (!((mask[i >> 5] >> (i & 31u)) & 1u)) continue;
        const uint32_t v = bg_hdr_len_at(c, i, nl);
        uint32_t run = bg_hdr_run_len(c, i, total), ni = off[i];
        if (v == 0) {
            while (run >= 11) {
                const uint32_t r = run > 138 ? 138 : run;
                items[ni++] = (uint16_t)(18 | ((r - 11) << 5));
                bg_add32(&pfreq[18], 1);
                run -= r;
            }
            if (run >= 3) {
                items[ni++] = (uint16_t)(17 | ((run - 3) << 5));
                bg_add32(&pfreq[17], 1);
                run = 0;
            }
        } else {
            items[ni++] = (uint16_t)v;
            bg_add32(&pfreq[v], 1);
            run--;
            while (run >= 3) {
                const uint32_t r = run > 6 ? 6 : run;
                items[ni++] = (uint16_t)(16 | ((r - 3) << 5));
                bg_add32(&pfreq[16], 1);
                run -= r;
            }
        }
        if (run) bg_add32(&pfreq[v], run);
        while (run > 0) { items[ni++] = (uint16_t)v; run--; }
    }
}

/* the precode alphabet's sort keys, one thread per symbol */
BG_HD void bg_phase_hdr4b(const BgCtx &c, uint32_t t, uint32_t T)
{
    for (uint32_t sym = t; sym < 19; sym += T)
        if (bg_rank_key((const uint32_t *)(c.regb + BG_B_PFREQ), 19, sym, (uint32_t *)(c.regb + BG_B_PKEYS))) bg_add32(&c.scal[BG_S_PM], 1);
}

BG_HD void bg_phase_hdr5(const BgCtx &c, uint32_t t, uint32_t T, uint32_t nitems)
{
    (void)T;
    if (t != 0) return;
    uint8_t *rb = c.regb;
    uint32_t nl, nd;
    bg_hdr_dims(c, &nl, &nd);
    const uint32_t *pfreq = (const uint32_t *)(rb + BG_B_PFREQ);
    uint8_t *plen = rb + BG_B_PLEN;
    uint32_t *pkeys = (uint32_t *)(rb + BG_B_PKEYS);
    for (uint32_t i = 0; i < 19; i++) plen[i] = 0;
    const uint32_t pm = c.scal[BG_S_PM];
    bg_huff_lengths(pkeys, pm, 7, (uint32_t *)(rb + BG_B_DTREEW), (uint16_t *)(rb + BG_B_DTREEP), (uint32_t *)(rb + BG_B_SCRATCH) + 16, plen);
    uint32_t np = 19;
    while (np > 4 && plen[bg_precode_order(np - 1)] == 0) np--;
    uint32_t hdr = 3 + 5 + 5 + 4 + 3 * np;
    for (uint32_t i = 0; i < 19; i++)
        hdr += pfreq[i] * (plen[i] + (i == 16 ? 2u : i == 17 ? 3u : i == 18 ? 7u : 0u));
    c.scal[BG_S_DYNHDR] = hdr;
    c.scal[BG_S_NITEMS] = nitems;
    c.scal[BG_S_NL] = nl;
    c.scal[BG_S_ND] = nd;
    c.scal[BG_S_NP] = np;
}

/* bytes of a coded block of `bits` bits; a non-final piece adds the empty stored block: 3 bits, padding, 00 00 ff ff */
BG_HD uint32_t bg_coded_bytes(const BgCtx &c, uint32_t bits) { return bg_f_final(c) ? (bits + 7) >> 3 : ((bits + 3 + 7) >> 3) + 4; }

/* block type from the exact costs: every thread evaluates the same few scalars */
BG_HD uint32_t bg_block_type(const BgCtx &c, uint32_t *hdrbits, uint32_t *tokbits, uint32_t *payload)
{
    const uint32_t n = c.n - bg_f_hist(c);                     /* payload bytes */
    const uint32_t hdr = c.scal[BG_S_DYNHDR], extra = c.scal[BG_S_EXTRA];
    const uint32_t dyn_bits = hdr + c.scal[BG_S_DYNSYMS] + extra;
    const uint32_t sta_bits = 3 + c.scal[BG_S_STASYMS] + extra;
    const uint32_t nstored = n ? (n + 65534u) / 65535u : 1u;
    const uint32_t sto_bits = 8 * (n + 5 * nstored);
    if (n != 0 && ((int)n <= c.prm.passthrough || (sto_bits <= sta_bits && sto_bits <= dyn_bits))) {
        *hdrbits = 0; *tokbits = 0; *payload = n + 5 * nstored;
        return 0;
    }
    if (sta_bits <= dyn_bits) {
        *hdrbits = 3; *tokbits = sta_bits - 3; *payload = bg_coded_bytes(c, sta_bits);
        return 1;
    }
    *hdrbits = hdr; *tokbits = dyn_bits - hdr; *payload = bg_coded_bytes(c, dyn_bits);
    return 2;
}

/* per-length counters / first codes of the three alphabets live in dead sort-key space */
#define BG_B_LCOUNT BG_B_KEYS            /* u32[16] litlen, u32[16] offset, u32[16] precode: counts per length */
#define BG_B_LFIRST (BG_B_KEYS + 192)    /* u32[16] x 3: first canonical codeword per length */

/* phase 14b: settle the block type; a static block swaps in the fixed code lengths; clear the counters */
BG_HD void bg_phase_decide_b(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    uint8_t *rb = c.regb;
    uint32_t hdrbits, tokbits, payload;
    const uint32_t btype = bg_block_type(c, &hdrbits, &tokbits, &payload);
    if (btype == 1) {
        if (t < 288) rb[BG_B_LLEN + t] = (uint8_t)bg_static_llen(t);
        if (t < 32) rb[BG_B_DLEN + t] = 5;
    }
    if (t < 96) ((uint32_t *)(rb + BG_B_LCOUNT))[t] = 0;
    if (t == 0) {
        c.scal[BG_S_BTYPE] = btype;
        c.scal[BG_S_HDRBITS] = hdrbits;
        c.scal[BG_S_TOKBITS] = tokbits;   /* includes the end-of-block symbol */
        c.scal[BG_S_PAYLOAD] = payload;
        c.scal[BG_S_STATUS] = (bg_f_hdr(c) + payload + bg_f_trl(c) > BG_SLOT_BYTES) ? 1u : 0u;
    }
}

/* which (alphabet, symbol) does thread t own: 0..287 litlen, 288..319 offset, 320..338 precode */
BG_HD bool bg_code_slot(const BgCtx &c, uint32_t t, uint32_t *alpha, uint32_t *sym, const uint8_t **lens, uint16_t **codes)
{
    uint8_t *rb = c.regb;
    if (t < 288) { *alpha = 0; *sym = t; *lens = rb + BG_B_LLEN; *codes = (uint16_t *)(rb + BG_B_LCODE); return true; }
    if (t < 320) { *alpha = 1; *sym = t - 288; *lens = rb + BG_B_DLEN; *codes = (uint16_t *)(rb + BG_B_DCODE); return true; }
    if (t < 339) { *alpha = 2; *sym = t - 320; *lens = rb + BG_B_PLEN; *codes = (uint16_t *)(rb + BG_B_PCODE); return true; }
    return false;
}

/* phase 14c: count codewords per length (one thread per symbol) */
BG_HD void bg_phase_codes_a(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    uint32_t alpha, sym;
    const uint8_t *lens;
    uint16_t *codes;
    if (c.scal[BG_S_BTYPE] == 0 || !bg_code_slot(c, t, &alpha, &sym, &lens, &codes)) return;
    const uint32_t l = lens[sym];
    if (l) bg_add32((uint32_t *)(c.regb + BG_B_LCOUNT) + 16 * alpha + l, 1);
}

/* phase 14d: first canonical codeword of every length (threads 0, 32, 64: one alphabet each) */
BG_HD void bg_phase_codes_b(const BgCtx &c, uint32_t t, uint32_t T)
{
    if (c.scal[BG_S_BTYPE] == 0) return;
    for (uint32_t alpha = 0; alpha < 3; alpha++) {
        if (t != (32 * alpha) % T) continue;
        const uint32_t *count = (const uint32_t *)(c.regb + BG_B_LCOUNT) + 16 * alpha;
        uint32_t *first = (uint32_t *)(c.regb + BG_B_LFIRST) + 16 * alpha;
        uint32_t code = 0, prevcount = 0;
        for (uint32_t l = 1; l <= 15; l++) {
            code = (code + prevcount) << 1;
            first[l] = code;
            prevcount = count[l];
        }
    }
}

/* phase 14e: codeword of symbol s = first[len] + (number of lower symbols with the same length), bit-reversed */
BG_HD void bg_phase_codes_c(const BgCtx &c, uint32_t t, uint32_t T)
{
    (void)T;
    uint32_t alpha, sym;
    const uint8_t *lens;
    uint16_t *codes;
    if (c.scal[BG_S_BTYPE] == 0 || !bg_code_slot(c, t, &alpha, &sym, &lens, &codes)) return;
    const uint32_t l = lens[sym];
    uint32_t code = 0;
    if (l) {
        uint32_t rank = 0;
        for (uint32_t j = 0; j < sym; j++) rank += lens[j] == l;
        code = bg_brev(((const uint32_t *)(c.regb + BG_B_LFIRST))[16 * alpha + l] + rank, (int)l);
    }
    codes[sym] = (uint16_t)code;
}

/* phase 14e': ready-made token tables for the two passes over the parse that follow (sizes, emit), in tree space that
 * is dead by now:  literal b -> code | bits << 24;  match length l -> (code | extra << codelen) | bits << 24;
 * offset slot s -> code | codelen << 24 */
#define BG_B_LITTAB BG_B_TREEW                 /* u32[256] */
#define BG_B_LENTAB (BG_B_TREEW + 1024u)       /* u32[260] (index = match length) */
#define BG_B_OFFTAB (BG_B_TREEW + 2064u)       /* u32[32]  */
BG_HD void bg_phase_tabs(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint8_t *rb = c.regb;
    if (c.scal[BG_S_BTYPE] == 0) return;
    const uint8_t *llen = rb + BG_B_LLEN, *dlen = rb + BG_B_DLEN;
    const uint16_t *lcode = (const uint16_t *)(rb + BG_B_LCODE), *dcode = (const uint16_t *)(rb + BG_B_DCODE);
    for (uint32_t i = t; i < 256 + 260 + 32; i += T) {
        if (i < 256) {
            ((uint32_t *)(rb + BG_B_LITTAB))[i] = (uint32_t)lcode[i] | ((uint32_t)llen[i] << 24);
        } else if (i < 516) {
            const uint32_t len = i - 256;
            uint32_t v = 0;
            if (len >= 3 && len <= 258) {
                uint32_t nb, ex;
                const uint32_t ls = 257 + bg_len_slot(len, &nb, &ex);
                v = ((uint32_t)lcode[ls] | (ex << llen[ls])) | ((llen[ls] + nb) << 24);
            }
            ((uint32_t *)(rb + BG_B_LENTAB))[len] = v;
        } else {
            const uint32_t sl = i - 516;
            ((uint32_t *)(rb + BG_B_OFFTAB))[sl] = sl < 30 ? (uint32_t)dcode[sl] | ((uint32_t)dlen[sl] << 24) : 0;
        }
    }
}

/* phase 14f: bits of every run-length item of the dynamic header (the driver turns them into bit offsets), so that
 * the header is written by one thread per item instead of one thread for all */
#define BG_B_IOFF BG_B_XTAB       /* u32[1024]; the walk tables are dead by now */
BG_HD void bg_phase_hdr_bits(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint8_t *plen = c.regb + BG_B_PLEN;
    const uint16_t *items = (const uint16_t *)(c.regb + BG_B_ITEMS);
    uint32_t *ioff = (uint32_t *)(c.regb + BG_B_IOFF);
    const uint32_t ni = c.scal[BG_S_BTYPE] == 2 ? c.scal[BG_S_NITEMS] : 0;
    for (uint32_t i = t; i < BG_MAX_CHUNKS; i += T) {
        uint32_t bits = 0;
        if (i < ni) {
            const uint32_t sym = items[i] & 31u;
            bits = plen[sym] + (sym < 16 ? 0u : sym == 16 ? 2u : sym == 17 ? 3u : 7u);
        }
        ioff[i] = bits;
    }
}

/* phase 15: bits per chunk with the final code */
BG_HD void bg_phase_sizes(const BgCtx &c, uint32_t t, uint32_t T)
{
    const uint32_t n = c.n;
    uint8_t *rb = c.regb;
    const uint32_t *littab = (const uint32_t *)(rb + BG_B_LITTAB), *lentab = (const uint32_t *)(rb + BG_B_LENTAB);
    const uint32_t *offtab = (const uint32_t *)(rb + BG_B_OFFTAB);
    const uint16_t *entry = (const uint16_t *)(rb + BG_B_ENTRY);
    uint32_t *cbits = (uint32_t *)(rb + BG_B_CBITS);
    const bool coded = c.scal[BG_S_BTYPE] != 0;
    for (uint32_t i = t; i < BG_MAX_CHUNKS; i += T) {
        const uint32_t ch = c.perm ? c.perm[i] : i;
        uint32_t bits = 0;
        uint32_t p = ch * BG_CHUNK < n && ch * BG_CHUNK >= bg_f_hist(c) ? entry[ch] : BG_NOPOS;
        if (coded && p != BG_NOPOS) {
            p += ch * BG_CHUNK;
            uint32_t end = ch * BG_CHUNK + BG_CHUNK;
            if (end > n) end = n;
            while (p < end) {
                if ((p & 3u) == 0 && p + 4 <= end && *(const uint32_t *)(c.stepcode + p) == 0) {
                    const uint32_t d = c.dataw[p >> 2];                 /* four literals in a row */
                    bits += (littab[d & 0xffu] >> 24) + (littab[(d >> 8) & 0xffu] >> 24) + (littab[(d >> 16) & 0xffu] >> 24) + (littab[d >> 24] >> 24);
                    p += 4;
                    continue;
                }
                uint32_t sc = c.stepcode[p];
                if (sc == 0) {
                    bits += littab[bg_ld8(c.dataw, p)] >> 24;
                    p++;
                } else {
                    uint32_t len = sc == 255 ? (c.R[p] >> 16) : sc + 2, nb, ex;
                    bits += lentab[len] >> 24;
                    bits += (offtab[bg_off_slot((uint32_t)c.offarr[p >> 1] + 1, &nb, &ex)] >> 24) + nb;
                    p += len;
                }
            }
        }
        cbits[ch] = bits;
    }
}

/* (between 15 and 16 the driver turns cbits[] into its exclusive prefix sum) */

/* phase 16: zero the output words this block will OR into */
BG_HD void bg_phase_zero_out(const BgCtx &c, uint32_t t, uint32_t T)
{
    uint32_t bytes = bg_f_hdr(c) + c.scal[BG_S_PAYLOAD] + bg_f_trl(c);
    if (bytes > BG_SLOT_BYTES) bytes = BG_SLOT_BYTES;
    uint32_t words = (bytes + 3) >> 2;
    for (uint32_t i = t; i < words; i += T)
        c.out[i] = 0;
}

struct BgWriter {
    uint32_t *out;
    uint32_t word;
    uint64_t acc;
    uint32_t nacc;
    bool shared;   /* the word being filled may also be written by a neighbour: OR it */
};

BG_HD void bg_w_init(BgWriter &w, uint32_t *out, uint32_t bitpos)
{
    w.out = out;
    w.word = bitpos >> 5;
    w.nacc = bitpos & 31u;
    w.acc = 0;
    w.shared = true;
}

BG_HD void bg_w_put(BgWriter &w, uint32_t val, uint32_t nbits)
{
    w.acc |= (uint64_t)val << w.nacc;
    w.nacc += nbits;
    if (w.nacc >= 32) {
        if (w.shared) bg_or32(&w.out[w.word], (uint32_t)w.acc);
        else w.out[w.word] = (uint32_t)w.acc;
        w.shared = false;
        w.word++;
        w.acc >>= 32;
        w.nacc -= 32;
    }
}

BG_HD void bg_w_flush(BgWriter &w)
{
    if (w.nacc > 0 && (uint32_t)w.acc != 0)
        bg_or32(&w.out[w.word], (uint32_t)w.acc);
}

/* framing: the member header, then CRC32 + ISIZE after the payload.  BGZF (bgzf_compress.c:191-196): 18 bytes, subfield
 * "BC" with BSIZE = member size - 1.  MiGz (applet/7migz.c:224-233): 20 bytes, subfield "MZ" with the DEFLATE size as u32. */
BG_HD void bg_emit_frame(const BgCtx &c)
{
    if (bg_f_piece(c)) return;                   /* the gaps stay zero: the host writes the container's framing */
    const uint32_t payload = c.scal[BG_S_PAYLOAD];
    const uint32_t total = bg_f_hdr(c) + payload + 8;
    BgWriter w;
    bg_w_init(w, c.out, 0);
    bg_w_put(w, 0x04088b1fu, 32);          /* 1f 8b 08 04 */
    bg_w_put(w, 0u, 32);                   /* MTIME */
    if (bg_f_hdr(c) == 18u) {
        bg_w_put(w, 0x0006ff00u, 32);      /* XFL 00, OS ff, XLEN 0006 */
        bg_w_put(w, 0x00024342u, 32);      /* 'B' 'C' SLEN 0002 */
        bg_w_put(w, (total - 1) & 0xffffu, 16);
    } else {
        bg_w_put(w, 0x0008ff00u, 32);      /* XFL 00, OS ff, XLEN 0008 */
        bg_w_put(w, 0x00045a4du, 32);      /* 'M' 'Z' SLEN 0004 */
        bg_w_put(w, payload, 32);
    }
    bg_w_flush(w);
    bg_w_init(w, c.out, (bg_f_hdr(c) + payload) * 8);
    bg_w_put(w, c.scal[BG_S_CRC], 32);
    bg_w_put(w, c.n - bg_f_hist(c), 32);
    bg_w_flush(w);
}

/* phase 17: write everything.  thread 0: frame + block header (+EOB); chunk threads: tokens;
 * stored blocks: all threads copy words. */
BG_HD void bg_phase_emit(const BgCtx &c, uint32_t t, uint32_t T)
{
    if (c.scal[BG_S_STATUS]) return;
    uint8_t *rb = c.regb;
    const uint32_t btype = c.scal[BG_S_BTYPE];
    const uint32_t base = bg_f_hdr(c) * 8;
    if (btype == 0) {
        /* stored: [01|00] LEN NLEN raw..., at most two stored blocks (n <= 65536) */
        const uint32_t hist = bg_f_hist(c), n = c.n - hist;   /* the payload: n bytes behind the history */
        const uint32_t first = n > 65535u ? 65535u : n;
        if (t == 0) {
            bg_emit_frame(c);
            BgWriter w;
            bg_w_init(w, c.out, base);
            bg_w_put(w, n > 65535u ? 0u : bg_f_final(c), 8);
            bg_w_put(w, first | ((~first & 0xffffu) << 16), 32);
            bg_w_flush(w);
            if (n > 65535u) {
                uint32_t rest = n - 65535u;
                bg_w_init(w, c.out, base + (5 + 65535u) * 8);
                bg_w_put(w, bg_f_final(c), 8);
                bg_w_put(w, rest | ((~rest & 0xffffu) << 16), 32);
                bg_w_flush(w);
            }
        }
        /* raw bytes: payload byte i lands at slot byte hdr+5+i (+5 more after the first 65535).
         * Output words whose four source bytes all lie in the first stored block are plain stores
         * of an unaligned read; the few bytes at either edge are OR-ed in one by one. */
        const uint32_t r0 = bg_f_hdr(c) + 5u;                        /* slot byte of payload byte 0 */
        const uint32_t w0 = (r0 + 3u) >> 2, hb = 4u * w0 - r0;  /* first full word; payload bytes before it */
        const uint32_t wend = (first + r0) >> 2;               /* first word that is not "full" */
        for (uint32_t wd = w0 + t; wd < wend; wd += T)
            c.out[wd] = bg_ld32(c.dataw, hist + 4 * wd - r0);
        const uint32_t s1 = wend > w0 ? 4 * wend - r0 : hb;    /* first source byte past the full words */
        if (t < hb + 15u) {
            uint32_t src = t < hb ? t : s1 + (t - hb);
            if (src < n) {
                uint32_t dst = r0 + src + (src >= 65535u ? 5 : 0);
                bg_or32(&c.out[dst >> 2], bg_ld8(c.dataw, hist + src) << (8 * (dst & 3)));
            }
        }
        return;
    }
    const uint8_t *llen = rb + BG_B_LLEN, *dlen = rb + BG_B_DLEN, *plen = rb + BG_B_PLEN;
    const uint16_t *lcode = (const uint16_t *)(rb + BG_B_LCODE), *dcode = (const uint16_t *)(rb + BG_B_DCODE);
    const uint16_t *pcode = (const uint16_t *)(rb + BG_B_PCODE), *items = (const uint16_t *)(rb + BG_B_ITEMS);
    const uint16_t *entry = (const uint16_t *)(rb + BG_B_ENTRY);
    const uint32_t *cbits = (const uint32_t *)(rb + BG_B_CBITS);
    const uint32_t *littab = (const uint32_t *)(rb + BG_B_LITTAB), *lentab = (const uint32_t *)(rb + BG_B_LENTAB);
    const uint32_t *offtab = (const uint32_t *)(rb + BG_B_OFFTAB);
    const uint32_t hdrbits = c.scal[BG_S_HDRBITS];
    const uint32_t n = c.n;
    if (t == 0) {
        bg_emit_frame(c);
        BgWriter w;
        bg_w_init(w, c.out, base);
        bg_w_put(w, bg_f_final(c) | (btype << 1), 3);
        if (btype == 2) {
            const uint32_t nl = c.scal[BG_S_NL], nd = c.scal[BG_S_ND], np = c.scal[BG_S_NP];
            bg_w_put(w, (nl - 257) | ((nd - 1) << 5) | ((np - 4) << 10), 14);
            for (uint32_t i = 0; i < np; i++)
                bg_w_put(w, plen[bg_precode_order(i)], 3);
        }
        bg_w_flush(w);
        /* end-of-block symbol closes the token stream */
        bg_w_init(w, c.out, base + hdrbits + c.scal[BG_S_TOKBITS] - llen[256]);
        bg_w_put(w, lcode[256], llen[256]);
        bg_w_flush(w);
        if (!bg_f_final(c)) {
            /* empty stored block: its three header bits and the padding are zeros already; LEN 0000, NLEN ffff close the piece */
            bg_w_init(w, c.out, (bg_f_hdr(c) + c.scal[BG_S_PAYLOAD] - 4u) * 8u);
            bg_w_put(w, 0xffff0000u, 32);
            bg_w_flush(w);
        }
    }
    if (btype == 2) {
        /* the run-length items of the dynamic header, one thread each, at the bit offsets of phase 14f */
        const uint32_t *ioff = (const uint32_t *)(rb + BG_B_IOFF);
        const uint32_t ni = c.scal[BG_S_NITEMS], ibase = base + 17 + 3 * c.scal[BG_S_NP];
        for (uint32_t i = t; i < ni; i += T) {
            const uint32_t sym = items[i] & 31u, ex = items[i] >> 5;
            BgWriter w;
            bg_w_init(w, c.out, ibase + ioff[i]);
            bg_w_put(w, pcode[sym], plen[sym]);
            if (sym >= 16) bg_w_put(w, ex, sym == 16 ? 2 : sym == 17 ? 3 : 7);
            bg_w_flush(w);
        }
    }
    for (uint32_t i = t; i < BG_MAX_CHUNKS; i += T) {
        const uint32_t ch = c.perm ? c.perm[i] : i;
        BG_ASSERT(ch < BG_MAX_CHUNKS);
        if (ch * BG_CHUNK >= n || ch * BG_CHUNK < bg_f_hist(c)) continue;
        uint32_t p = entry[ch];
        if (p == BG_NOPOS) continue;
        p += ch * BG_CHUNK;
        uint32_t end = ch * BG_CHUNK + BG_CHUNK;
        if (end > n) end = n;
        BG_ASSERT(p < end && (base + hdrbits + cbits[ch]) / 8u < BG_SLOT_BYTES);
        BgWriter w;
        bg_w_init(w, c.out, base + hdrbits + cbits[ch]);
        while (p < end) {
            /* every turn ends in the same two puts (the second one may be empty): the three kinds of token differ only in how
             * the two (value, bits) pairs are made, so the lanes of a warp are together again for the packing */
            uint32_t v1, n1, v2 = 0, n2 = 0;
            const uint32_t sc = c.stepcode[p];
            if ((p & 3u) == 0 && p + 4 <= end && *(const uint32_t *)(c.stepcode + p) == 0) {
                /* four literals in a row: two puts of two code words each (<= 30 bits) */
                const uint32_t d = c.dataw[p >> 2];
                const uint32_t e0 = littab[d & 0xffu], e1 = littab[(d >> 8) & 0xffu], e2 = littab[(d >> 16) & 0xffu], e3 = littab[d >> 24];
                const uint32_t l0 = e0 >> 24, l2 = e2 >> 24;
                v1 = (e0 & 0xffffffu) | ((e1 & 0xffffffu) << l0);
                n1 = l0 + (e1 >> 24);
                v2 = (e2 & 0xffffffu) | ((e3 & 0xffffffu) << l2);
                n2 = l2 + (e3 >> 24);
                p += 4;
            } else if (sc == 0) {
                const uint32_t e = littab[bg_ld8(c.dataw, p)];
                v1 = e & 0xffffffu;
                n1 = e >> 24;
                p++;
            } else {
                uint32_t len = sc == 255 ? (c.R[p] >> 16) : sc + 2, nb, ex;
                const uint32_t el = lentab[len];
                v1 = el & 0xffffffu;
                n1 = el >> 24;
                const uint32_t eo = offtab[bg_off_slot((uint32_t)c.offarr[p >> 1] + 1, &nb, &ex)];
                v2 = (eo & 0xffffffu) | (ex << (eo >> 24));
                n2 = (eo >> 24) + nb;
                p += len;
            }
            bg_w_put(w, v1, n1);
            bg_w_put(w, v2, n2);
        }
        bg_w_flush(w);
    }
}

#endif /* BGZF_BLOCK_H */
