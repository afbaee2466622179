/* bgzf_inflate_dev.h — the DEFLATE decoder pieces shared by the inflate kernels (bgzf_inflate.cu) and the whole-stream
 * gzip kernels (bgzf_gzip.cu): decode-table layout and builder, bit reader, error codes. */
#ifndef BGZF_INFLATE_DEV_H
#define BGZF_INFLATE_DEV_H
#include <cuda_runtime.h>
#include <stdint.h>

#include "bgzf_block.h"

#ifndef INF_LROOT
#define INF_LROOT 9     /* 9-bit litlen root + 512-byte window + 64 registers: 6.0 KB and one warp per member => 32 members per SM (the CTA limit) */
#endif
#define INF_DROOT 8
#define INF_LTAB ((1u << INF_LROOT) + 352u)   /* litlen root + sub-tables (valid codes need <= 1334 with a 10-bit root, 852 with 9) */
#define INF_DTAB (256 + 160)    /* offset root + sub-tables (valid codes need <= 402) */
#define INF_PTAB 128
#define INF_WARPS_PER_CTA 1

/* decode-table entry: [3:0] bits to consume, [7:4] extra-bit count, [10:8] kind, [15:11] sub-table bits,
 * [31:16] value (literal / base length / base offset / sub-table start).  0 = invalid. */
#define K_LIT 1u
#define K_BASE 2u
#define K_EOB 3u
#define K_SUB 4u
#define F_LIT 0x8000u    /* literal entry (also set on LIT2) */
#define F_LIT2 0x4000u   /* two literals: value = lit1 | lit2 << 8, [3:0] total bits, [7:4] bits of the first */
#define ENT(nb, xb, kind, sb, val) ((uint32_t)(nb) | ((uint32_t)(xb) << 4) | ((uint32_t)(kind) << 8) | ((uint32_t)(sb) << 11) | ((uint32_t)(val) << 16))

/* per-member error codes (status[]) */
#define INF_OK 0u
#define INF_E_HEADER 1u     /* not a BGZF member header */
#define INF_E_BTYPE 2u      /* reserved block type */
#define INF_E_CODE 3u       /* over-subscribed / unusable Huffman code */
#define INF_E_SYMBOL 4u     /* invalid codeword in the data */
#define INF_E_DIST 5u       /* offset reaches before the start of the member */
#define INF_E_OVERRUN 6u    /* more output than ISIZE / input exhausted */
#define INF_E_STORED 7u     /* LEN != ~NLEN */
#define INF_E_SHORT 8u      /* output shorter than ISIZE */

#ifndef INF_WIN
#define INF_WIN 512u             /* bytes of recent output kept in shared memory per member (power of two) */
#endif

struct InfSmem {
    uint32_t ltab[INF_LTAB];
    uint32_t dtab[INF_DTAB];      /* the precode table (128 entries) borrows the start of this while lengths are read */
    uint32_t offs[16];
    uint8_t lens[320 + 16];
    uint32_t win[INF_WIN / 4];    /* circular window of the output, indexed by absolute address & (INF_WIN-1) */
};

/* Bit reader: all 32 lanes hold identical state.  The stream is fetched as coalesced 128-byte chunks (one word per
 * lane) and handed out with __shfl_sync; the reader keeps two consecutive words in registers and exposes the next
 * 32 bits of the stream with one funnel shift (no 64-bit arithmetic on the decode path). */
struct BitReader {
    const uint32_t *base;   /* word-aligned start */
    uint32_t nwords;        /* words that may be read (beyond: zeros) */
    uint32_t chunk;         /* this lane's word of the chunk that holds word wi+1 */
    uint32_t lane;
    uint32_t w0, w1;        /* words wi and wi+1 */
    uint32_t wi;
    uint32_t bit;           /* next unread bit inside w0, 0..31 */
    uint32_t skip;          /* bits of the first word that precede the start */
    uint32_t avail;         /* real input bits from the start to the end of the DEFLATE data */
};

__device__ __forceinline__ uint32_t br_fetch(BitReader &r, uint32_t idx)
{
    if ((idx & 31u) == 0u || idx == 0u) {
        const uint32_t i = (idx & ~31u) + r.lane;
        r.chunk = i < r.nwords ? __ldg(r.base + i) : 0u;
    }
    return __shfl_sync(0xffffffffu, r.chunk, idx & 31u);
}

__device__ __forceinline__ void br_init(BitReader &r, const uint8_t *p, const uint8_t *end, uint32_t lane)
{
    const uint32_t mis = (uint32_t)((uintptr_t)p & 3u);
    r.base = (const uint32_t *)(p - mis);
    r.nwords = (uint32_t)(((end - (p - mis)) + 3) >> 2);
    r.lane = lane;
    r.skip = 8 * mis;
    r.avail = (uint32_t)(end - p) * 8u;
    r.wi = 0;
    r.bit = r.skip;
    r.w0 = br_fetch(r, 0);
    r.w1 = br_fetch(r, 1);
}

/* the next 32 bits of the stream */
__device__ __forceinline__ uint32_t br_window(const BitReader &r) { return __funnelshift_r(r.w0, r.w1, r.bit); }

/* n <= 32 */
__device__ __forceinline__ void br_consume(BitReader &r, uint32_t n)
{
    r.bit += n;
    if (r.bit >= 32u) {
        r.bit -= 32u;
        r.w0 = r.w1;
        r.wi++;
        r.w1 = br_fetch(r, r.wi + 1);
    }
}
__device__ __forceinline__ uint32_t br_take(BitReader &r, uint32_t n)
{
    const uint32_t v = br_window(r) & ((n >= 32u) ? 0xffffffffu : ((1u << n) - 1u));
    br_consume(r, n);
    return v;
}
/* true once more bits were consumed than the member holds (the reference's overread check,
 * decompress_template.h: "overread_count <= bitsleft>>3") */
__device__ __forceinline__ bool br_overrun(const BitReader &r) { return r.wi * 32u + r.bit - r.skip > r.avail; }

__device__ __forceinline__ uint32_t litlen_entry(uint32_t sym, uint32_t nb)
{
    if (sym < 256) return ENT(nb, 0, K_LIT, 0, sym) | F_LIT;
    if (sym == 256) return ENT(nb, 0, K_EOB, 0, 0);
    if (sym > 285) sym = 285;   /* 286/287 decode as length 258, as in the reference's litlen_decode_results */
    const uint32_t s = sym - 257;
    uint32_t xb = bg_len_slot_extra_bits(s);
    uint32_t base = s < 8 ? 3 + s : s == 28 ? 258 : 3 + ((4 + (s & 3)) << xb);
    return ENT(nb, xb, K_BASE, 0, base);
}
__device__ __forceinline__ uint32_t offset_entry(uint32_t sym, uint32_t nb)
{
    if (sym > 29) sym = 29;     /* 30/31 decode like 29, as in the reference's offset_decode_results */
    uint32_t xb = bg_off_slot_extra_bits(sym);
    uint32_t base = sym < 4 ? 1 + sym : 1 + ((2 + (sym & 1)) << xb);
    return ENT(nb, xb, K_BASE, 0, base);
}

/*
 * Build a root+sub-table decoder for the canonical code given by lens[0..nsym) (warp-cooperative).
 * kind: 0 litlen, 1 offset, 2 precode.  Returns false for an over-subscribed code or table overflow.
 * Incomplete codes follow the reference's rule (only the empty code and a lone 1-bit codeword are valid).
 */
static __device__ bool build_table(const uint8_t *lens, uint32_t nsym, uint32_t root, uint32_t *tab, uint32_t cap, int kind,
                            uint32_t *offs, uint32_t lane)
{
    /* 1. per-length counts: lane l counts codewords of length l */
    uint32_t cnt = 0;
    if (lane >= 1 && lane <= 15)
        for (uint32_t s = 0; s < nsym; s++) cnt += (lens[s] == lane);
    /* 2. first code per length, Kraft check, longest length (uniform, via shuffles) */
    uint32_t code = 0, maxlen = 0, prevcnt = 0;
    int left = 1;
    bool bad = false;
    uint32_t myfirst = 0;
    for (uint32_t l = 1; l <= 15; l++) {
        const uint32_t cl = __shfl_sync(0xffffffffu, cnt, l);
        code = (code + prevcnt) << 1;
        if (lane == l) myfirst = code;
        prevcnt = cl;
        left = (left << 1) - (int)cl;
        if (left < 0) bad = true;
        if (cl) maxlen = l;
    }
    if (bad) return false;
    if (left > 0) {
        /* incomplete code: the reference (deflate_decompress.c:799-853) accepts only the empty code and a lone
         * 1-bit codeword, and lets both bit values decode to that symbol */
        const uint32_t c1 = __shfl_sync(0xffffffffu, cnt, 1);
        uint32_t sym = 0;
        if (maxlen != 0) {
            if (maxlen != 1 || c1 != 1) return false;
            for (uint32_t s = 0; s < nsym; s++) if (lens[s] == 1) sym = s;
        }
        const uint32_t e = kind == 0 ? litlen_entry(sym, 1) : kind == 1 ? offset_entry(sym, 1) : ENT(1, 0, K_LIT, 0, sym);
        for (uint32_t i = lane; i < (1u << root); i += 32) tab[i] = e;
        __syncwarp();
        return true;
    }
    if (lane >= 1 && lane <= 15) offs[lane] = myfirst;
    for (uint32_t i = lane; i < cap; i += 32) tab[i] = 0;
    __syncwarp();

    /* 3. pass 1: short codes fill the root; long codes leave the longest length seen under their root prefix */
    for (uint32_t b0 = 0; b0 < nsym; b0 += 32) {
        const uint32_t sym = b0 + lane;
        const uint32_t L = sym < nsym ? lens[sym] : 0u;
        const unsigned grp = __match_any_sync(0xffffffffu, L);
        const uint32_t rank = __popc(grp & ((1u << lane) - 1u));
        const uint32_t first = offs[L & 15u];
        __syncwarp();
        if (L && rank == 0) offs[L] = first + __popc(grp);
        __syncwarp();
        if (L) {
            const uint32_t rev = __brev(first + rank) >> (32 - L);
            if (L <= root) {
                const uint32_t e = kind == 0 ? litlen_entry(sym, L) : kind == 1 ? offset_entry(sym, L) : ENT(L, 0, K_LIT, 0, sym);
                for (uint32_t i = rev; i < (1u << root); i += (1u << L)) tab[i] = e;
            } else {
                atomicMax(&tab[rev & ((1u << root) - 1u)], L);
            }
        }
    }
    __syncwarp();
    if (maxlen <= root) return true;

    /* 4. allocate sub-tables in root-index order (warp scan over the markers) */
    uint32_t next = 1u << root;
    for (uint32_t b0 = 0; b0 < (1u << root); b0 += 32) {
        const uint32_t v = tab[b0 + lane];
        const bool marker = v > root && v <= 15;   /* valid entries are >= 256 */
        const uint32_t sz = marker ? 1u << (v - root) : 0u;
        uint32_t inc = sz;
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= (uint32_t)d) inc += y;
        }
        if (marker) tab[b0 + lane] = ENT(root, 0, K_SUB, v - root, next + inc - sz);
        next += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (next > cap) return false;
    __syncwarp();
    /* restore the canonical first codes consumed in pass 1 */
    if (lane >= 1 && lane <= 15) offs[lane] = myfirst;
    __syncwarp();

    /* 5. pass 2: long codes fill their sub-tables */
    for (uint32_t b0 = 0; b0 < nsym; b0 += 32) {
        const uint32_t sym = b0 + lane;
        const uint32_t L = sym < nsym ? lens[sym] : 0u;
        const unsigned grp = __match_any_sync(0xffffffffu, L);
        const uint32_t rank = __popc(grp & ((1u << lane) - 1u));
        const uint32_t first = offs[L & 15u];
        __syncwarp();
        if (L && rank == 0) offs[L] = first + __popc(grp);
        __syncwarp();
        if (L > root) {
            const uint32_t rev = __brev(first + rank) >> (32 - L);
            const uint32_t pe = tab[rev & ((1u << root) - 1u)];
            const uint32_t sb = (pe >> 11) & 31u, start = pe >> 16;
            const uint32_t e = kind == 0 ? litlen_entry(sym, L - root) : offset_entry(sym, L - root);
            for (uint32_t i = rev >> root; i < (1u << sb); i += (1u << (L - root))) tab[start + i] = e;
        }
    }
    __syncwarp();
    return true;
}

/* Root entries whose literal leaves room for a second literal inside the root index get both: the decoder then
 * emits two bytes per lookup on literal runs (most of FASTQ/SAM text under a long-match parse is literals).
 * A paired entry still carries its first literal and that literal's length, so lanes may read entries that
 * other lanes have already paired. */
static __device__ void pair_literals(uint32_t *tab, uint32_t root, uint32_t lane)
{
    for (uint32_t i = lane; i < (1u << root); i += 32) {
        const uint32_t e1 = tab[i];
        if (!(e1 & F_LIT)) continue;
        const uint32_t nb1 = (e1 & F_LIT2) ? ((e1 >> 4) & 15u) : (e1 & 15u);
        if (nb1 >= root) continue;
        const uint32_t e2 = tab[i >> nb1];
        if (!(e2 & F_LIT)) continue;
        const uint32_t nb2 = (e2 & F_LIT2) ? ((e2 >> 4) & 15u) : (e2 & 15u);
        if (nb1 + nb2 > root) continue;      /* the second codeword must lie wholly inside the index bits */
        const uint32_t lit1 = (e1 >> 16) & 0xffu, lit2 = (e2 >> 16) & 0xffu;
        tab[i] = (nb1 + nb2) | (nb1 << 4) | (K_LIT << 8) | F_LIT | F_LIT2 | ((lit1 | (lit2 << 8)) << 16);
    }
    __syncwarp();
}

/* decode one symbol from the 32-bit window; *nb = codeword bits (root + sub-table part) */
__device__ __forceinline__ uint32_t lookup(const uint32_t *tab, uint32_t root, uint32_t win, uint32_t *nb)
{
    uint32_t e = tab[win & ((1u << root) - 1u)];
    uint32_t used = 0;
    if (((e >> 8) & 7u) == K_SUB) {
        e = tab[(e >> 16) + ((win >> root) & ((1u << ((e >> 11) & 31u)) - 1u))];
        used = root;
    }
    *nb = used + (e & 15u);
    return e;
}

#endif
