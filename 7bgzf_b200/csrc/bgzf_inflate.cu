/*
 * bgzf_inflate.cu — sm_100a BGZF inflate kernels.
 *
 *   bgzf_inflate_kernel : one CTA (= one warp) per BGZF member, ~10 KiB of shared memory each, so ~22 members
 *       decode concurrently per SM; the last 2 KiB of output live in a shared-memory window (near back-references
 *       never leave the SM, output leaves as whole 128-byte lines).  All 32 lanes run the bit reader in lock-step (uniform control flow,
 *       broadcast LUT reads); the compressed bytes arrive as coalesced 128-byte chunks, one word per lane,
 *       and are handed to the reader with __shfl_sync; back-references are copied by all lanes.
 *       Table-driven Huffman decode from shared-memory LUTs: 10-bit root + sub-tables for the litlen code,
 *       8-bit root + sub-tables for the offset code, 7-bit precode table.
 *   bgzf_index_* : finds the members of a device-resident BGZF stream in parallel (signature scan, ordered
 *       compaction, BSIZE chain validation, exclusive scan of ISIZE) — the device form of the applet's
 *       header walk.
 *
 * Replaces in the reference: applet/7bgzf.c:295-365 (_decompress), :81-131 (_read_gz_header),
 * lib/zlibutil.c:82-93,194-204 (auto_inflate -> libdeflate_inflate), lib/libdeflate/deflate_decompress.c:721-1004
 * (build_decode_table) and decompress_template.h:44-772 (the decode loop).  Any valid DEFLATE stream is
 * accepted (stored / static / dynamic, several blocks per member); malformed input yields a per-member
 * error code, never an out-of-bounds write.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <atomic>

#include "bgzf_block.h"
#include "bgzf_inflate_dev.h"
#include "bgzf_kernels.h"

/* Output side of the decoder.  Every byte is first written to the shared-memory window (so that near
 * back-references cost a shared-memory read, not an L2 round trip) and leaves for global memory as whole
 * 128-byte lines, one 4-byte store per lane, as soon as a line is complete.  `apos` counts bytes from the
 * 128-byte-aligned address at or below the member's first output byte. */
struct OutWin {
    uint8_t *gline;      /* 128-byte aligned global base (gline + apos = address of output byte) */
    uint8_t *win;
    uint32_t first;      /* apos of the member's first byte (0..127) */
    uint32_t end;        /* apos one past the member's last byte (first + ISIZE): nothing at or beyond it is stored */
    uint32_t apos;       /* apos of the next byte to produce */
    uint32_t flushed;    /* lines below this index are in global memory */
    uint32_t lane;
};

__device__ __forceinline__ void ow_flush_lines(OutWin &o, uint32_t upto_line)
{
    /* lines [flushed, upto_line) are complete in the window */
    for (uint32_t L = o.flushed; L < upto_line; L++) {
        const uint32_t a = L * 128u + o.lane * 4u;
        const uint32_t v = *(const uint32_t *)(o.win + (a & (INF_WIN - 1u)));
        if (a >= o.first && a + 4 <= o.end) {
            *(uint32_t *)(o.gline + a) = v;                /* whole word belongs to this member */
        } else {
            for (uint32_t k = 0; k < 4; k++)               /* ragged first / last word */
                if (a + k >= o.first && a + k < o.end) o.gline[a + k] = (uint8_t)(v >> (8 * k));
        }
    }
    o.flushed = upto_line;
}

/* Literals are not checked against the end of the output one by one: the window is circular, so a corrupt stream
 * can do no harm there, and what leaves for global memory is clipped to the member.  The check happens here, when a
 * line completes (at most 128 + 258 bytes late).  Returns true when the stream has produced more than ISIZE.
 * (Running past the INPUT is only tested at the end of a block: beyond it the reader yields zeros, which a corrupt member
 * decodes until its ISIZE claim is used up.  Testing it here as well cost 1.5 % of the kernel, on every match 4 %; instead the
 * host bounds every claim by DEFLATE's maximum expansion of the member's input — b200bgzf_api.cu — so that a corrupt member
 * costs no more than a legitimate one of its size can.) */
__device__ __forceinline__ bool ow_advance(OutWin &o, uint32_t nbytes)
{
    o.apos += nbytes;
    const uint32_t complete = o.apos >> 7;
    if (complete != o.flushed) {
        __syncwarp();
        ow_flush_lines(o, complete);
        return o.apos > o.end;
    }
    return false;
}

/* the tail that never completed a line */
__device__ __forceinline__ void ow_finish(OutWin &o)
{
    __syncwarp();
    const uint32_t base = o.flushed * 128u;
    const uint32_t stop = o.apos < o.end ? o.apos : o.end;
    for (uint32_t a = (base > o.first ? base : o.first) + o.lane; a < stop; a += 32)
        o.gline[a] = o.win[a & (INF_WIN - 1u)];
}

#ifndef INF_MINCTAS
#define INF_MINCTAS 32
#endif
__global__ void __launch_bounds__(32 * INF_WARPS_PER_CTA, INF_MINCTAS)
bgzf_inflate_kernel(BgzfInflateArgs a)
{
    __shared__ InfSmem sm;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t m = blockIdx.x;
    if (m >= a.nblocks) return;

    const uint8_t *mem = a.in + a.in_off[m];
    uint32_t err = INF_OK;
    uint32_t msize, hlen;
    if (a.hdr_len) {
        /* the host has parsed the header (BGZF, MiGz, mgzip: applet/7bgzf.c:81-131) */
        hlen = a.hdr_len[m];
        msize = a.msize[m];
    } else {
        /* header: 1f 8b 08 04 .... XLEN=6 'B' 'C' 02 00 BSIZE */
        const bool hdr_ok = mem[0] == 0x1f && mem[1] == 0x8b && mem[2] == 8 && (mem[3] & 4) && mem[10] == 6 && mem[11] == 0 &&
                            mem[12] == 'B' && mem[13] == 'C' && mem[14] == 2 && mem[15] == 0;
        if (!hdr_ok) {
            if (lane == 0) { a.status[m] = INF_E_HEADER; atomicOr(a.err_flag, 1u); }
            return;
        }
        hlen = 18;
        msize = ((uint32_t)mem[16] | ((uint32_t)mem[17] << 8)) + 1u;
    }
    if (msize < hlen + 8u && !(a.unit_isize && a.unit_isize[m] != 0xffffffffu && msize >= hlen)) {
        if (lane == 0) { a.status[m] = INF_E_HEADER; atomicOr(a.err_flag, 1u); }
        return;
    }
    /* a piece (unit_isize given and not ~0): raw DEFLATE data without a trailer, e.g. one dictzip chunk or RAZF block; it is
     * complete when it has produced its share of the output at a block boundary (its blocks are not final: the reference
     * clears the bit and appends an empty stored block, applet/7dictzip.c:92-126) */
    const bool piece = a.unit_isize && a.unit_isize[m] != 0xffffffffu;
    const uint8_t *trailer = piece ? mem + msize : mem + msize - 8;
    const uint32_t isize = piece ? a.unit_isize[m]
                                 : (uint32_t)trailer[4] | ((uint32_t)trailer[5] << 8) | ((uint32_t)trailer[6] << 16) | ((uint32_t)trailer[7] << 24);
    uint8_t *out = a.out + a.out_off[m];
    if (!a.hdr_len && isize > 65536u) {                 /* (a BGZF payload is at most 64 KiB; other containers' members may be larger) */
        if (lane == 0) { a.status[m] = INF_E_HEADER; atomicOr(a.err_flag, 1u); }
        return;
    }

    BitReader r;
    br_init(r, mem + hlen, trailer, lane);
    OutWin o;
    o.first = (uint32_t)((uintptr_t)out & 127u);
    o.gline = out - o.first;
    o.win = (uint8_t *)sm.win;
    o.apos = o.first;
    o.end = o.first + isize;
    o.flushed = 0;
    o.lane = lane;
    const uint32_t end_apos = o.end;
    bool last = false;
    uint32_t nblk = 0;
    while (!last && err == INF_OK && !(piece && nblk && o.apos == end_apos)) {
        nblk++;
        last = br_take(r, 1);
        const uint32_t btype = br_take(r, 2);
        if (btype == 0) {
            /* stored: drop to a byte boundary, LEN, NLEN, raw bytes */
            br_consume(r, (8u - (r.bit & 7u)) & 7u);
            const uint32_t len = br_take(r, 16);
            const uint32_t nlen = br_take(r, 16);
            if ((len ^ nlen) != 0xffffu) { err = INF_E_STORED; break; }
            if (o.apos + len > end_apos) { err = INF_E_OVERRUN; break; }
            const uint8_t *raw = (const uint8_t *)(r.base + r.wi) + (r.bit >> 3);
            if (raw + len > trailer) { err = INF_E_OVERRUN; break; }
            for (uint32_t done = 0; done < len; done += 32) {
                const uint32_t k = done + lane;
                if (k < len) o.win[(o.apos + lane) & (INF_WIN - 1u)] = raw[k];
                ow_advance(o, len - done < 32 ? len - done : 32);
            }
            __syncwarp();
            if (!last) br_init(r, raw + len, trailer, lane);
            continue;
        }
        if (btype == 3) { err = INF_E_BTYPE; break; }
        if (btype == 1) {
            for (uint32_t i = lane; i < 288; i += 32) sm.lens[i] = (uint8_t)bg_static_llen(i);
            sm.lens[288 + lane] = 5;
            __syncwarp();
            if (!build_table(sm.lens, 288, INF_LROOT, sm.ltab, INF_LTAB, 0, sm.offs, lane) ||
                !build_table(sm.lens + 288, 32, INF_DROOT, sm.dtab, INF_DTAB, 1, sm.offs, lane)) { err = INF_E_CODE; break; }
            pair_literals(sm.ltab, INF_LROOT, lane);
        } else {
            const uint32_t nl = br_take(r, 5) + 257, nd = br_take(r, 5) + 1, np = br_take(r, 4) + 4;
            if (lane < 19) sm.lens[lane] = 0;
            __syncwarp();
            for (uint32_t i = 0; i < np; i++) {
                const uint32_t v = br_take(r, 3);
                if (lane == 0) sm.lens[bg_precode_order(i)] = (uint8_t)v;
            }
            __syncwarp();
            if (!build_table(sm.lens, 19, 7, sm.dtab, INF_PTAB, 2, sm.offs, lane)) { err = INF_E_CODE; break; }
            /* code lengths for litlen + offset, run-length coded */
            uint32_t i = 0, prevlen = 0;
            const uint32_t total = nl + nd;
            while (i < total) {
                const uint32_t e = sm.dtab[br_window(r) & 127u];
                if (e == 0) { err = INF_E_SYMBOL; break; }
                br_consume(r, e & 15u);
                const uint32_t sym = e >> 16;
                uint32_t rep, val;
                if (sym < 16) { rep = 1; val = sym; prevlen = sym; }
                else if (sym == 16) { if (i == 0) { err = INF_E_CODE; break; } rep = 3 + br_take(r, 2); val = prevlen; }
                else if (sym == 17) { rep = 3 + br_take(r, 3); val = 0; prevlen = 0; }
                else { rep = 11 + br_take(r, 7); val = 0; prevlen = 0; }
                if (i + rep > total) { err = INF_E_CODE; break; }
                for (uint32_t k = lane; k < rep; k += 32) sm.lens[i + k] = (uint8_t)val;
                i += rep;
            }
            if (err) break;
            __syncwarp();
            /* the offset lengths follow the litlen lengths; move them to a 16-byte-friendly spot for the builder */
            if (!build_table(sm.lens, nl, INF_LROOT, sm.ltab, INF_LTAB, 0, sm.offs, lane) ||
                !build_table(sm.lens + nl, nd, INF_DROOT, sm.dtab, INF_DTAB, 1, sm.offs, lane)) { err = INF_E_CODE; break; }
            pair_literals(sm.ltab, INF_LROOT, lane);
        }
        /* ---- the decode loop ---- */
        for (;;) {
            uint32_t win = br_window(r);
            uint32_t e = sm.ltab[win & ((1u << INF_LROOT) - 1u)];
            uint32_t nb = e & 15u;
            if (!(e & F_LIT) && ((e >> 8) & 7u) == K_SUB) {
                e = sm.ltab[(e >> 16) + ((win >> INF_LROOT) & ((1u << ((e >> 11) & 7u)) - 1u))];
                nb = INF_LROOT + (e & 15u);
            }
            if (e & F_LIT) {
                const uint32_t cnt = 1u + ((e >> 14) & 1u);          /* F_LIT2: two literals in one entry */
                br_consume(r, nb);
                if (lane < cnt) o.win[(o.apos + lane) & (INF_WIN - 1u)] = (uint8_t)(e >> (16 + 8 * lane));
                if (ow_advance(o, cnt)) { err = INF_E_OVERRUN; break; }
                continue;
            }
            const uint32_t kind = (e >> 8) & 7u;
            if (kind == K_EOB) { br_consume(r, nb); break; }
            if (kind != K_BASE) { err = INF_E_SYMBOL; break; }
            const uint32_t xb = (e >> 4) & 15u;
            const uint32_t len = (e >> 16) + ((win >> nb) & ((1u << xb) - 1u));
            br_consume(r, nb + xb);
            win = br_window(r);
            const uint32_t d = lookup(sm.dtab, INF_DROOT, win, &nb);
            if (((d >> 8) & 7u) != K_BASE) { err = INF_E_SYMBOL; break; }
            const uint32_t dxb = (d >> 4) & 15u;
            const uint32_t dist = (d >> 16) + ((win >> nb) & ((1u << dxb) - 1u));
            br_consume(r, nb + dxb);
            if (dist > o.apos - o.first) { err = INF_E_DIST; break; }
            if (o.apos + len > end_apos) { err = INF_E_OVERRUN; break; }
            __syncwarp();   /* earlier window/global stores of this warp are visible to all its lanes */
            if (dist + len <= INF_WIN) {
                /* near: the source is still in the window.  Bytes are produced 32 at a time; with an overlapping
                 * copy (dist < len) byte k repeats byte k mod dist, which is always older than this match. */
                for (uint32_t done = 0; done < len; done += 32) {
                    const uint32_t k = done + lane;
                    if (k < len) {
                        const uint32_t sk = dist >= len ? k : (dist == 1 ? 0u : k % dist);
                        const uint8_t v = o.win[(o.apos - done - dist + sk) & (INF_WIN - 1u)];
                        o.win[(o.apos + lane) & (INF_WIN - 1u)] = v;
                    }
                    ow_advance(o, len - done < 32 ? len - done : 32);
                }
            } else {
                /* far: dist > INF_WIN - 258, so the source lies in lines that were flushed long ago */
                const uint8_t *srcp = o.gline + o.apos - dist;
                for (uint32_t done = 0; done < len; done += 32) {
                    const uint32_t k = done + lane;
                    if (k < len) o.win[(o.apos + lane) & (INF_WIN - 1u)] = __ldcg(srcp + k);
                    ow_advance(o, len - done < 32 ? len - done : 32);
                }
            }
        }
        if (br_overrun(r) && err == INF_OK) err = INF_E_OVERRUN;
    }
    ow_finish(o);
    if (err == INF_OK && o.apos != end_apos) err = INF_E_SHORT;
    if (lane == 0) {
        a.status[m] = err;
        if (err) atomicOr(a.err_flag, 1u);
    }
}

/* ------------------------------------------------------------------------------------------------ */
/* B200BGZF_VERIFY: CRC-32 of every member's output against the trailer (the reference's decompress loop checks
 * neither CRC32 nor ISIZE, applet/7bgzf.c:350-354; htslib does).  One CTA per member: the payload is staged in
 * shared memory and summed with the compressor's own slice-and-combine phase (bg_phase_scan: 1024 right-aligned
 * 68-byte slices, each multiplied by x^(8*68*k) mod P — zlib's crc32_combine algebra, lib/zlib/crc32.c:1021-1026). */
#define INF_E_CRC 9u
#define VER_SMEM (BG_DATA_BYTES + 1024u + 256u + 4u * BG_S_COUNT)

__global__ void __launch_bounds__(BG_THREADS, 2)
bgzf_verify_kernel(BgzfInflateArgs a)
{
    extern __shared__ __align__(16) uint8_t vs[];
    const uint32_t t = threadIdx.x, m = blockIdx.x;
    if (m >= a.nblocks || a.status[m] != INF_OK) return;          /* (uniform for the CTA) */
    /* a piece has no trailer of its own: its CRC goes to unit_crc[] for the host to combine (host/containers.c) */
    const bool piece = a.unit_isize && a.unit_isize[m] != 0xffffffffu;
    if (piece && !a.unit_crc) return;
    const uint8_t *mem = a.in + a.in_off[m];
    const uint32_t msize = a.hdr_len ? a.msize[m] : ((uint32_t)mem[16] | ((uint32_t)mem[17] << 8)) + 1u;
    const uint8_t *tr = mem + msize - 8;
    uint32_t want = 0, isize;
    if (piece) {
        isize = a.unit_isize[m];
    } else {
        want = (uint32_t)tr[0] | ((uint32_t)tr[1] << 8) | ((uint32_t)tr[2] << 16) | ((uint32_t)tr[3] << 24);
        isize = (uint32_t)tr[4] | ((uint32_t)tr[5] << 8) | ((uint32_t)tr[6] << 16) | ((uint32_t)tr[7] << 24);
    }
    const uint8_t *out = a.out + a.out_off[m];
    BgCtx c;
    memset(&c, 0, sizeof c);
    c.dataw = (uint32_t *)vs;
    c.crctab = (uint32_t *)(vs + BG_DATA_BYTES);
    c.litflag = vs + BG_DATA_BYTES + 1024u;
    c.scal = (uint32_t *)(vs + BG_DATA_BYTES + 1024u + 256u);
    c.crcpow = a.crcpow;
    c.frame = bg_frame(18u, 8u, 1u, 0u);
    if (t < 256) c.crctab[t] = a.crctab[t];
    /* members of the other containers may be larger than a BGZF block: tiles of 64 KiB, their CRCs combined as zlib's
     * crc32_combine does (lib/zlib/crc32.c:1021-1026): crc(A||B) = crc(A) * x^(8 len B) + crc(B) */
    uint32_t crc = 0;
    for (uint32_t done = 0; done < isize; done += BG_MAX_BLOCK) {
        const uint32_t len = isize - done < BG_MAX_BLOCK ? isize - done : BG_MAX_BLOCK;
        const uint8_t *src = out + done;
        c.n = len;
        __syncthreads();                                 /* (the previous tile's thread 0 is done with the buffer) */
        /* stage: bytes up to the first 16-byte boundary of the source, 16-byte loads for the body, bytes for the rest */
        const uint32_t head = len < 16 ? len : (uint32_t)((16u - ((uintptr_t)src & 15u)) & 15u);
        const uint32_t body = (len - head) & ~15u;
        if (t < head) vs[t] = src[t];
        for (uint32_t i = t * 16u; i < body; i += BG_THREADS * 16u) {
            const uint4 v = __ldcs((const uint4 *)(src + head + i));
            const uint32_t w[4] = { v.x, v.y, v.z, v.w };
            for (uint32_t k = 0; k < 16; k++) vs[head + i + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));   /* (destination is not aligned when head != 0) */
        }
        for (uint32_t i = head + body + t; i < len; i += BG_THREADS) vs[i] = src[i];
        if (t < 28) vs[len + t] = 0;
        if (t < BG_S_COUNT) c.scal[t] = 0;
        __syncthreads();
        bg_phase_scan(c, t, BG_THREADS);
        __syncthreads();
        if (t == 0) {
            uint32_t r = c.scal[BG_S_CRC];
            if ((len >> 2) == 0) r = 0xFFFFFFFFu;
            for (uint32_t p = len & ~3u; p < len; p++) r = bg_crc_byte(c.crctab, r, vs[p]);
            if (done == 0) {
                crc = ~r;
            } else {
                uint32_t shift = 0x80000000u, sq = 0x00800000u;          /* 1, x^8 (reflected: bit 31 is x^0) */
                for (uint32_t e = len; e; e >>= 1) {
                    if (e & 1u) shift = bg_crc_mul(shift, sq);
                    sq = bg_crc_mul(sq, sq);
                }
                crc = bg_crc_mul(crc, shift) ^ ~r;
            }
        }
    }
    if (t == 0) {
        if (piece) {
            a.unit_crc[m] = crc;
        } else {
            if (a.unit_crc) a.unit_crc[m] = crc;
            if (crc != want) {
                a.status[m] = INF_E_CRC;
                atomicOr(a.err_flag, 2u);
            }
        }
    }
}

/* ------------------------------------------------------------------------------------------------ */
/* member index of a device-resident stream                                                         */

#define IDX_TILE 32768u
#define IDX_THREADS 256u
#define IDX_PER_THREAD (IDX_TILE / IDX_THREADS)

__device__ __forceinline__ bool is_member_start(const uint8_t *p, uint64_t i, uint64_t n)
{
    if (i + 28 > n) return false;
    const uint8_t *q = p + i;
    return q[0] == 0x1f && q[1] == 0x8b && q[2] == 0x08 && q[3] == 0x04 && q[10] == 0x06 && q[11] == 0 && q[12] == 'B' &&
           q[13] == 'C' && q[14] == 2 && q[15] == 0;
}

/* 128-bit candidate mask for the 128 positions [base, base+128) owned by one thread */
__device__ __forceinline__ void scan_positions(const uint8_t *in, uint64_t n, uint64_t base, bool vec_ok, uint32_t mask[4])
{
    mask[0] = mask[1] = mask[2] = mask[3] = 0;
    for (uint32_t k = 0; k < IDX_PER_THREAD / 16; k++) {
        const uint64_t off = base + 16u * k;
        if (off >= n) break;
        uint32_t hit = 0;   /* bit j: byte j of this 16-byte group is 0x1f */
        if (vec_ok && off + 16 <= n) {
            const uint4 v = __ldg((const uint4 *)(in + off));
            const uint32_t w[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t x = w[q] ^ 0x1f1f1f1fu;
                const uint32_t z = (x - 0x01010101u) & ~x & 0x80808080u;   /* may over-report; verified below */
                if (z) hit |= 0xfu << (4 * q);
            }
        } else {
            hit = 0xffffu;
        }
        while (hit) {
            const uint32_t j = __ffs(hit) - 1;
            hit &= hit - 1;
            const uint64_t i = off + j;
            if (i < n && in[i] == 0x1f && is_member_start(in, i, n)) {
                const uint32_t bit = 16u * k + j;
                mask[bit >> 5] |= 1u << (bit & 31u);
            }
        }
    }
}

/* pass 0 (write == 0): candidates per tile.  pass 1: ordered list of candidate offsets. */
__global__ void __launch_bounds__(IDX_THREADS)
bgzf_index_scan_kernel(const uint8_t *in, uint64_t n, uint32_t *tile_count, const uint64_t *tile_off, uint64_t *in_off,
                       uint32_t max_blocks, int write)
{
    __shared__ uint32_t wsum[IDX_THREADS / 32];
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    const uint64_t base = (uint64_t)blockIdx.x * IDX_TILE + (uint64_t)t * IDX_PER_THREAD;
    uint32_t mask[4];
    scan_positions(in, n, base, ((uintptr_t)in & 15u) == 0, mask);
    const uint32_t cnt = __popc(mask[0]) + __popc(mask[1]) + __popc(mask[2]) + __popc(mask[3]);
    uint32_t inc = cnt;
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += y;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (uint32_t w = 0; w < IDX_THREADS / 32; w++) {
        if (w < warp) before += wsum[w];
        total += wsum[w];
    }
    if (!write) {
        if (t == 0) tile_count[blockIdx.x] = total;
        return;
    }
    uint64_t slot = tile_off[blockIdx.x] + before + inc - cnt;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint32_t mm = mask[q];
        while (mm) {
            const uint32_t j = __ffs(mm) - 1;
            mm &= mm - 1;
            if (slot < max_blocks) in_off[slot] = base + 32u * q + j;
            slot++;
        }
    }
}

/* ---- which candidates are members?  The reference walks the headers strictly one after the other (applet/7bgzf.c:306-330):
 * a member starts at offset 0, the next one where BSIZE says this one ends.  A signature hit that is not on that chain is
 * payload (a stored member that carries BGZF data: bgzip of a .bam, a tar of .bgz files) and must be ignored, not
 * rejected.  On the device the walk is a reachability question over the sorted candidate list:
 *   next   nxt[k] = index of the candidate that starts exactly where candidate k's member ends (binary search);
 *          nc = "ends exactly at the end of the stream", nc + 1 = "ends nowhere" (both absorbing)
 *   chain  pointer doubling from candidate 0 (one CTA; log2(nc) rounds): reach[k] = 1 for every candidate on the chain
 *   pick   ordered compaction of the reached candidates (scan of reach[]) + their ISIZE                           ---- */
__global__ void __launch_bounds__(256)
bgzf_index_next_kernel(const uint8_t *in, uint64_t n, const uint64_t *cand_off, const uint64_t *count, uint32_t max_blocks,
                       uint32_t *nxt, uint32_t *reach, uint32_t *status)
{
    const uint64_t nc64 = *count;
    if (nc64 > max_blocks || nc64 == 0) {
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(status, nc64 == 0 ? 1u : 2u);
        return;
    }
    const uint32_t nc = (uint32_t)nc64;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nc + 2; k += gridDim.x * blockDim.x) {
        reach[k] = 0;
        if (k >= nc) { nxt[k] = k; continue; }
        const uint64_t o = cand_off[k];
        const uint64_t next = o + ((uint32_t)in[o + 16] | ((uint32_t)in[o + 17] << 8)) + 1u;
        uint32_t r = nc + 1;
        if (next == n) r = nc;
        else if (next < n) {
            uint32_t lo = k + 1, hi = nc;                 /* first candidate at or past `next` */
            while (lo < hi) {
                const uint32_t mid = lo + ((hi - lo) >> 1);
                if (cand_off[mid] < next) lo = mid + 1; else hi = mid;
            }
            if (lo < nc && cand_off[lo] == next) r = lo;
        }
        nxt[k] = r;
    }
}

/* one CTA.  jump[] starts as nxt[] and is squared every round (jump <- jump o jump); every reached node marks its jump
 * target, so after round r everything within 2^(r+1) - 1 steps of the start is marked.  Marks only ever name true
 * successors, so reading a mark that another thread sets in the same round is harmless. */
__global__ void __launch_bounds__(1024, 1)
bgzf_index_chain_kernel(const uint64_t *cand_off, const uint64_t *count, uint32_t max_blocks, uint32_t *jump, uint32_t *jump2,
                        uint32_t *reach, uint32_t *status)
{
    const uint64_t nc64 = *count;
    if (nc64 > max_blocks || nc64 == 0) return;            /* (reported by the kernel before) */
    const uint32_t nc = (uint32_t)nc64, t = threadIdx.x;
    if (t == 0) reach[0] = cand_off[0] == 0 ? 1u : 0u;
    __syncthreads();
    uint32_t *cur = jump, *nx = jump2;
    for (uint32_t span = 1; span < nc + 1; span <<= 1) {
        for (uint32_t k = t; k < nc; k += 1024)
            if (reach[k]) reach[cur[k]] = 1u;
        for (uint32_t k = t; k < nc + 2; k += 1024) nx[k] = cur[cur[k]];
        __syncthreads();
        uint32_t *tmp = cur; cur = nx; nx = tmp;
    }
    for (uint32_t k = t; k < nc; k += 1024)
        if (reach[k]) reach[cur[k]] = 1u;
    __syncthreads();
    if (t == 0 && !reach[nc]) atomicOr(status, 1u);         /* the walk from offset 0 does not end at the end of the stream */
}

/* the reached candidates, in order, with their ISIZE; idx[] = exclusive scan of reach[] */
__global__ void __launch_bounds__(256)
bgzf_index_pick_kernel(const uint8_t *in, const uint64_t *cand_off, const uint64_t *count, uint32_t max_blocks, const uint32_t *reach,
                       const uint64_t *idx, uint64_t *in_off, uint32_t *isize, uint32_t *status)
{
    const uint64_t nc64 = *count;
    if (nc64 > max_blocks || nc64 == 0) return;
    const uint32_t nc = (uint32_t)nc64;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nc; k += gridDim.x * blockDim.x) {
        if (!reach[k]) continue;
        const uint64_t o = cand_off[k];
        const uint64_t next = o + ((uint32_t)in[o + 16] | ((uint32_t)in[o + 17] << 8)) + 1u;
        const uint8_t *tr = in + next - 4;
        const uint32_t v = (uint32_t)tr[0] | ((uint32_t)tr[1] << 8) | ((uint32_t)tr[2] << 16) | ((uint32_t)tr[3] << 24);
        in_off[idx[k]] = o;
        isize[idx[k]] = v;
        if (v > 65536u) atomicOr(status, 1u);
    }
}

extern "C" cudaError_t bgzf_launch_inflate(const BgzfInflateArgs *a, cudaStream_t stream)
{
    if (a->nblocks == 0) return cudaSuccess;
    static std::atomic<unsigned long long> configured{0};     /* per device, once (function attributes are per device) */
    int dev0 = 0;
    cudaGetDevice(&dev0);
    if (!((configured.load() >> dev0) & 1ull)) {
        cudaFuncSetAttribute(bgzf_inflate_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured.fetch_or(1ull << dev0);
    }
    bgzf_inflate_kernel<<<a->nblocks, 32 * INF_WARPS_PER_CTA, 0, stream>>>(*a);
    if (a->verify_crc) return bgzf_launch_verify(a, stream);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_verify(const BgzfInflateArgs *a, cudaStream_t stream)
{
    if (a->nblocks == 0) return cudaSuccess;
    static std::atomic<unsigned long long> vconf{0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!((vconf.load() >> dev) & 1ull)) {
        cudaError_t e = cudaFuncSetAttribute(bgzf_verify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)VER_SMEM);
        if (e != cudaSuccess) return e;
        vconf.fetch_or(1ull << dev);
    }
    bgzf_verify_kernel<<<a->nblocks, BG_THREADS, VER_SMEM, stream>>>(*a);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_chain(const uint64_t *cand_off, const uint64_t *count, uint32_t max_blocks, uint32_t *jump,
                                         uint32_t *jump2, uint32_t *reach, uint32_t *status, cudaStream_t stream)
{
    bgzf_index_chain_kernel<<<1, 1024, 0, stream>>>(cand_off, count, max_blocks, jump, jump2, reach, status);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_index(const uint8_t *in, uint64_t in_bytes, const BgzfIndexWork *w, cudaStream_t stream)
{
    const uint32_t tiles = (uint32_t)((in_bytes + IDX_TILE - 1) / IDX_TILE);
    if (tiles == 0) return cudaErrorInvalidValue;
    /* candidates: every position that carries the 16-byte BGZF signature, in order */
    bgzf_index_scan_kernel<<<tiles, IDX_THREADS, 0, stream>>>(in, in_bytes, w->tile_count, nullptr, nullptr, w->max_blocks, 0);
    bgzf_launch_scan(w->tile_count, w->tile_off, tiles, nullptr, nullptr, w->ncand, stream);
    bgzf_index_scan_kernel<<<tiles, IDX_THREADS, 0, stream>>>(in, in_bytes, w->tile_count, w->tile_off, w->cand_off, w->max_blocks, 1);
    /* members: the candidates on the BSIZE chain from offset 0 */
    bgzf_index_next_kernel<<<64, 256, 0, stream>>>(in, in_bytes, w->cand_off, w->ncand, w->max_blocks, w->jump, w->reach, w->status);
    bgzf_launch_chain(w->cand_off, w->ncand, w->max_blocks, w->jump, w->jump2, w->reach, w->status, stream);
    bgzf_launch_scan(w->reach, w->pick_idx, w->max_blocks, w->ncand, nullptr, w->nmembers, stream);
    bgzf_index_pick_kernel<<<64, 256, 0, stream>>>(in, w->cand_off, w->ncand, w->max_blocks, w->reach, w->pick_idx, w->in_off, w->isize, w->status);
    /* out_off = exclusive scan of ISIZE over the members (count read on the device) */
    bgzf_launch_scan(w->isize, w->out_off, w->max_blocks, w->nmembers, nullptr, w->out_bytes, stream);
    return cudaGetLastError();
}

extern "C" size_t bgzf_index_tiles(uint64_t in_bytes) { return (size_t)((in_bytes + IDX_TILE - 1) / IDX_TILE); }
