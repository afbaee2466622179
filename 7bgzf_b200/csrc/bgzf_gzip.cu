/*
 * bgzf_gzip.cu — sm_100a kernels that inflate one whole-stream gzip member in parallel, cut at its byte-aligned flush points.
 *
 * Every non-final piece our GZIP writer emits, every pigz chunk and every zlib Z_SYNC_FLUSH / Z_FULL_FLUSH ends with an
 * empty stored block: 3 header bits, padding, then 00 00 ff ff.  So a block starts at the byte after each such pattern, and
 * a decoder can start there with nothing but the 32 KiB of output before it.  The pipeline (host side: b200bgzf_api.cu):
 *   gz_cand_scan_kernel    every position after 00 00 ff ff in the DEFLATE data (ordered tile-count -> scan -> write, as
 *                          bgzf_index_scan_kernel); the data start is candidate 0
 *   gz_bound_kernel        one warp per candidate decodes symbols without output: where its chunk ends (right after the first
 *                          non-final empty stored block it decodes, or at the end of the final block), its output length, status
 *   gz_next_kernel         successor links: the candidate at a chunk's end; then bgzf_launch_chain (pointer doubling) keeps the
 *                          candidates on the chain from candidate 0 — the exact bit path of a sequential decoder
 *   gz_pick_kernel         the chained chunks in order (scan of reach[]), their output offsets (scan of their lengths)
 *   gz_marker_kernel       one warp per chained chunk decodes into u16 scratch: < 256 a byte, 256 + j byte j of the 32 KiB of
 *                          output before the chunk (a back-reference that leaves the chunk)
 *   gz_anchor_kernel       a chunk whose preceding 32 KiB hold no marker is an anchor (prefix max of the last-marker positions)
 *   gz_resolve_kernel      one CTA per anchor resolves, chunk after chunk up to the next anchor, the markers of every chunk's last
 *                          32 KiB (the only bytes a later window can name) in place
 *   gz_narrow_kernel       bytes into the caller's output; a marker reads the resolved window of its chunk
 * A false candidate (the pattern inside a stored block or by chance in Huffman data) is never on the chain: it costs one warp
 * of the boundary pass, whose compressed length is capped.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "bgzf_block.h"
#include "bgzf_inflate_dev.h"
#include "bgzf_kernels.h"

#define GZ_TILE 32768u
#define GZ_THREADS 256u
#define GZ_PER_THREAD (GZ_TILE / GZ_THREADS)
#define GZ_WIN 32768u               /* DEFLATE's window: the scratch of a batch starts with the 32 KiB before it */
#define GZ_MAX_CHUNK 0x7fffffffu    /* output of one chunk (the one-warp path's bound on a member's ISIZE) */

/* ---- candidates ---- */

/* bit j of mask: position base + j follows 00 00 ff ff */
__device__ __forceinline__ void flush_positions(const uint8_t *d, uint64_t n, uint64_t base, uint32_t mask[4])
{
    mask[0] = mask[1] = mask[2] = mask[3] = 0;
    uint32_t w = 0x01010101u;                           /* the 4 bytes before the position, newest in the top byte */
    for (uint32_t k = 4; k >= 1; k--)
        if (base >= k && base - k < n) w = (w >> 8) | ((uint32_t)__ldg(d + base - k) << 24);
    for (uint32_t j = 0; j < GZ_PER_THREAD; j++) {
        const uint64_t i = base + j;
        if (i >= n) break;
        if (w == 0xffff0000u) mask[j >> 5] |= 1u << (j & 31u);
        w = (w >> 8) | ((uint32_t)__ldg(d + i) << 24);
    }
}

/* pass 0 (write == 0): candidates per tile.  pass 1: cand[0] = 0, then every candidate in order; ncand = 1 + their count. */
__global__ void __launch_bounds__(GZ_THREADS)
gz_cand_scan_kernel(const uint8_t *d, uint64_t n, uint32_t *tile_count, const uint64_t *tile_off, uint64_t *cand, uint64_t *counts,
                    int write)
{
    __shared__ uint32_t wsum[GZ_THREADS / 32];
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    const uint64_t base = (uint64_t)blockIdx.x * GZ_TILE + (uint64_t)t * GZ_PER_THREAD;
    uint32_t mask[4];
    flush_positions(d, n, base, mask);
    const uint32_t cnt = __popc(mask[0]) + __popc(mask[1]) + __popc(mask[2]) + __popc(mask[3]);
    uint32_t inc = cnt;
    for (int s = 1; s < 32; s <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, s);
        if (lane >= (uint32_t)s) inc += y;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (uint32_t w = 0; w < GZ_THREADS / 32; w++) {
        if (w < warp) before += wsum[w];
        total += wsum[w];
    }
    if (!write) {
        if (t == 0) tile_count[blockIdx.x] = total;
        return;
    }
    if (blockIdx.x == 0 && t == 0) {
        cand[0] = 0;
        counts[1] = counts[0] + 1;
    }
    uint64_t slot = 1 + tile_off[blockIdx.x] + before + inc - cnt;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint32_t mm = mask[q];
        while (mm) {
            const uint32_t j = __ffs(mm) - 1;
            mm &= mm - 1;
            cand[slot++] = base + 32u * q + j;
        }
    }
}

/* ---- decoding one chunk ---- */

struct GzChunk {
    uint64_t end;       /* byte offset (in the DEFLATE data) one past the chunk */
    uint32_t olen;      /* output bytes */
    uint32_t status;
    uint32_t lastm;     /* EMIT: one past the last marker written (0: none) */
    uint32_t dist_err;  /* EMIT: a back-reference before the member start */
};

/* One warp decodes the blocks from `p` (a byte-aligned block start) as bgzf_inflate_kernel would, up to the end of the chunk.
 * EMIT: writes u16 symbols to out[0..olen) — bytes, or 256 + j for byte j of the 32 KiB before the chunk; abs0 = the chunk's
 * output offset in the member (a reference further back is INF_E_DIST).  Without EMIT only the lengths are counted, and a
 * reference before the chunk is an error only for the chunk at the member start (first).  Reading stops at `lim` (the
 * trailer, or the compressed-length cap): more input is GZ_FAIL, and so is more output than max_out.
 * BITS (the searched route): the chunk starts `skip` bits into byte p, ends at the first block boundary at or after bit `stop`
 * of the DEFLATE data, or with the final block, and c.end is a bit offset; an empty stored block ends nothing. */
template <bool EMIT, bool BITS = false>
__device__ GzChunk gz_decode_chunk(InfSmem &sm, const uint8_t *data, const uint8_t *p, const uint8_t *lim, bool first, uint16_t *out,
                                   uint32_t max_out, uint64_t abs0, uint32_t lane, uint32_t skip = 0, uint64_t stop = 0)
{
    GzChunk c;
    c.end = 0;
    c.olen = 0;
    c.status = GZ_FAIL;
    c.lastm = 0;
    c.dist_err = 0;
    uint32_t pos = 0, lastm = 0;
    bool fail = false;
    BitReader r;
    br_init(r, p, lim, lane);
    if (BITS) br_consume(r, skip);
    for (;;) {
        const bool last = br_take(r, 1);
        const uint32_t btype = br_take(r, 2);
        if (btype == 0) {
            br_consume(r, (8u - (r.bit & 7u)) & 7u);
            const uint32_t len = br_take(r, 16);
            const uint32_t nlen = br_take(r, 16);
            if ((len ^ nlen) != 0xffffu) { fail = true; break; }
            const uint8_t *raw = (const uint8_t *)(r.base + r.wi) + (r.bit >> 3);
            if (raw + len > lim || pos + len > max_out) { fail = true; break; }
            if (EMIT)
                for (uint32_t k = lane; k < len; k += 32) out[pos + k] = raw[k];
            pos += len;
            if (BITS) {
                const uint64_t eb = 8ull * (uint64_t)(raw + len - data);
                if (last || eb >= stop) {
                    c.end = eb;
                    c.status = last ? GZ_END_FINAL : GZ_END_FLUSH;
                    break;
                }
            } else if (last || len == 0) {
                c.end = (uint64_t)(raw + len - data);
                c.status = last ? GZ_END_FINAL : GZ_END_FLUSH;
                break;
            }
            br_init(r, raw + len, lim, lane);
            continue;
        }
        if (btype == 3) { fail = true; break; }
        if (btype == 1) {
            for (uint32_t i = lane; i < 288; i += 32) sm.lens[i] = (uint8_t)bg_static_llen(i);
            sm.lens[288 + lane] = 5;
            __syncwarp();
            if (!build_table(sm.lens, 288, INF_LROOT, sm.ltab, INF_LTAB, 0, sm.offs, lane) ||
                !build_table(sm.lens + 288, 32, INF_DROOT, sm.dtab, INF_DTAB, 1, sm.offs, lane)) { fail = true; break; }
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
            if (!build_table(sm.lens, 19, 7, sm.dtab, INF_PTAB, 2, sm.offs, lane)) { fail = true; break; }
            uint32_t i = 0, prevlen = 0;
            const uint32_t total = nl + nd;
            while (i < total) {
                const uint32_t e = sm.dtab[br_window(r) & 127u];
                if (e == 0) { fail = true; break; }
                br_consume(r, e & 15u);
                const uint32_t sym = e >> 16;
                uint32_t rep, val;
                if (sym < 16) { rep = 1; val = sym; prevlen = sym; }
                else if (sym == 16) { if (i == 0) { fail = true; break; } rep = 3 + br_take(r, 2); val = prevlen; }
                else if (sym == 17) { rep = 3 + br_take(r, 3); val = 0; prevlen = 0; }
                else { rep = 11 + br_take(r, 7); val = 0; prevlen = 0; }
                if (i + rep > total) { fail = true; break; }
                for (uint32_t k = lane; k < rep; k += 32) sm.lens[i + k] = (uint8_t)val;
                i += rep;
            }
            if (fail) break;
            __syncwarp();
            if (!build_table(sm.lens, nl, INF_LROOT, sm.ltab, INF_LTAB, 0, sm.offs, lane) ||
                !build_table(sm.lens + nl, nd, INF_DROOT, sm.dtab, INF_DTAB, 1, sm.offs, lane)) { fail = true; break; }
            pair_literals(sm.ltab, INF_LROOT, lane);
        }
        for (;;) {
            /* (the input cap is tested per symbol: a false candidate may decode garbage for a long time) */
            if (br_overrun(r)) { fail = true; break; }
            uint32_t win = br_window(r);
            uint32_t e = sm.ltab[win & ((1u << INF_LROOT) - 1u)];
            uint32_t nb = e & 15u;
            if (!(e & F_LIT) && ((e >> 8) & 7u) == K_SUB) {
                e = sm.ltab[(e >> 16) + ((win >> INF_LROOT) & ((1u << ((e >> 11) & 7u)) - 1u))];
                nb = INF_LROOT + (e & 15u);
            }
            if (e & F_LIT) {
                const uint32_t cnt = 1u + ((e >> 14) & 1u);
                br_consume(r, nb);
                if (pos + cnt > max_out) { fail = true; break; }
                if (EMIT && lane < cnt) out[pos + lane] = (uint16_t)((e >> (16 + 8 * lane)) & 0xffu);
                pos += cnt;
                continue;
            }
            const uint32_t kind = (e >> 8) & 7u;
            if (kind == K_EOB) { br_consume(r, nb); break; }
            if (kind != K_BASE) { fail = true; break; }
            const uint32_t xb = (e >> 4) & 15u;
            const uint32_t len = (e >> 16) + ((win >> nb) & ((1u << xb) - 1u));
            br_consume(r, nb + xb);
            win = br_window(r);
            const uint32_t d = lookup(sm.dtab, INF_DROOT, win, &nb);
            if (((d >> 8) & 7u) != K_BASE) { fail = true; break; }
            const uint32_t dxb = (d >> 4) & 15u;
            const uint32_t dist = (d >> 16) + ((win >> nb) & ((1u << dxb) - 1u));
            br_consume(r, nb + dxb);
            if (first && dist > pos) { fail = true; break; }
            if (pos + len > max_out) { fail = true; break; }
            if (EMIT) {
                if (dist > abs0 + pos) { c.dist_err = 1; fail = true; break; }
                __syncwarp();   /* the literals and matches before this one are visible to every lane */
                for (uint32_t k = lane; k < len; k += 32) {
                    /* byte k repeats byte k mod dist of an overlapping copy, always older than this match */
                    const uint32_t sk = dist >= len ? k : (dist == 1 ? 0u : k % dist);
                    const int64_t src = (int64_t)pos - dist + sk;
                    const uint16_t v = src >= 0 ? out[src] : (uint16_t)(256 + GZ_WIN + src);
                    out[pos + k] = v;
                    if (v >= 256) lastm = pos + k + 1;
                }
            }
            pos += len;
        }
        if (fail) break;
        if (br_overrun(r)) { fail = true; break; }
        if (BITS) {
            const uint64_t eb = 8ull * (uint64_t)((const uint8_t *)r.base - data) + r.wi * 32u + r.bit;
            if (last || eb >= stop) {
                c.end = eb;
                c.status = last ? GZ_END_FINAL : GZ_END_FLUSH;
                break;
            }
        } else if (last) {
            c.end = (uint64_t)((const uint8_t *)r.base - data) + (r.wi * 32u + r.bit + 7u) / 8u;
            c.status = GZ_END_FINAL;
            break;
        }
    }
    if (fail) c.status = GZ_FAIL;
    c.olen = pos;
    if (EMIT) {
        __syncwarp();
        c.lastm = __reduce_max_sync(0xffffffffu, lastm);
    }
    return c;
}

/* one warp per candidate: where its chunk ends, how much it yields */
__global__ void __launch_bounds__(32, 32)
gz_bound_kernel(BgzfGzipArgs a)
{
    __shared__ InfSmem sm;
    const uint32_t lane = threadIdx.x, k = blockIdx.x;
    if (k >= *a.ncand) return;
    const uint64_t s = a.cand[k];
    const uint8_t *lim = a.data + (a.data_len - s > a.max_in ? s + a.max_in : a.data_len);
    const GzChunk c = gz_decode_chunk<false>(sm, a.data, a.data + s, lim, k == 0, nullptr, GZ_MAX_CHUNK, 0, lane);
    if (lane == 0) {
        a.end[k] = c.end;
        a.olen[k] = c.olen;
        a.status[k] = c.status;
    }
}

/* nxt[k] = the candidate where chunk k ends; nc = "the member's DEFLATE data ends here", nc + 1 = "nowhere" (both absorbing) */
__global__ void __launch_bounds__(256)
gz_next_kernel(BgzfGzipArgs a)
{
    const uint32_t nc = (uint32_t)*a.ncand;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nc + 2; k += gridDim.x * blockDim.x) {
        a.reach[k] = 0;
        if (k >= nc) { a.jump[k] = k; continue; }
        uint32_t r = nc + 1;
        const uint64_t e = a.end[k];
        if (a.status[k] == GZ_END_FINAL) {
            if (e == a.data_len) r = nc;
        } else if (a.status[k] == GZ_END_FLUSH) {
            uint32_t lo = k + 1, hi = nc;
            while (lo < hi) {
                const uint32_t mid = lo + ((hi - lo) >> 1);
                if (a.cand[mid] < e) lo = mid + 1; else hi = mid;
            }
            if (lo < nc && a.cand[lo] == e) r = lo;
        }
        a.jump[k] = r;
    }
}

/* the chained chunks in order: their start and length (pick = exclusive scan of reach[]) */
__global__ void __launch_bounds__(256)
gz_pick_kernel(BgzfGzipArgs a)
{
    const uint32_t nc = (uint32_t)*a.ncand;
    for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nc; k += gridDim.x * blockDim.x) {
        if (!a.reach[k]) continue;
        const uint64_t j = a.pick[k];
        a.c_start[j] = a.cand[k];
        a.c_len[j] = a.olen[k];
    }
}

/* ---- one batch: chained chunks [j0, j1), output [base, base + bytes) ---- */

/* scratch[0, GZ_WIN) = the 32 KiB of output before the batch (already written by the batches before it) */
__global__ void gz_prefix_kernel(BgzfGzipArgs a, uint64_t base)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < GZ_WIN; i += gridDim.x * blockDim.x) {
        const int64_t at = (int64_t)base - GZ_WIN + i;
        a.scratch[i] = at >= 0 ? a.out[at] : 0;
    }
}

/* one warp per chained chunk, in u16 scratch at its exact offset */
__global__ void __launch_bounds__(32, 32)
gz_marker_kernel(BgzfGzipArgs a, uint32_t j0, uint64_t base)
{
    __shared__ InfSmem sm;
    const uint32_t lane = threadIdx.x, j = j0 + blockIdx.x;
    const uint64_t s = a.c_start[j], o = a.c_off[j];
    const uint8_t *lim = a.data + (a.data_len - s > a.max_in ? s + a.max_in : a.data_len);
    const GzChunk c = gz_decode_chunk<true>(sm, a.data, a.data + s, lim, s == 0, a.scratch + GZ_WIN + (o - base), a.c_len[j], o, lane);
    if (lane == 0) {
        a.lastm[j] = c.lastm;
        if (c.status == GZ_FAIL || c.olen != a.c_len[j]) atomicOr(a.err, c.dist_err ? 1u : 2u);
    }
}

/* ---- members without flush points (DESIGN §6g): chunk starts at bit offsets, found by a search for block headers ----
 * Region r >= 1 (GZ_REGION compressed bytes each) proposes the first bit offset inside it whose bits read as a dynamic block
 * header gz_decode_chunk would accept: BTYPE 2, a precode, code lengths and litlen / distance codes that build_table takes, and
 * a code for end-of-block.  The search only proposes: a missed start merges two regions, a false one costs a repair round of
 * the host's chain walk.  The boundary and marker passes then decode chunks between bit offsets. */
#ifndef GZ_REGION
#define GZ_REGION (256u << 10)
#endif
#define GZ_SEARCH_WARPS 4u

/* 32 bits of the stream from bit b of the word-aligned base w (words from nwords on read as zeros) */
__device__ __forceinline__ uint32_t gz_bits_at(const uint32_t *w, uint32_t nwords, uint64_t b)
{
    const uint64_t i = b >> 5;
    const uint32_t lo = i < nwords ? __ldg(w + i) : 0u, hi = i + 1 < nwords ? __ldg(w + i + 1) : 0u;
    return __funnelshift_r(lo, hi, (uint32_t)b & 31u);
}

/* where precode symbol s stands in the header's length list (the inverse of bg_precode_order) */
__device__ __forceinline__ uint32_t gz_precode_pos(uint32_t s)
{
    const uint64_t lo = 3ull | 17ull << 5 | 15ull << 10 | 13ull << 15 | 11ull << 20 | 9ull << 25 | 7ull << 30 | 5ull << 35 |
                        4ull << 40 | 6ull << 45 | 8ull << 50 | 10ull << 55;
    const uint64_t hi = 12ull | 14ull << 5 | 16ull << 10 | 18ull << 15 | 0ull << 20 | 1ull << 25 | 2ull << 30;
    return (uint32_t)((s < 12 ? lo >> (5 * s) : hi >> (5 * (s - 12))) & 31u);
}

/* one lane: does a dynamic block header the decoder accepts start at bit b?  srt: this lane's 19 bytes of shared memory */
__device__ bool gz_dynamic_header(const uint32_t *w, uint32_t nwords, uint64_t b, uint8_t *srt)
{
    const uint32_t x = gz_bits_at(w, nwords, b);
    if (((x >> 1) & 3u) != 2u) return false;
    const uint32_t nl = ((x >> 3) & 31u) + 257, nd = ((x >> 8) & 31u) + 1, np = ((x >> 13) & 15u) + 4;
    b += 17;
    const uint64_t pc = ((uint64_t)gz_bits_at(w, nwords, b) | (uint64_t)gz_bits_at(w, nwords, b + 32) << 32) &
                        ((1ull << (3 * np)) - 1ull);
    b += 3 * np;
    /* the precode: complete, or one 1-bit codeword (build_table's rule; an empty one leaves end-of-block without a code) */
    uint32_t kraft = 0, ncodes = 0;
    uint64_t cnt = 0;                                   /* 5 bits per length */
    for (uint32_t i = 0; i < np; i++) {
        const uint32_t l = (uint32_t)(pc >> (3 * i)) & 7u;
        if (!l) continue;
        kraft += 128u >> l;
        ncodes++;
        cnt += 1ull << (5 * l);
    }
    const bool lone = ncodes == 1 && kraft == 64;
    if (kraft != 128 && !lone) return false;
    uint32_t lone_sym = 0;
    {
        uint32_t offs[8], at = 0;
        for (uint32_t l = 1; l <= 7; l++) { offs[l] = at; at += (uint32_t)(cnt >> (5 * l)) & 31u; }
        for (uint32_t s = 0; s < 19; s++) {
            const uint32_t i = gz_precode_pos(s);
            const uint32_t l = i < np ? (uint32_t)(pc >> (3 * i)) & 7u : 0u;
            if (l) { srt[offs[l]++] = (uint8_t)s; lone_sym = s; }
        }
    }
    /* the code lengths, decoded as gz_decode_chunk does; Kraft sums of the litlen and distance codes on the way */
    const uint32_t total = nl + nd;
    uint32_t i = 0, prev = 0, kl = 0, kd = 0, cl = 0, cd = 0, l1 = 0, d1 = 0, eob = 0;
    while (i < total) {
        uint32_t v = gz_bits_at(w, nwords, b), sym = lone_sym, nb = 1;
        if (!lone) {
            int code = 0, first = 0, index = 0;
            for (nb = 1; nb <= 7; nb++) {
                code |= (int)((v >> (nb - 1)) & 1u);
                const int count = (int)((cnt >> (5 * nb)) & 31u);
                if (code - count < first) { sym = srt[index + (code - first)]; break; }
                index += count;
                first = (first + count) << 1;
                code <<= 1;
            }
        }
        v >>= nb;
        uint32_t rep, val, xb = 0;
        if (sym < 16) { rep = 1; val = sym; prev = sym; }
        else if (sym == 16) { if (i == 0) return false; xb = 2; rep = 3 + (v & 3u); val = prev; }
        else if (sym == 17) { xb = 3; rep = 3 + (v & 7u); val = 0; prev = 0; }
        else { xb = 7; rep = 11 + (v & 127u); val = 0; prev = 0; }
        b += nb + xb;
        if (i + rep > total) return false;
        if (val) {
            const uint32_t nlit = i < nl ? min(i + rep, nl) - i : 0u, ndist = rep - nlit;
            kl += nlit << (15 - val);
            kd += ndist << (15 - val);
            cl += nlit;
            cd += ndist;
            if (val == 1) { l1 += nlit; d1 += ndist; }
            if (i <= 256 && 256 < i + rep) eob = val;
            if (kl > (1u << 15) || kd > (1u << 15)) return false;
        }
        i += rep;
    }
    if (!eob) return false;
    if (kl != (1u << 15) && !(cl == 1 && l1 == 1)) return false;
    return kd == (1u << 15) || cd == 0 || (cd == 1 && d1 == 1);
}

/* one warp per region r >= 1, one lane per bit offset: found[r - 1] = the first accepted offset (bits), or ~0 */
__global__ void __launch_bounds__(GZ_SEARCH_WARPS * 32)
gz_search_kernel(const uint8_t *data, uint64_t data_len, uint32_t nreg, uint64_t *found)
{
    __shared__ uint8_t srt[GZ_SEARCH_WARPS * 32][20];
    const uint32_t lane = threadIdx.x & 31u, r = 1 + blockIdx.x * GZ_SEARCH_WARPS + (threadIdx.x >> 5);
    if (r >= nreg) return;
    const uint32_t mis = (uint32_t)((uintptr_t)data & 3u);
    const uint32_t *w = (const uint32_t *)(data - mis);
    const uint32_t nwords = (uint32_t)((data_len + mis + 3) >> 2);
    const uint64_t b0 = 8ull * GZ_REGION * r, b1 = min(b0 + 8ull * GZ_REGION, 8ull * data_len);
    uint64_t hit = ~0ull;
    for (uint64_t b = b0; b < b1; b += 32) {
        const bool ok = b + lane < b1 && gz_dynamic_header(w, nwords, 8ull * mis + b + lane, srt[threadIdx.x]);
        const uint32_t m = __ballot_sync(0xffffffffu, ok);
        if (m) { hit = b + __ffs(m) - 1; break; }
    }
    if (lane == 0) found[r - 1] = hit;
}

/* gz_bound_kernel between bit offsets: candidate k = cand[k] (bits) decodes up to the first block boundary at or after stop[k] */
__global__ void __launch_bounds__(32, 32)
gz_bit_bound_kernel(BgzfGzipArgs a, const uint64_t *stop)
{
    __shared__ InfSmem sm;
    const uint32_t lane = threadIdx.x, k = blockIdx.x;
    const uint64_t sb = a.cand[k], s = sb >> 3;
    const uint8_t *lim = a.data + (a.data_len - s > a.max_in ? s + a.max_in : a.data_len);
    const GzChunk c = gz_decode_chunk<false, true>(sm, a.data, a.data + s, lim, sb == 0, nullptr, GZ_MAX_CHUNK, 0, lane,
                                                   (uint32_t)(sb & 7u), stop[k]);
    if (lane == 0) {
        a.end[k] = c.end;
        a.olen[k] = c.olen;
        a.status[k] = c.status;
    }
}

/* gz_marker_kernel between bit offsets: chunk j runs from c_start[j] to exactly bit_end[j] */
__global__ void __launch_bounds__(32, 32)
gz_bit_marker_kernel(BgzfGzipArgs a, const uint64_t *bit_end, uint32_t j0, uint64_t base)
{
    __shared__ InfSmem sm;
    const uint32_t lane = threadIdx.x, j = j0 + blockIdx.x;
    const uint64_t sb = a.c_start[j], s = sb >> 3, o = a.c_off[j];
    const uint8_t *lim = a.data + (a.data_len - s > a.max_in ? s + a.max_in : a.data_len);
    const GzChunk c = gz_decode_chunk<true, true>(sm, a.data, a.data + s, lim, sb == 0, a.scratch + GZ_WIN + (o - base), a.c_len[j], o,
                                                  lane, (uint32_t)(sb & 7u), bit_end[j]);
    if (lane == 0) {
        a.lastm[j] = c.lastm;
        if (c.status == GZ_FAIL || c.olen != a.c_len[j] || c.end != bit_end[j]) atomicOr(a.err, c.dist_err ? 1u : 2u);
    }
}

/* one CTA: anchor[j] = no chunk before j (in the batch) has a marker in the 32 KiB before j's first byte (an exclusive prefix max
 * of "scratch position one past the chunk's last marker"; the batch's first chunk sees only the prefix: bytes) */
__global__ void __launch_bounds__(1024, 1)
gz_anchor_kernel(BgzfGzipArgs a, uint32_t j0, uint32_t j1, uint64_t base)
{
    __shared__ uint64_t wmax[32];
    __shared__ uint64_t carry;
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    if (t == 0) carry = 0;
    __syncthreads();
    for (uint32_t b = j0; b < j1; b += 1024) {
        const uint32_t j = b + t;
        uint64_t e = 0, sp = 0;
        if (j < j1) {
            sp = GZ_WIN + a.c_off[j] - base;
            if (a.lastm[j]) e = sp + a.lastm[j];
        }
        uint64_t inc = e;
        for (int s = 1; s < 32; s <<= 1) {
            const uint64_t y = __shfl_up_sync(0xffffffffu, inc, s);
            if (lane >= (uint32_t)s && y > inc) inc = y;
        }
        if (lane == 31) wmax[warp] = inc;
        __syncthreads();
        uint64_t before = carry, all = carry;
        for (uint32_t w = 0; w < 32; w++) {
            if (w < warp && wmax[w] > before) before = wmax[w];
            if (wmax[w] > all) all = wmax[w];
        }
        uint64_t excl = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0 || excl < before) excl = before;
        if (j < j1) a.anchor[j] = excl + GZ_WIN <= sp ? 1u : 0u;
        __syncthreads();
        if (t == 0) carry = all;
        __syncthreads();
    }
}

/* One CTA per anchor: the markers in the last 32 KiB of every chunk from the anchor up to the next one, chunk after chunk.  A
 * marker names a byte of the 32 KiB before its chunk: that lies in the resolved tail of a chunk before it in this run, or — when
 * it is before the anchor — in the anchor's window, which holds bytes only.  Only markers are written, so runs never race. */
#define GZ_RESOLVE_THREADS 1024u
#define GZ_RESOLVE_PER_THREAD (GZ_WIN / GZ_RESOLVE_THREADS)
__global__ void __launch_bounds__(GZ_RESOLVE_THREADS, 1)
gz_resolve_kernel(BgzfGzipArgs a, uint32_t j0, uint32_t j1, uint64_t base)
{
    const uint32_t j = j0 + blockIdx.x;
    if (!a.anchor[j]) return;
    for (uint32_t k = j; k < j1; k++) {
        if (k > j && a.anchor[k]) break;
        const uint32_t m = a.lastm[k], len = a.c_len[k];
        if (m == 0) continue;
        uint16_t *s = a.scratch + GZ_WIN + (a.c_off[k] - base);
        const uint16_t *w = s - GZ_WIN;
        const uint32_t lo = (len > GZ_WIN ? len - GZ_WIN : 0u) + threadIdx.x;
        /* the run is sequential, so a step's latency is what counts: all loads of the tail first, then all window reads,
         * then the stores (with a loop of load -> dependent load -> store per position, whole calls took 16-18 us per chunk) */
        uint16_t v[GZ_RESOLVE_PER_THREAD];
#pragma unroll
        for (uint32_t i = 0; i < GZ_RESOLVE_PER_THREAD; i++) {
            const uint32_t q = lo + i * GZ_RESOLVE_THREADS;
            v[i] = q < m ? s[q] : 0;
        }
#pragma unroll
        for (uint32_t i = 0; i < GZ_RESOLVE_PER_THREAD; i++)
            if (v[i] >= 256) v[i] = w[v[i] - 256] | 0x8000u;     /* (bit 15: resolved here, to be stored) */
#pragma unroll
        for (uint32_t i = 0; i < GZ_RESOLVE_PER_THREAD; i++)
            if (v[i] & 0x8000u) s[lo + i * GZ_RESOLVE_THREADS] = v[i] & 0xffu;
        __syncthreads();
    }
}

/* 16 consecutive output bytes per thread; the chunk of a byte is found by a binary search over the batch's chunk offsets */
#define GZ_NARROW 16u
__global__ void __launch_bounds__(256)
gz_narrow_kernel(BgzfGzipArgs a, uint32_t j0, uint32_t j1, uint64_t base, uint64_t bytes)
{
    const uint64_t q0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * GZ_NARROW;
    if (q0 >= bytes) return;
    uint32_t lo = j0, hi = j1 - 1;                      /* last chunk that starts at or before q0 */
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo + 1) >> 1);
        if (a.c_off[mid] - base <= q0) lo = mid; else hi = mid - 1;
    }
    uint32_t k = lo;
    uint64_t ks = a.c_off[k] - base;
    const uint16_t *s = a.scratch + GZ_WIN;
    uint8_t b[GZ_NARROW];
    const uint32_t cnt = bytes - q0 < GZ_NARROW ? (uint32_t)(bytes - q0) : GZ_NARROW;
#pragma unroll
    for (uint32_t i = 0; i < GZ_NARROW; i++) {
        if (i >= cnt) break;
        const uint64_t q = q0 + i;
        while (k + 1 < j1 && a.c_off[k + 1] - base <= q) ks = a.c_off[++k] - base;
        uint16_t v = s[q];
        if (v >= 256) v = s[ks - GZ_WIN + (v - 256)];
        b[i] = (uint8_t)v;
    }
    uint8_t *dst = a.out + base + q0;
    if (cnt == GZ_NARROW && ((uintptr_t)dst & 15u) == 0) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = b[4 * i] | (b[4 * i + 1] << 8) | (b[4 * i + 2] << 16) | ((uint32_t)b[4 * i + 3] << 24);
        *(uint4 *)dst = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
        for (uint32_t i = 0; i < cnt; i++) dst[i] = b[i];
    }
}

/* ---- random access through a checkpoint index: runs of chunks, each from an access point, each behind its own window ----
 * A batch lays its runs out back to back in scratch: 32 KiB of window (u16 bytes), then the run's chunks.  c_off[j] is a
 * chunk's place in that layout (so the anchor, resolve and narrow passes work unchanged: the window is a run of bytes that
 * separates a run from the markers of the one before it), m_off[j] its offset in the member (the "reference before the
 * member start" check). */

/* scratch[dst[r], + GZ_WIN) = window r, widened and right-aligned; zeros before a window shorter than 32 KiB (the member start) */
__global__ void __launch_bounds__(256)
gz_window_kernel(uint16_t *scratch, const uint8_t *win, const uint64_t *src, const uint32_t *len, const uint64_t *dst)
{
    const uint32_t r = blockIdx.x, n = len[r], pad = GZ_WIN - n;
    uint16_t *d = scratch + dst[r];
    for (uint32_t i = threadIdx.x; i < GZ_WIN; i += blockDim.x) d[i] = i >= pad ? win[src[r] + (i - pad)] : 0;
}

/* gz_marker_kernel for a run layout (chunks [0, gridDim.x) of the batch) */
__global__ void __launch_bounds__(32, 32)
gz_run_marker_kernel(BgzfGzipArgs a, const uint64_t *m_off)
{
    __shared__ InfSmem sm;
    const uint32_t lane = threadIdx.x, j = blockIdx.x;
    const uint64_t s = a.c_start[j], o = a.c_off[j];
    const uint8_t *lim = a.data + (a.data_len - s > a.max_in ? s + a.max_in : a.data_len);
    const GzChunk c = gz_decode_chunk<true>(sm, a.data, a.data + s, lim, false, a.scratch + GZ_WIN + o, a.c_len[j], m_off[j], lane);
    if (lane == 0) {
        a.lastm[j] = c.lastm;
        if (c.status == GZ_FAIL || c.olen != a.c_len[j]) atomicOr(a.err, c.dist_err ? 1u : 2u);
    }
}

extern "C" cudaError_t bgzf_launch_gzip_runs(const BgzfGzipArgs *a, const BgzfGzipRunArgs *r, uint64_t bytes, cudaStream_t stream)
{
    if (r->nchunks == 0) return cudaSuccess;
    if (r->nwin) gz_window_kernel<<<r->nwin, 256, 0, stream>>>(a->scratch, r->win, r->win_src, r->win_len, r->win_dst);
    gz_run_marker_kernel<<<r->nchunks, 32, 0, stream>>>(*a, r->m_off);
    gz_anchor_kernel<<<1, 1024, 0, stream>>>(*a, 0, r->nchunks, 0);
    gz_resolve_kernel<<<r->nchunks, GZ_RESOLVE_THREADS, 0, stream>>>(*a, 0, r->nchunks, 0);
    const uint64_t threads = (bytes + GZ_NARROW - 1) / GZ_NARROW;
    if (threads) gz_narrow_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(*a, 0, r->nchunks, 0, bytes);
    return cudaGetLastError();
}

extern "C" size_t bgzf_gzip_tiles(uint64_t data_len) { return (size_t)((data_len + GZ_TILE - 1) / GZ_TILE); }
extern "C" size_t bgzf_gzip_window(void) { return GZ_WIN; }

extern "C" cudaError_t bgzf_launch_gzip_count(const BgzfGzipArgs *a, cudaStream_t stream)
{
    const uint32_t tiles = (uint32_t)bgzf_gzip_tiles(a->data_len);
    if (tiles == 0) return cudaErrorInvalidValue;
    gz_cand_scan_kernel<<<tiles, GZ_THREADS, 0, stream>>>(a->data, a->data_len, a->tile_count, nullptr, nullptr, nullptr, 0);
    return bgzf_launch_scan(a->tile_count, a->tile_off, tiles, nullptr, nullptr, a->counts, stream);
}

extern "C" cudaError_t bgzf_launch_gzip_chain(const BgzfGzipArgs *a, uint32_t ncand, cudaStream_t stream)
{
    const uint32_t tiles = (uint32_t)bgzf_gzip_tiles(a->data_len);
    gz_cand_scan_kernel<<<tiles, GZ_THREADS, 0, stream>>>(a->data, a->data_len, a->tile_count, a->tile_off, a->cand, a->counts, 1);
    gz_bound_kernel<<<ncand, 32, 0, stream>>>(*a);
    gz_next_kernel<<<(ncand + 2 + 255) / 256, 256, 0, stream>>>(*a);
    cudaError_t e = bgzf_launch_chain(a->cand, a->ncand, ncand, a->jump, a->jump2, a->reach, a->chain_status, stream);
    if (e != cudaSuccess) return e;
    bgzf_launch_scan(a->reach, a->pick, ncand, a->ncand, nullptr, a->counts + 2, stream);
    gz_pick_kernel<<<(ncand + 255) / 256, 256, 0, stream>>>(*a);
    bgzf_launch_scan(a->c_len, a->c_off, ncand, a->nchunks, nullptr, a->total, stream);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_gzip_batch(const BgzfGzipArgs *a, uint32_t j0, uint32_t j1, uint64_t base, uint64_t bytes,
                                              const uint64_t *bit_end, cudaStream_t stream)
{
    if (j1 <= j0) return cudaSuccess;
    gz_prefix_kernel<<<32, 256, 0, stream>>>(*a, base);
    if (bit_end) gz_bit_marker_kernel<<<j1 - j0, 32, 0, stream>>>(*a, bit_end, j0, base);
    else gz_marker_kernel<<<j1 - j0, 32, 0, stream>>>(*a, j0, base);
    gz_anchor_kernel<<<1, 1024, 0, stream>>>(*a, j0, j1, base);
    gz_resolve_kernel<<<j1 - j0, GZ_RESOLVE_THREADS, 0, stream>>>(*a, j0, j1, base);
    const uint64_t threads = (bytes + GZ_NARROW - 1) / GZ_NARROW;
    if (threads) gz_narrow_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(*a, j0, j1, base, bytes);
    return cudaGetLastError();
}

extern "C" size_t bgzf_gzip_region(void) { return GZ_REGION; }

extern "C" cudaError_t bgzf_launch_gzip_search(const BgzfGzipArgs *a, uint32_t nreg, uint64_t *found, cudaStream_t stream)
{
    if (nreg < 2) return cudaSuccess;
    gz_search_kernel<<<(nreg - 1 + GZ_SEARCH_WARPS - 1) / GZ_SEARCH_WARPS, GZ_SEARCH_WARPS * 32, 0, stream>>>(a->data, a->data_len, nreg, found);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_gzip_bit_bound(const BgzfGzipArgs *a, const uint64_t *stop, uint32_t n, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    gz_bit_bound_kernel<<<n, 32, 0, stream>>>(*a, stop);
    return cudaGetLastError();
}
