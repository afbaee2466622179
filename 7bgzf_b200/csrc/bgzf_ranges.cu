/*
 * bgzf_ranges.cu — random access: the planning and the gather around the unchanged inflate kernel.
 *
 *   bgzf_range_plan_kernel    one thread per requested range: first / last member, length, +1/-1 into a difference array
 *                             over the members (device-resident variant; the host variant plans on the host)
 *   bgzf_range_touch_kernel   one CTA: the scan of that difference array ("touched"), the compaction of the touched members
 *                             with their scratch offsets (a scan of ISIZE), and the scans of the range lengths and tile counts
 *   bgzf_range_gather_kernel  one CTA per 32 KiB tile of a range: copies the requested bytes out of the decoded members
 *                             (scratch, every touched member once, in member order) to the caller's output, in caller order
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "bgzf_kernels.h"

#define RNG_THREADS 1024u
#define GATHER_THREADS 256u

/* ---- plan ---- */

/* largest i in [0, n) with a[i] <= x (a ascending, a[0] <= x) */
__device__ __forceinline__ uint32_t rng_last_le(const uint64_t *a, uint32_t n, uint64_t x)
{
    uint32_t lo = 0, hi = n;                 /* first index with a[i] > x */
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (a[mid] <= x) lo = mid + 1; else hi = mid;
    }
    return lo - 1;
}

/* a BGZF virtual offset -> uncompressed position; false if coffset is no member start (or the end of the stream with
 * uoffset 0) or uoffset is past the member's ISIZE */
__device__ __forceinline__ bool rng_resolve(const BgzfRangePlanArgs &a, uint32_t n, uint64_t total, uint64_t v, uint64_t *pos)
{
    const uint64_t c = v >> 16, u = v & 0xffffu;
    if (c == a.in_bytes) {
        *pos = total;
        return u == 0;
    }
    if (n == 0 || c < a.in_off[0]) return false;
    const uint32_t m = rng_last_le(a.in_off, n, c);
    if (a.in_off[m] != c || u > a.isize[m]) return false;
    *pos = a.out_off[m] + u;
    return true;
}

__global__ void __launch_bounds__(256)
bgzf_range_plan_kernel(BgzfRangePlanArgs a)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.nranges) return;
    const uint32_t n = (uint32_t)*a.nmembers;
    const uint64_t total = *a.total;
    uint64_t beg = a.ranges[2 * i], end = a.ranges[2 * i + 1];
    bool ok = true;
    if (a.voffsets) ok = rng_resolve(a, n, total, beg, &beg) && rng_resolve(a, n, total, end, &end);
    ok = ok && beg <= end && end <= total;
    const uint64_t len = ok ? end - beg : 0;
    uint32_t first = 0;
    uint64_t delta = 0;
    if (len) {
        /* the member holding byte `beg` (an empty member shares its start with the next one and never starts a range) and
         * the one holding byte end - 1 */
        first = rng_last_le(a.out_off, n, beg);
        const uint32_t last = rng_last_le(a.out_off, n, end - 1);
        delta = beg - a.out_off[first];
        atomicAdd(&a.diff[first], 1);
        atomicAdd(&a.diff[last + 1], -1);
    }
    if (!ok) atomicOr(a.status, 1u);
    a.first[i] = first;
    a.delta[i] = delta;
    a.len[i] = len;
}

/* ---- touch: one CTA of 1024 threads, chunks of 1024 with running carries ---- */

template <typename T>
__device__ __forceinline__ T rng_block_scan(T v, T *wsum, T *total)
{
    const uint32_t t = threadIdx.x, lane = t & 31u, warp = t >> 5;
    T inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += y;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        T w = wsum[lane], wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= (uint32_t)d) wi += y;
        }
        wsum[lane] = wi - w;                  /* exclusive warp offsets */
        if (lane == 31) wsum[32] = wi;
    }
    __syncthreads();
    const T ex = wsum[warp] + inc - v;
    *total = wsum[32];
    __syncthreads();                          /* (wsum is reused by the next call) */
    return ex;
}

__global__ void __launch_bounds__(RNG_THREADS, 1)
bgzf_range_touch_kernel(BgzfRangeTouchArgs a)
{
    __shared__ int32_t ws_i[33];
    __shared__ uint32_t ws_u[33];
    __shared__ unsigned long long ws_l[33];
    const uint32_t t = threadIdx.x;
    int32_t cover = 0;
    uint32_t nt = 0;
    unsigned long long soff = 0;
    for (uint32_t start = 0; start < a.nmembers; start += RNG_THREADS) {
        const uint32_t m = start + t;
        int32_t tot_i;
        uint32_t tot_u;
        unsigned long long tot_l;
        const int32_t d = m < a.nmembers ? a.diff[m] : 0;
        const int32_t c = cover + rng_block_scan<int32_t>(d, ws_i, &tot_i) + d;   /* ranges covering member m */
        const uint32_t touched = m < a.nmembers && c > 0 ? 1u : 0u;
        const unsigned long long sz = touched ? a.isize[m] : 0u;
        const uint32_t k = nt + rng_block_scan<uint32_t>(touched, ws_u, &tot_u);
        const unsigned long long s = soff + rng_block_scan<unsigned long long>(sz, ws_l, &tot_l);
        if (touched) {
            a.t_in_off[k] = a.in_off[m];
            a.t_soff[k] = s;
            a.m_soff[m] = s;
        }
        cover += tot_i;
        nt += tot_u;
        soff += tot_l;
    }
    __syncthreads();                          /* m_soff of every member is written before the ranges read it */
    unsigned long long out = 0, tiles = 0;
    for (uint32_t start = 0; start < a.nranges; start += RNG_THREADS) {
        const uint32_t i = start + t;
        unsigned long long tot_o, tot_t;
        const unsigned long long len = i < a.nranges ? a.len[i] : 0ull;
        const unsigned long long nti = (len + BGZF_GATHER_TILE - 1) / BGZF_GATHER_TILE;
        const unsigned long long o = out + rng_block_scan<unsigned long long>(len, ws_l, &tot_o);
        const unsigned long long tt = tiles + rng_block_scan<unsigned long long>(nti, ws_l, &tot_t);
        if (i < a.nranges) {
            a.range_off[i] = o;
            a.tile_off[i] = tt;
            a.src[i] = len ? a.m_soff[a.first[i]] + a.delta[i] : 0ull;
        }
        out += tot_o;
        tiles += tot_t;
    }
    if (t == 0) {
        a.counts[0] = nt;
        a.counts[1] = soff;
        a.counts[2] = out;
        a.counts[3] = tiles;
    }
}

/* ---- gather ---- */

/* 16 bytes starting `Q * 4 + r / 8` bytes into w0 || w1 */
template <int Q>
__device__ __forceinline__ uint4 rng_realign(const uint4 w0, const uint4 w1, uint32_t r)
{
    const uint32_t x[8] = { w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w };
    uint4 o;
    o.x = __funnelshift_r(x[Q], x[Q + 1], r);
    o.y = __funnelshift_r(x[Q + 1], x[Q + 2], r);
    o.z = __funnelshift_r(x[Q + 2], x[Q + 3], r);
    o.w = __funnelshift_r(x[Q + 3], x[Q + 4], r);
    return o;
}

/* words aligned 16-byte destination words from a source that is `Q * 4 + r / 8` bytes past the aligned words at `s` */
template <int Q>
__device__ __forceinline__ void rng_copy_words(uint4 *d, const uint4 *s, uint32_t words, uint32_t r)
{
    for (uint32_t j = threadIdx.x; j < words; j += GATHER_THREADS)
        d[j] = rng_realign<Q>(s[j], s[j + 1], r);
}

__global__ void __launch_bounds__(GATHER_THREADS)
bgzf_range_gather_kernel(BgzfRangeGatherArgs a)
{
    const uint64_t tile = blockIdx.x;
    /* the range this tile belongs to: the last i with tile_off[i] <= tile (an empty range shares its tile_off with the
     * next one and owns no tile) */
    uint32_t lo = 0, hi = a.nranges;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (a.tile_off[mid] <= tile) lo = mid + 1; else hi = mid;
    }
    if (lo == 0) return;
    const uint32_t i = lo - 1;
    const uint64_t len = a.len[i], src = a.src[i];
    const uint64_t b0 = (tile - a.tile_off[i]) * BGZF_GATHER_TILE;
    if (b0 >= len) return;
    const uint64_t b1 = b0 + BGZF_GATHER_TILE < len ? b0 + BGZF_GATHER_TILE : len;
    /* the part of this tile whose decoded bytes are in the scratch window [win_lo, win_hi) */
    const uint64_t s0 = src + b0 > a.win_lo ? src + b0 : a.win_lo;
    const uint64_t s1 = src + b1 < a.win_hi ? src + b1 : a.win_hi;
    if (s0 >= s1) return;
    const uint8_t *s = a.scratch + (s0 - a.win_lo);
    uint8_t *d = a.out + a.range_off[i] + (s0 - src);
    const uint32_t n = (uint32_t)(s1 - s0);
    const uint32_t t = threadIdx.x;
    /* bytes up to the first 16-byte boundary of the destination, then aligned 16-byte stores fed by aligned 16-byte loads
     * shifted into place (the source's misalignment is the same for every word of the tile), then the tail */
    uint32_t head = (uint32_t)((16u - ((uintptr_t)d & 15u)) & 15u);
    if (head > n) head = n;
    if (t < head) d[t] = s[t];
    const uint32_t words = (n - head) >> 4;
    if (words) {
        const uint8_t *sp = s + head;
        const uint32_t mis = (uint32_t)((uintptr_t)sp & 15u), r = (mis & 3u) * 8u;
        const uint4 *sw = (const uint4 *)(sp - mis);          /* (reads up to 16 bytes past the source: the scratch is padded) */
        uint4 *dw = (uint4 *)(d + head);
        switch (mis >> 2) {
        case 0: rng_copy_words<0>(dw, sw, words, r); break;
        case 1: rng_copy_words<1>(dw, sw, words, r); break;
        case 2: rng_copy_words<2>(dw, sw, words, r); break;
        default: rng_copy_words<3>(dw, sw, words, r); break;
        }
    }
    const uint32_t done = head + words * 16u;
    if (t < n - done) d[done + t] = s[done + t];
}

extern "C" cudaError_t bgzf_launch_range_plan(const BgzfRangePlanArgs *a, cudaStream_t stream)
{
    if (a->nranges == 0) return cudaSuccess;
    bgzf_range_plan_kernel<<<(a->nranges + 255u) / 256u, 256, 0, stream>>>(*a);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_range_touch(const BgzfRangeTouchArgs *a, cudaStream_t stream)
{
    bgzf_range_touch_kernel<<<1, RNG_THREADS, 0, stream>>>(*a);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_range_gather(const BgzfRangeGatherArgs *a, uint64_t ntiles, cudaStream_t stream)
{
    if (ntiles == 0 || a->nranges == 0) return cudaSuccess;
    if (ntiles > 0x7fffffffull) return cudaErrorInvalidValue;
    bgzf_range_gather_kernel<<<(unsigned)ntiles, GATHER_THREADS, 0, stream>>>(*a);
    return cudaGetLastError();
}
