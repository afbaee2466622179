/*
 * bgzf_compress.cu — sm_100a BGZF compress kernels.
 *
 *   bgzf_compress_kernel : persistent, one CTA (1024 threads) per SM; each CTA takes BGZF blocks b, b+grid, ...
 *       1. the <=64 KiB payload is staged into shared memory with one TMA bulk copy (cp.async.bulk + mbarrier)
 *       2. CRC-32 slices + literal census, hash of every position             (bgzf_block.h phases)
 *       3. hash chains: equal-hash lanes found with one ballot per hash bit (all warps), then linked through the
 *          head table by a relay of 4 warps taking turns tile by tile (position order => deterministic)
 *       4. all-position chain search, 1024 positions at a time, results to an L2-resident scratch
 *          (levels 10-12: up to four matches per position, then min-cost-path passes, one warp per 1/32 of the block)
 *       5. local lazy rule -> step codes, per-chunk jump table, chunk-to-chunk walk
 *       6. histograms, length-limited Huffman (keys ranked by comparison, two-queue merge, parallel depths), block type choice
 *       7. per-chunk bit sizes, block-wide prefix sums, parallel bit packing, BGZF header/BSIZE/CRC/ISIZE
 *   bgzf_scan_kernel / bgzf_gather_kernel : exclusive scan of member sizes and compaction of the
 *       fixed-stride slots into one contiguous BGZF stream (+ the 28-byte EOF marker).
 *
 * Shared memory map (bytes): [0,65568) payload | [65568,196640) region A | [196640,229408) region B |
 * crc table 1 KiB | literal flags | scalars | mbarrier | scan scratch  = 230,968 B of the 232,448 B a CTA may own.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstring>

#include "bgzf_block.h"
#include "bgzf_kernels.h"

#define SM_DATA 0u
#define SM_REGA (BG_DATA_BYTES)
#define SM_REGB (SM_REGA + 131072u)
#define SM_CRCTAB (SM_REGB + 32768u)
#define SM_LITFLAG (SM_CRCTAB + 1024u)
#define SM_SCAL (SM_LITFLAG + 256u)
#define SM_MBAR (SM_SCAL + 4u * BG_S_COUNT)
#define SM_FRONTIER (SM_MBAR + 8u)
#define SM_SCAN (SM_MBAR + 16u)
#define SM_READY (SM_SCAN + 4u * 36u)       /* u8[128]: tile k's peers are found (the peers -> link pipeline) */
#define SM_TOTAL (SM_READY + 128u)

extern "C" size_t bgzf_compress_smem_bytes(void) { return SM_TOTAL; }

/* ---- TMA bulk copy + mbarrier (PTX ISA: cp.async.bulk, mbarrier) ---- */
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

/* ---- hash chains: prev[p] = nearest earlier position with p's hash (exactly what a sequential insert gives).
 * Two phases, so that only a thin loop stays sequential:
 *   A (all warps)  per group of 32 consecutive positions, find the lanes that share a hash with one ballot per
 *                  hash bit (match.any serialises over distinct values: 400+ cycles per group here).  A lane
 *                  with a lower peer gets its final link at once; the lowest lane of each peer set keeps its
 *                  hash and notes (hi[] byte, in the L2-resident scratch) which lane is the highest peer.
 *   B (warp 0)     walks the groups in order: every noted lane reads head[hash] as its link and stores the
 *                  highest peer's position as the new head.  ~12 instructions per group. ---- */
__device__ __forceinline__ unsigned hash_peers(uint32_t h, bool valid)
{
    unsigned peers = __ballot_sync(0xffffffffu, valid);
    /* per hash bit: the vote, the lane's bit as a mask (SEL) and peers &= ~(ballot ^ mask) in one LOP3; ptxas takes the
     * predicates for 7 bits at a time from h with one R2P.  (Written in C, the same step compiles to six instructions.) */
#pragma unroll
    for (int k = 0; k < BG_HASH_BITS; k++) {
        asm volatile("{\n\t.reg .pred p;\n\t.reg .b32 b, t;\n\t"
                     "and.b32 t, %1, %2;\n\t"
                     "setp.ne.u32 p, t, 0;\n\t"
                     "vote.sync.ballot.b32 b, p, 0xffffffff;\n\t"
                     "selp.b32 t, -1, 0, p;\n\t"
                     "lop3.b32 %0, %0, b, t, 0x90;\n\t}"
                     : "+r"(peers)
                     : "r"(h), "r"(1u << k));
    }
    return peers;
}

/* bg_hash for any window width without a branch: the second word contributes nothing for 3 and 4 bytes, its low byte for 5,
 * all of it for 8 (the block is followed by zero bytes: the second word of a position near the end stays inside the buffer) */
__device__ __forceinline__ uint32_t hash_any_width(const uint32_t *dataw, uint32_t p, uint32_t m0, uint32_t m1)
{
    const uint32_t v0 = bg_ld32(dataw, p) & m0, v1 = bg_ld32(dataw, p + 4u) & m1;
    return ((v0 * 0x1E35A7BDu) ^ (v1 * 0x9E3779B1u)) >> (32 - BG_HASH_BITS);
}

/* notes layout: tile = 16 consecutive groups (512 positions); tile i holds 32 lanes x 16 bytes, so that in phase
 * B each lane fetches the notes of its next 16 groups with one coalesced 16-byte load, a whole tile ahead. */
/* (first, step, xprev): a CTA of a cluster takes tiles first, first + step, ... and also leaves each finished tile of
 * prev[] in global memory for the other CTAs (import_peer_tiles); the one-CTA kernel passes 0, 1, nullptr */
/* (warp, nwarps): the producer warps share the tiles, warp k of nwarps taking tiles first + step * (k, k + nwarps, ...);
 * ready (optional): one flag per tile in shared memory, raised when the tile's links and notes are out — the linking
 * relay (build_link_phase) runs at the same time on other warps and waits for it */
__device__ __forceinline__ void build_peers_phase(const BgCtx &c, uint4 *notes, uint32_t lane, uint32_t warp, uint32_t nwarps, uint32_t first,
                                                  uint32_t step, uint4 *xprev, volatile uint8_t *ready, unsigned long long *prof, long long t0)
{
    const uint32_t n = c.n, hb = c.scal[BG_S_HBYTES];
    const uint32_t m0 = hb == 3 ? 0xffffffu : 0xffffffffu, m1 = hb == 8 ? 0xffffffffu : hb == 5 ? 0xffu : 0u;
    BG_ASSERT(hb == 3 || hb == 4 || hb == 5 || hb == 8);
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t ntiles = (n + 511u) >> 9;
    for (uint32_t tile = first + step * warp; tile < ntiles; tile += step * nwarps) {
        uint32_t w[4] = { 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu };
#pragma unroll
        for (uint32_t g = 0; g < 16; g++) {
            const uint32_t base = tile * 512u + g * 32u;
            if (base >= n) break;               /* uniform for the warp */
            const uint32_t p = base + lane;
            /* (the hash phase proper is folded in: a position's hash goes straight from the multiply into the ballots) */
            const bool valid = p + hb <= n;
            const uint32_t h = valid ? hash_any_width(c.dataw, p, m0, m1) : BG_NOPOS;
            const unsigned peers = hash_peers(h, valid);
            uint32_t link = h;                                            /* a leader keeps its hash for the relay; no hash window: BG_NOPOS */
            if (valid) {
                const unsigned lower = peers & lt;
                if (lower) {
                    link = base + (31u - (uint32_t)__clz(lower));
                } else {
                    const uint32_t note = 31u - (uint32_t)__clz(peers);   /* lane of the highest position with this hash */
                    w[g >> 2] = (w[g >> 2] & ~(0xffu << (8 * (g & 3)))) | (note << (8 * (g & 3)));
                }
            }
            if (p < n) c.prev[p] = (uint16_t)link;
        }
        notes[tile * 32u + lane] = make_uint4(w[0], w[1], w[2], w[3]);
        if (xprev) {
            __syncwarp();
            const uint4 *ts = (const uint4 *)(c.prev + tile * 512u);      /* 1 KiB of links: two 16-byte pieces per lane */
            xprev[tile * 64u + lane] = ts[lane];
            xprev[tile * 64u + 32u + lane] = ts[32u + lane];
        }
        if (ready) {
            __threadfence_block();
            __syncwarp();
            if (lane == 0) ready[tile] = 1;
            if (prof && lane == 0) atomicAdd(&prof[BGZF_PROF_READY + tile], (unsigned long long)(clock64() - t0));
        }
    }
}

/* the other CTAs' tiles of prev[], after the cluster barrier: 64 pieces of 16 bytes per tile */
__device__ __forceinline__ void import_peer_tiles(const BgCtx &c, const uint4 *xprev, uint32_t t, uint32_t rank, uint32_t parts)
{
    const uint32_t pieces = ((c.n + 511u) >> 9) * 64u;
    uint4 *dst = (uint4 *)c.prev;
    for (uint32_t i = t; i < pieces; i += BG_THREADS)
        if ((i >> 6) % parts != rank) dst[i] = __ldcg(xprev + i);
}

/* Phase B, a relay of BG_LINKERS warps: warp k takes tiles k, k+BG_LINKERS, ...  Only the head-table part of a tile
 * must run in tile order (and inside it, group order: shared-memory instructions of one warp execute in program order,
 * the accesses are volatile so the compiler keeps that order); it is entered when the `turn` word in shared memory
 * reaches the tile and hands the turn on as soon as its last head update is out.  Fetching the notes and the
 * leaders' hashes before, and storing the links after, overlap with the other warps' turns.
 * The ordered section was the critical path of the chain build (profiles/r03_link_split.txt: the relay handed on its
 * last turn 28 k cycles after the last producer was done) and it competes for issue slots with 28 producer warps, so it
 * is kept to three instructions per group: every access is prepared before the turn as one word, head byte offset << 16 |
 * new head, and lanes without a leader go to a sink word instead of being predicated.  The turn is handed on with a
 * release store and taken with an acquire load (one MEMBAR.ALL.CTA by the passing lane instead of two MEMBAR.SC.CTA
 * per lane). */
#define BG_LINKERS 4u
#define BG_LINK_SINK (SM_SCAN + 4u * 33u - SM_REGB)   /* byte offset from head[] of a u16 nobody reads (scan scratch word 33) */
__device__ __forceinline__ uint32_t ld_acquire_cta(const volatile uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32((const void *)p)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_cta(volatile uint32_t *p, uint32_t v)
{
    asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(smem_u32((const void *)p)), "r"(v) : "memory");
}
/* prof (optional): cycles since t0 at which each tile's turn is taken; the relay's waits on ready[] and on `turn` */
__device__ __forceinline__ void build_link_phase(const BgCtx &c, const uint4 *notes, uint32_t warp, uint32_t lane, volatile uint32_t *turn,
                                                 volatile uint8_t *ready, unsigned long long *prof, long long t0)
{
    const uint32_t n = c.n;
    const uint32_t ntiles = (n + 511u) >> 9;
    volatile uint8_t *vhead = (volatile uint8_t *)c.head;
    static_assert(BG_LINK_SINK >= 2u * BG_HASH_SIZE && BG_LINK_SINK < 65536u, "the sink lies outside head[] and within 16 bits");
    for (uint32_t tile = warp; tile < ntiles; tile += BG_LINKERS) {
        BG_ASSERT(tile < 128u);
        const long long w0 = prof ? clock64() : 0;
        if (ready) {
            while (!ready[tile]) __nanosleep(40);
            __threadfence_block();
        }
        const long long w1 = prof ? clock64() : 0;
        const uint4 cur = __ldcg(notes + tile * 32u + lane);
        const uint32_t w[4] = { cur.x, cur.y, cur.z, cur.w };
        /* the hash slots of this tile's leaders are untouched until their links are stored below: fetch them all now */
        uint32_t op[16];
#pragma unroll
        for (uint32_t g = 0; g < 16; g++) {
            const uint32_t note = (w[g >> 2] >> (8 * (g & 3))) & 0xffu;
            const uint32_t h = c.prev[tile * 512u + g * 32u + lane];
            BG_ASSERT(note == 0xffu || h < BG_HASH_SIZE);
            op[g] = note != 0xffu ? (h << 17) | (tile * 512u + g * 32u + note) : BG_LINK_SINK << 16;
        }
        const long long w2 = prof ? clock64() : 0;
        while (ld_acquire_cta(turn) != tile) {}
        const long long w3 = prof ? clock64() : 0;
        uint32_t old[16];
#pragma unroll
        for (uint32_t g = 0; g < 16; g++) {
            volatile uint16_t *slot = (volatile uint16_t *)(vhead + (op[g] >> 16));
            old[g] = *slot;
            *slot = (uint16_t)op[g];
        }
        __syncwarp();
        if (lane == 0) st_release_cta(turn, tile + 1);
        if (prof && lane == 0) {
            atomicAdd(&prof[23], (unsigned long long)(w1 - w0));
            atomicAdd(&prof[24], (unsigned long long)(w3 - w2));
            atomicAdd(&prof[BGZF_PROF_TURN + tile], (unsigned long long)(w3 - t0));
            if (tile + 1 == ntiles) atomicAdd(&prof[25], (unsigned long long)(clock64() - t0));
        }
#pragma unroll
        for (uint32_t g = 0; g < 16; g++)
            if ((op[g] >> 16) != BG_LINK_SINK) c.prev[tile * 512u + g * 32u + lane] = (uint16_t)old[g];
    }
}

/* ---- the search of the greedy / lazy classes (bgzf_block.h: "the search in three passes").  `own`/`parts`: CTA `own` of
 * a cluster of `parts` that shares ONE block keeps every parts-th group of 32 positions (the one-CTA kernel: 0, 1). ---- */

/* a bit of the landing bitmap of CTA `owner` of this cluster (distributed shared memory: mapa + red.or) */
__device__ __forceinline__ void mark_remote(uint32_t *local_word, uint32_t owner, uint32_t bits)
{
    uint32_t raddr;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(smem_u32(local_word)), "r"(owner));
    asm volatile("red.relaxed.cluster.shared::cluster.or.b32 [%0], %1;" ::"r"(raddr), "r"(bits) : "memory");
}

/* Landing marks for word `word` (32 positions).  One-CTA kernel: a shared-memory atomicOr.  Cluster: the bits go to the CTA
 * that owns the word; its two highest bits also to the owner of the next word, which needs them for the positions the lazy
 * rule looks at right after a landing (bg_phase_search_todo reads them from "the word before"). */
template <bool SPLIT>
__device__ __forceinline__ void mark_bits(uint32_t *mark, uint32_t word, uint32_t bits, uint32_t own, uint32_t parts)
{
    BG_ASSERT(word < 2064u);
    if (!SPLIT) {
        atomicOr(&mark[word], bits);
        return;
    }
    const uint32_t owner = word % parts;
    if (owner == own) atomicOr(&mark[word], bits);
    else mark_remote(&mark[word], owner, bits);
    if (bits & 0xC0000000u) {
        const uint32_t next = (word + 1u) % parts;
        if (next == own) atomicOr(&mark[word], bits & 0xC0000000u);
        else if (next != owner) mark_remote(&mark[word], next, bits & 0xC0000000u);
    }
}

/* pass 1: nearest-candidate match of every position; landing marks and eligibility bits with one ballot per 32 positions.
 * SPLIT: a cluster shares ONE block; CTA `own` of `parts` takes every parts-th group of 32 positions, and a landing
 * mark goes to the bitmap of the CTA that owns the landing position's group (it alone reads that word afterwards). */
template <bool SPLIT, bool H3>
__device__ __forceinline__ void search_nearest_t(const BgCtx &c, uint32_t t, uint32_t own, uint32_t parts)
{
    const uint32_t n = c.n, lane = t & 31u;
    uint32_t *elig = (uint32_t *)(c.regb + BG_B_TODO), *mark = (uint32_t *)(c.regb + BG_B_MARK);
    const BgSearchPrm sp = bg_search_prm(c);
    if (sp.depth <= 1) {                                            /* depth 1 (level 1): the nearest candidate is the whole search */
        const uint32_t hist1 = bg_f_hist(c);
        for (uint32_t p = t; p < n; p += BG_THREADS) {
            if (SPLIT && (p >> 5) % parts != own) continue;
            bool deep;
            uint32_t target;
            c.R[p] = p < hist1 ? 0u : bg_nearest_t<H3>(c, sp, p, &deep, &target);
        }
        return;
    }
    const bool opt = c.prm.opt_passes > 0;
    const uint32_t hist = bg_f_hist(c);                             /* history: never a token, never searched (bg_phase_search1) */
    if (t == 0 && own == 0) mark_bits<SPLIT>(mark, hist >> 5, 1u << (hist & 31u), own, parts);
    for (uint32_t p0 = t - lane; p0 < n; p0 += BG_THREADS) {       /* (warp-uniform trip count) */
        const uint32_t word = p0 >> 5;
        BG_ASSERT(word < 2048u);
        if (SPLIT && word % parts != own) continue;
        const uint32_t p = p0 + lane;
        if (p0 + 32u <= hist) {                                     /* (uniform) */
            c.R[p] = 0;
            if (opt) ((uint4 *)c.cand)[p] = make_uint4(0u, 0u, 0u, 0u);
            continue;
        }
        bool deep = false;
        uint32_t target = p + 1, r = 0;
        const bool live = p < n && p >= hist;
        if (live) r = bg_nearest_t<H3>(c, sp, p, &deep, &target);
        if (p < n) c.R[p] = r;
        if (opt) {
            /* near-optimal class: every eligible position is searched (no landing marks); the nearest match opens its offset range */
            if (p < n) {
                const uint32_t k = r ? bg_off_bin(bg_mw_off(r)) : 4u;
                ((uint4 *)c.cand)[p] = make_uint4(k == 0 ? r : 0u, k == 1 ? r : 0u, k == 2 ? r : 0u, k == 3 ? r : 0u);
            }
            const unsigned em = __ballot_sync(0xffffffffu, deep);
            if (lane == 0) elig[word] = em;
            continue;
        }
        const bool lit = live && target == p + 1;
        const unsigned lm = __ballot_sync(0xffffffffu, lit), em = __ballot_sync(0xffffffffu, deep);
        const uint32_t before = __shfl_up_sync(0xffffffffu, target, 1);
        if (lane == 0) {
            elig[word] = em;
            if (lm << 1) mark_bits<SPLIT>(mark, word, lm << 1, own, parts);
            if (lm >> 31) mark_bits<SPLIT>(mark, word + 1, 1u, own, parts);
        }
        /* consecutive positions inside one match land on the same position: one of them marks it */
        if (live && !lit && (lane == 0 || before != target)) mark_bits<SPLIT>(mark, target >> 5, 1u << (target & 31u), own, parts);
    }
}

template <bool SPLIT>
__device__ __forceinline__ void search_nearest(const BgCtx &c, uint32_t t, uint32_t own, uint32_t parts)
{
    if (c.scal[BG_S_HBYTES] == 3) search_nearest_t<SPLIT, true>(c, t, own, parts);      /* (uniform for the CTA) */
    else search_nearest_t<SPLIT, false>(c, t, own, parts);
}

/* pass 3: up to 32 queued candidates, one per lane: full extension, merged into the position's match word (near-optimal
 * class: also into the word of the candidate's offset range) */
template <bool H3>
__device__ __forceinline__ void drain_queue(const BgCtx &c, const uint32_t *queue, uint32_t from, uint32_t count, uint32_t lane)
{
    if (lane < count) {
        const uint32_t e = queue[from + lane];
        const uint32_t p = e >> 16, q = e & 0xffffu;
        BG_ASSERT(p < c.n && q < p && p - q <= 32768u);
        const uint32_t v = bg_deep_extend(c, H3, p, q);
        if (v) {
            atomicMax(&c.R[p], v);
            if (c.cand) atomicMax(&c.cand[4u * p + bg_off_bin(p - q)], v);
        }
    }
}

/* pass 2 for a batch of todo positions (one per lane): walk the chain beyond the nearest candidate; candidates that agree on
 * the 4 bytes ending just past the nearest match go to the warp's queue (one ballot per chain step places them), which is
 * drained whenever it holds a full batch.  cnt = entries waiting in the queue (warp-uniform, < 32 on entry and on exit). */
template <bool H3>
__device__ __forceinline__ void deep_batch(const BgCtx &c, uint32_t *queue, uint32_t &cnt, uint32_t p, bool active, uint32_t lane)
{
    uint32_t q = BG_NOPOS, b1 = 3, tail = 0;
    int depth = (int)c.scal[BG_S_DEPTH] - 1;
    const unsigned lt = (1u << lane) - 1u;
    uint32_t tmask = 0xffffffffu;
    if (active) {
        const uint32_t r1 = __ldcg(c.R + p);
        b1 = r1 ? r1 >> 16 : 3u;
        tmask = bg_tail_mask(H3, r1);
        tail = bg_ld32(c.dataw, p + b1 - 3u) & tmask;
        q = c.prev[c.prev[p]];
    }
    bool live = active && depth > 0 && bg_in_window(p, q);
    const uint32_t f4 = H3 && active ? bg_ld32(c.dataw, p) : 0u;   /* 3-byte hash window: see BG_DEEP_SCAN */
    int cap = 4 * depth;
    while (__any_sync(0xffffffffu, live)) {
#pragma unroll
        for (uint32_t k = 0; k < BG_SCAN_CHUNK_SHALLOW; k++) {
            bool pass = false;
            const uint32_t qc = q;
            if (live) {
                const uint32_t qn = c.prev[q];
                pass = (bg_ld32(c.dataw, q + b1 - 3u) & tmask) == tail;
                if (!H3 || bg_ld32(c.dataw, q) == f4) depth--;
                if (H3) cap--;
                q = qn;
                live = depth > 0 && (!H3 || cap > 0) && bg_in_window(p, q);
            }
            const unsigned m = __ballot_sync(0xffffffffu, pass);
            if (m) {
                BG_ASSERT(cnt + __popc(m) <= BG_QUEUE_WORDS_SHALLOW);
                if (pass) queue[cnt + __popc(m & lt)] = (p << 16) | qc;
                cnt += __popc(m);
            }
        }
        if (cnt >= 32u) {
            __syncwarp();
            do {
                cnt -= 32u;
                drain_queue<H3>(c, queue, cnt, 32u, lane);
            } while (cnt >= 32u);
            __syncwarp();
            /* some of this position's candidates may have been measured by now: test the rest of the chain against the longer
             * match.  (Whenever this happens, the final word is the same: a candidate is only ever dropped for not being
             * longer than a nearer one that has already been measured.) */
            if (live) {
                const uint32_t r = __ldcg(c.R + p);
                if ((r >> 16) > b1) {
                    b1 = r >> 16;
                    tmask = 0xffffffffu;
                    uint32_t maxl = c.n - p;
                    if (maxl > 258u) maxl = 258u;
                    if (b1 >= maxl) live = false;
                    else tail = bg_ld32(c.dataw, p + b1 - 3u);
                }
            }
        }
    }
}

template <bool H3>
__device__ __forceinline__ void search_deep_batches(const BgCtx &c, uint32_t t, uint32_t own, uint32_t parts)
{
    const uint32_t lane = t & 31u, warp = t >> 5;
    const uint32_t *todo = (const uint32_t *)(c.regb + BG_B_TODO);
    uint32_t *queue = (uint32_t *)(c.regb + BG_B_QUEUE) + warp * BG_QUEUE_WORDS_SHALLOW;
    volatile uint16_t *gather = (volatile uint16_t *)(c.regb + BG_B_RING) + warp * 64u;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t nwords = (c.n + 31u) >> 5;
    uint32_t fill = 0, cnt = 0;                                  /* todo positions waiting in gather[], candidates in queue[] (warp-uniform) */
    /* warp w takes every 32nd of this CTA's words (32 positions each): records alternate between cheap (sequence) and
     * deep (quality) stretches, so the work spreads evenly */
    for (uint32_t i = own + parts * warp; i < nwords; i += parts * (BG_THREADS / 32u)) {
        const uint32_t w = todo[i];
        if (w == 0) continue;
        BG_ASSERT(fill + __popc(w) <= 64u);
        if ((w >> lane) & 1u) gather[fill + __popc(w & lt)] = (uint16_t)(i * 32u + lane);
        fill += __popc(w);
        __syncwarp();
        if (fill >= 32u) {
            const uint32_t p = gather[lane];
            const uint32_t rest = lane + 32u < fill ? gather[lane + 32u] : 0u;
            __syncwarp();
            if (lane + 32u < fill) gather[lane] = (uint16_t)rest;
            fill -= 32u;
            deep_batch<H3>(c, queue, cnt, p, true, lane);
        }
    }
    __syncwarp();
    if (fill) deep_batch<H3>(c, queue, cnt, lane < fill ? gather[lane] : 0u, lane < fill, lane);
    __syncwarp();
    drain_queue<H3>(c, queue, 0u, cnt, lane);
}

__device__ __forceinline__ void cp_async4(void *dst_smem, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

/* pass 2: the deep search of the todo positions.  Every lane walks the chain of ONE position; a lane whose chain has ended
 * takes the next todo position of its warp at once (chains are anything from 1 to `depth` nodes long: a warp that walked 32
 * positions side by side would idle most of its lanes most of the time).  The warp's todo positions wait in a small ring
 * that is topped up from the todo bitmap, and the match word of the nearest candidate — which says what a deeper candidate
 * has to beat — is fetched into the ring with cp.async when the position enters it, a turn or more before a lane needs it.
 * Candidates that agree with the position on the 4 bytes ending just past the match to beat are placed on the warp's queue
 * by one ballot per chain step; the queue is drained whenever it holds a full batch of 32 (pass 3). */
template <bool H3>
__device__ __forceinline__ void search_deep(const BgCtx &c, uint32_t t, uint32_t own, uint32_t parts)
{
    const uint32_t lane = t & 31u, warp = t >> 5;
    const uint32_t *todo = (const uint32_t *)(c.regb + BG_B_TODO);
    uint32_t *queue = (uint32_t *)(c.regb + BG_B_QUEUE) + warp * BG_QUEUE_WORDS;
    volatile uint16_t *ring = (volatile uint16_t *)(c.regb + BG_B_RING) + warp * 64u;
    volatile uint32_t *ringr = (volatile uint32_t *)(c.regb + BG_B_RINGR) + warp * 64u;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t nwords = (c.n + 31u) >> 5;
    const int depth0 = (int)c.scal[BG_S_DEPTH] - 1;
    /* warp w takes every 32nd of this CTA's words (32 positions each): records alternate between cheap (sequence) and
     * deep (quality) stretches, so the work spreads evenly */
    uint32_t word = own + parts * warp;
    const uint32_t wstep = parts * (BG_THREADS / 32u);
    uint32_t head = 0, tail = 0, cnt = 0;                          /* ring [head, tail), queue entries: warp-uniform */
    uint32_t p = 0, q = BG_NOPOS, b1 = 3, tailw = 0, tmask = 0xffffffffu, f4 = 0;
    int depth = 0, cap = 0;
    bool live = false;
    for (;;) {
        /* top the ring up to 32 or more waiting positions */
        while (tail - head < 32u && word < nwords) {
            const uint32_t w = todo[word];
            if (w) {
                BG_ASSERT(tail - head + __popc(w) <= 64u);
                if ((w >> lane) & 1u) {
                    const uint32_t slot = (tail + __popc(w & lt)) & 63u, pos = word * 32u + lane;
                    BG_ASSERT(pos < c.n);
                    ring[slot] = (uint16_t)pos;
                    cp_async4((void *)(ringr + slot), c.R + pos);
                }
                tail += __popc(w);
            }
            word += wstep;
        }
        /* lanes without a chain take the oldest waiting positions */
        const unsigned need = __ballot_sync(0xffffffffu, !live);
        if (need && head != tail) {
            cp_async_wait_all();
            __syncwarp();
            const uint32_t avail = tail - head, rank = __popc(need & lt);
            if (!live && rank < avail) {
                const uint32_t slot = (head + rank) & 63u;
                p = ring[slot];
                const uint32_t r1 = ringr[slot];
                b1 = r1 ? r1 >> 16 : 3u;
                tmask = bg_tail_mask(H3, r1);
                tailw = bg_ld32(c.dataw, p + b1 - 3u) & tmask;
                if (H3) f4 = bg_ld32(c.dataw, p);
                q = c.prev[c.prev[p]];
                depth = depth0;
                cap = 4 * depth0;
                live = depth > 0 && bg_in_window(p, q);
            }
            head += min(avail, (uint32_t)__popc(need));
            __syncwarp();
            if (head != tail || word < nwords) continue;           /* (more may be waiting: fill and hand out again before walking) */
        }
        if (!__any_sync(0xffffffffu, live)) break;
#pragma unroll
        for (uint32_t k = 0; k < BG_SCAN_CHUNK; k++) {
            bool pass = false;
            const uint32_t qc = q;
            if (live) {
                const uint32_t qn = c.prev[q];
                pass = (bg_ld32(c.dataw, q + b1 - 3u) & tmask) == tailw;
                if (!H3 || bg_ld32(c.dataw, q) == f4) depth--;
                if (H3) cap--;
                q = qn;
                live = depth > 0 && (!H3 || cap > 0) && bg_in_window(p, q);
            }
            const unsigned m = __ballot_sync(0xffffffffu, pass);
            if (m) {
                BG_ASSERT(cnt + __popc(m) <= BG_QUEUE_WORDS);
                if (pass) queue[cnt + __popc(m & lt)] = (p << 16) | qc;
                cnt += __popc(m);
            }
        }
        if (cnt >= 32u) {
            __syncwarp();
            do {
                cnt -= 32u;
                drain_queue<H3>(c, queue, cnt, 32u, lane);
            } while (cnt >= 32u);
            __syncwarp();
            /* some of this position's candidates may have been measured by now: test the rest of the chain against the longer
             * match.  (Whenever this happens, the final words are the same where it matters: a candidate is only ever dropped
             * for not being longer than a nearer one that has already been measured.) */
            if (live) {
                const uint32_t r = __ldcg(c.R + p);
                if ((r >> 16) > b1) {
                    b1 = r >> 16;
                    tmask = 0xffffffffu;
                    uint32_t maxl = c.n - p;
                    if (maxl > 258u) maxl = 258u;
                    if (b1 >= maxl) live = false;
                    else tailw = bg_ld32(c.dataw, p + b1 - 3u);
                }
            }
        }
    }
    __syncwarp();
    drain_queue<H3>(c, queue, 0u, cnt, lane);
}

__device__ __forceinline__ uint32_t cluster_rank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_size()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
/* all threads of all CTAs of the cluster; global-memory writes before it are visible after it */
__device__ __forceinline__ void cluster_sync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

/* ---- near-optimal class: one backward min-cost pass, warp w owning segment w.  Same arithmetic as bg_phase_dp().
 * Positions are taken in tiles of 32: each lane fetches the four matches of ITS position of the tile (one coalesced
 * 16-byte load per lane, issued a tile ahead), prices their offsets and its literal, and parks the packed result in a
 * 512-byte staging row of shared memory.  The sequential part then costs, per position: one broadcast 16-byte load
 * of the staged row, the candidate lengths spread over the lanes (lane j prices lengths 3+j, 35+j, ...), one
 * redux.min on the packed (cost, length, candidate) word, and the owning lane (which still holds the offsets in
 * registers) recording cost and decision — nothing on that path goes further than shared memory. ---- */
__device__ __forceinline__ void dp_segment_warp(const BgCtx &c, uint32_t w, uint32_t lane, uint32_t *ring)
{
    uint32_t a, b, e;
    bg_dp_segment_bounds(c.n, w, 32, &a, &b, &e);
    if (a >= b) return;
    const uint8_t *rb = c.regb;
    const uint4 *cand4 = (const uint4 *)c.cand;
    uint4 *stage = (uint4 *)(c.regb + BG_B_XTAB) + w * 32u;        /* the walk tables are dead during the passes */
    if (lane == 0) ring[e & (BG_DP_RING - 1)] = 0;
    const uint4 zero4 = make_uint4(0, 0, 0, 0);
    uint32_t top = e - 1;                                            /* first position of the current tile */
    uint4 next = top >= lane && top - lane >= a ? __ldcg(cand4 + (top - lane)) : zero4;
    for (;;) {
        const uint4 mine = next;
        const uint32_t q = top - lane;                               /* my position of this tile (may be below a: unused) */
        const bool more = top >= a + 32u;
        if (more) next = top - 32u >= lane && top - 32u - lane >= a ? __ldcg(cand4 + (top - 32u - lane)) : zero4;
        {
            /* staged per position: M0..M3 = running maxima of the four ranges' lengths from the nearest range outwards (range k
             * serves the lengths in (M[k-1], M[k]]), the four offset costs, the literal cost */
            uint32_t oc = 0, litc = 0, m0 = 0, m1 = 0, m2 = 0, m3 = 0;
            if (top >= lane && q >= a) {
                const uint32_t cd[4] = { mine.x, mine.y, mine.z, mine.w };
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    uint32_t nbx, exx;
                    if (cd[k]) oc |= (uint32_t)rb[BG_B_OFFCOST + bg_off_slot(bg_mw_off(cd[k]), &nbx, &exx)] << (8 * k);
                }
                m0 = mine.x >> 16;
                m1 = max(m0, mine.y >> 16);
                m2 = max(m1, mine.z >> 16);
                m3 = max(m2, mine.w >> 16);
                litc = rb[BG_B_LITCOST + bg_ld8(c.dataw, q)];
            }
            stage[lane] = make_uint4(m0 | (m1 << 16), m2 | (m3 << 16), oc, litc);
        }
        __syncwarp();
        const uint32_t steps = top - a + 1 < 32u ? top - a + 1 : 32u;
        uint32_t mybest = 0;
        for (uint32_t j = 0; j < steps; j++) {
            const uint32_t p = top - j;
            const uint4 st = stage[j];
            const uint32_t M0 = st.x & 0xffffu, M1 = st.x >> 16, M2 = st.y & 0xffffu, M3 = st.y >> 16;
            uint32_t maxl = e - p;
            if (M3 < maxl) maxl = M3;
            uint32_t best = 0xffffffffu;
            if (lane == 0) best = bg_dp_pack(st.w + ring[(p + 1) & (BG_DP_RING - 1)], 1, 0);
            /* (most matches are shorter than 35: one length per lane; the loop proper is kept rolled so that the common
             * step does not run through an unrolled loop's prologue and remainder code) */
            uint32_t l = 3 + lane;
            if (l <= maxl) {
#pragma unroll 1
                do {
                    const uint32_t k = (l > M0 ? 1u : 0u) + (l > M1 ? 1u : 0u) + (l > M2 ? 1u : 0u);
                    const uint32_t oc = (st.z >> (8 * k)) & 0xffu;
                    const uint32_t v = bg_dp_pack(rb[BG_B_LENCOST + l] + oc + ring[(p + l) & (BG_DP_RING - 1)], l, k);
                    best = v < best ? v : best;
                    l += 32;
                } while (l <= maxl);
            }
            best = __reduce_min_sync(0xffffffffu, best);
            if (lane == j) {
                ring[p & (BG_DP_RING - 1)] = best >> 11;
                mybest = best;                          /* my position's decision: recorded after the tile, all lanes at once */
            }
            __syncwarp();
        }
        if (lane < steps && q < b) {
            const uint32_t l = (mybest >> 2) & 511u, k = mybest & 3u;
            if (l == 1) {
                c.stepcode[q] = 0;
            } else {
                const uint32_t off = bg_mw_off(k == 0 ? mine.x : k == 1 ? mine.y : k == 2 ? mine.z : mine.w);
                c.stepcode[q] = (uint8_t)(l <= 256 ? l - 2 : 255);
                c.R[q] = bg_mw(l, off);
            }
        }
        if (!more) break;
        top -= 32u;
    }
}

/* ---- chunk order of the token passes.  A thread walks the tokens of one 68-byte chunk in tally, sizes and emit; a warp
 * pays for its longest walk and for every kind of token its lanes meet.  Sequence stretches are literal runs (17 steps of
 * four literals), quality stretches a handful of matches: chunks are therefore classed by how many of their positions
 * carry a literal step code, and each warp gets chunks of one class (a stable 8-way partition: ballots per warp, one scan
 * of the 8 x 32 counts).  Only the execution order changes; every chunk's bits are what they would be anyway. ---- */
__device__ __forceinline__ uint32_t chunk_class(const BgCtx &c, uint32_t ch)
{
    if (ch * BG_CHUNK >= c.n) return 0u;
    const uint32_t *sc = (const uint32_t *)(c.stepcode + ch * BG_CHUNK);
    uint32_t zeros = 0;
#pragma unroll
    for (uint32_t k = 0; k < BG_CHUNK / 4u; k++) {
        const uint32_t v = sc[k];
        /* bytes equal to zero: the classic (v - 0x01010101) & ~v & 0x80808080, exact enough for a classification */
        zeros += __popc((v - 0x01010101u) & ~v & 0x80808080u);
    }
    return zeros >= 64u ? 7u : zeros >> 3;
}

__device__ __forceinline__ void chunk_order_count(const BgCtx &c, uint32_t t, uint32_t &cls, uint32_t &rank)
{
    const uint32_t lane = t & 31u, warp = t >> 5;
    uint32_t *cnt = (uint32_t *)(c.regb + BG_B_CLASSCNT);
    cls = chunk_class(c, t);
    rank = 0;
#pragma unroll
    for (uint32_t k = 0; k < 8u; k++) {
        const unsigned m = __ballot_sync(0xffffffffu, cls == k);
        if (cls == k) rank = __popc(m & ((1u << lane) - 1u));
        if (lane == k) cnt[k * 32u + warp] = __popc(m);
    }
}

/* (warp 0) exclusive scan of the 256 counts, class-major: class k of warp w starts after all smaller classes and after class k of the warps before */
__device__ __forceinline__ void chunk_order_scan(const BgCtx &c, uint32_t t)
{
    if (t >= 32u) return;
    uint32_t *cnt = (uint32_t *)(c.regb + BG_B_CLASSCNT);
    uint32_t v[8], sum = 0;
#pragma unroll
    for (uint32_t k = 0; k < 8u; k++) { v[k] = cnt[t * 8u + k]; sum += v[k]; }
    uint32_t inc = sum;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
        if (t >= (uint32_t)d) inc += y;
    }
    uint32_t run = inc - sum;
#pragma unroll
    for (uint32_t k = 0; k < 8u; k++) { cnt[t * 8u + k] = run; run += v[k]; }
}

__device__ __forceinline__ void chunk_order_place(const BgCtx &c, uint32_t t, uint32_t cls, uint32_t rank)
{
    const uint32_t *cnt = (const uint32_t *)(c.regb + BG_B_CLASSCNT);
    BG_ASSERT(cls < 8u && cnt[cls * 32u + (t >> 5)] + rank < BG_MAX_CHUNKS);
    ((uint16_t *)(c.regb + BG_B_PERM))[cnt[cls * 32u + (t >> 5)] + rank] = (uint16_t)t;
}

/* ---- the litlen code's sort keys, ranked instead of sorted (the emulator's bg_phase_lkeys + std::sort + bg_phase_huff_prep).
 * Keys (freq << 9 | sym) are distinct, so a used symbol's place in the ascending order is the number of smaller keys: each
 * of threads 0..287 counts them over all 288 keys, 4 per broadcast load, with no block barrier in between.  Only the m used
 * keys are placed (keys[m..) are never read).  Step 1 writes every symbol's key, ~0 for an unused one, to the parent-link
 * array, which the tree merge fills only later. ---- */
#define BG_B_RANKKEYS BG_B_TREEP         /* u32[288] (16-byte aligned) */

__device__ __forceinline__ void litlen_keys(const BgCtx &c, uint32_t t)
{
    const uint32_t *lfreq = (const uint32_t *)(c.regb + BG_B_LFREQ);
    if (t < 288) {
        const uint32_t f = lfreq[t];
        ((uint32_t *)(c.regb + BG_B_RANKKEYS))[t] = f ? (f << 9) | t : 0xFFFFFFFFu;
        if (f) atomicAdd(&c.scal[BG_S_HM], 1u);
    }
}

/* step 2: place keys and leaf weights; what bg_phase_huff_prep clears; the distance alphabet's keys on the next warp */
__device__ __forceinline__ void litlen_rank(const BgCtx &c, uint32_t t)
{
    uint8_t *rb = c.regb;
    if (t < 288) {
        const uint4 *all = (const uint4 *)(rb + BG_B_RANKKEYS);
        const uint32_t k = ((const uint32_t *)all)[t];
        rb[BG_B_LLEN + t] = 0;
        if (k != 0xFFFFFFFFu) {
            uint32_t rank = 0;
#pragma unroll 8
            for (uint32_t j = 0; j < 72; j++) {
                const uint4 q = all[j];
                rank += (q.x < k) + (q.y < k) + (q.z < k) + (q.w < k);
            }
            ((uint32_t *)(rb + BG_B_KEYS))[rank] = k;
            ((uint32_t *)(rb + BG_B_TREEW))[rank] = k >> 9;
        }
    } else if (t < 288 + 30) {
        if (bg_rank_key((const uint32_t *)(rb + BG_B_DFREQ), 30, t - 288, (uint32_t *)(rb + BG_B_DKEYS))) atomicAdd(&c.scal[BG_S_DM], 1u);
    } else if (t < 288 + 32 + 16) {
        ((uint32_t *)(rb + BG_B_BLC))[t - 320] = 0;
        if (t == 320) c.scal[BG_S_HOVF] = 0;
    }
}

/* ---- a small alphabet's code lengths on one warp: bg_huff_lengths() split as for litlen (one lane merges, the warp takes
 * the depths, lane 0 repairs the overflow, the warp assigns the lengths), handed on with __syncwarp().  Same lengths: a node
 * deeper than maxbits counts as one overflow here as it does in the sequential depth pass.  keys: m ascending keys (m <= 32);
 * w, par: 2m node slots; blc: u32[16]; lens[0..nzero) is cleared first.  All 32 lanes call it. ---- */
__device__ __forceinline__ void warp_huff_lengths(const uint32_t *keys, uint32_t m, uint32_t maxbits, uint32_t nzero, uint32_t *w,
                                                  uint16_t *par, uint32_t *blc, uint8_t *lens, uint32_t lane)
{
    if (lane < nzero) lens[lane] = 0;
    if (lane < m) w[lane] = keys[lane] >> 9;
    if (lane < 16) blc[lane] = 0;
    __syncwarp();
    if (m < 2) {                                                      /* (m is the same on every lane) */
        if (lane == 0) {
            const uint32_t s = m ? keys[0] & 511u : 0u;
            lens[s] = 1;
            lens[s ? 0 : 1] = 1;
        }
        return;
    }
    if (lane == 0) bg_huff_merge(m, w, par);
    __syncwarp();
    const uint32_t root = 2 * m - 2;
    uint32_t ovf = 0;
    for (uint32_t i = lane; i < root; i += 32) {
        uint32_t d = 0;
        for (uint32_t x = i; x != root && d < 64; x = par[x]) d++;
        if (d > maxbits) { d = maxbits; ovf++; }
        if (i < m) atomicAdd(&blc[d], 1u);
    }
    int overflow = (int)__reduce_add_sync(0xffffffffu, ovf);
    __syncwarp();
    if (lane == 0) {
        while (overflow > 0) {
            uint32_t bits = maxbits - 1;
            while (bits > 1 && blc[bits] == 0) bits--;
            blc[bits]--;
            blc[bits + 1] += 2;
            blc[maxbits]--;
            overflow -= 2;
        }
    }
    __syncwarp();
    for (uint32_t i = lane; i < m; i += 32) {
        uint32_t bits = maxbits, cum = blc[maxbits];
        while (cum <= i && bits > 1) cum += blc[--bits];
        lens[keys[i] & 511u] = (uint8_t)bits;
    }
}

/* the distance code on warp 1 (the slots bg_phase_huff's thread 32 uses) */
__device__ __forceinline__ void dist_tree_warp(const BgCtx &c, uint32_t lane)
{
    uint8_t *rb = c.regb;
    warp_huff_lengths((const uint32_t *)(rb + BG_B_DKEYS), c.scal[BG_S_DM], 15, 32, (uint32_t *)(rb + BG_B_DTREEW),
                      (uint16_t *)(rb + BG_B_DTREEP), (uint32_t *)(rb + BG_B_SCRATCH) + 32, rb + BG_B_DLEN, lane);
}

/* bg_phase_hdr5 on warp 0: the precode lengths on the warp, then HCLEN by a ballot and the header bit count by a sum */
__device__ __forceinline__ void precode_hdr_warp(const BgCtx &c, uint32_t lane, uint32_t nitems)
{
    uint8_t *rb = c.regb;
    uint32_t nl, nd;
    bg_hdr_dims(c, &nl, &nd);
    const uint32_t *pfreq = (const uint32_t *)(rb + BG_B_PFREQ);
    uint8_t *plen = rb + BG_B_PLEN;
    warp_huff_lengths((const uint32_t *)(rb + BG_B_PKEYS), c.scal[BG_S_PM], 7, 19, (uint32_t *)(rb + BG_B_DTREEW),
                      (uint16_t *)(rb + BG_B_DTREEP), (uint32_t *)(rb + BG_B_SCRATCH) + 16, plen, lane);
    __syncwarp();
    const unsigned used = __ballot_sync(0xffffffffu, lane < 19 && plen[bg_precode_order(lane)] != 0);
    uint32_t np = used ? 32u - (uint32_t)__clz(used) : 0u;            /* one past the last length HCLEN must carry, at least 4 */
    if (np < 4) np = 4;
    const uint32_t bits = lane < 19 ? pfreq[lane] * (plen[lane] + (lane == 16 ? 2u : lane == 17 ? 3u : lane == 18 ? 7u : 0u)) : 0u;
    const uint32_t hdr = 3 + 5 + 5 + 4 + 3 * np + __reduce_add_sync(0xffffffffu, bits);
    if (lane == 0) {
        c.scal[BG_S_DYNHDR] = hdr;
        c.scal[BG_S_NITEMS] = nitems;
        c.scal[BG_S_NL] = nl;
        c.scal[BG_S_ND] = nd;
        c.scal[BG_S_NP] = np;
    }
}

/* ---- named barrier of the tree warps (warps 0 .. BG_TREE_WARPS-1): the other warps run the CRC slices meanwhile ---- */
#define BG_TREE_WARPS 4u
__device__ __forceinline__ void tree_bar()
{
    asm volatile("bar.sync 1, %0;" :: "n"(BG_TREE_WARPS * 32) : "memory");
}

/* ---- exclusive prefix sum over 1024 u32 in shared memory; returns the grand total ---- */
__device__ __forceinline__ uint32_t block_exclusive_scan_1024(uint32_t *v, uint32_t *scratch, uint32_t t)
{
    const uint32_t lane = t & 31u, warp = t >> 5;
    uint32_t x = v[t], inc = x;
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += y;
    }
    if (lane == 31) scratch[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = scratch[lane], winc = w;
        for (int d = 1; d < 32; d <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, winc, d);
            if (lane >= (uint32_t)d) winc += y;
        }
        scratch[lane] = winc - w;
        if (lane == 31) scratch[32] = winc;
    }
    __syncthreads();
    v[t] = scratch[warp] + inc - x;
    uint32_t total = scratch[32];
    __syncthreads();
    return total;
}

/* one member, slot -> its place in the stream, by `nthr` threads (thread `t` of them); the destination may start at any byte */
__device__ __forceinline__ void gather_member(const uint32_t *src, uint32_t n, uint8_t *dst, uint32_t t, uint32_t nthr)
{
    const uint32_t head = (uint32_t)((4u - ((uintptr_t)dst & 3u)) & 3u);   /* bytes until dst is word aligned */
    if (n <= head + 4) {
        for (uint32_t i = t; i < n; i += nthr) dst[i] = (uint8_t)(__ldcg(src + (i >> 2)) >> (8u * (i & 3u)));
        return;
    }
    if (t < head) dst[t] = (uint8_t)(__ldcg(src) >> (8u * t));
    const uint32_t words = (n - head) >> 2;
    uint32_t *dw = (uint32_t *)(dst + head);
    const uint32_t sh = head * 8u;
    for (uint32_t i = t; i < words; i += nthr)
        dw[i] = __funnelshift_r(__ldcg(src + i), __ldcg(src + i + 1), sh);   /* src word i+1 stays inside the 64 KiB slot + pad */
    const uint32_t done = head + words * 4u;
    if (t < n - done) dst[done + t] = (uint8_t)(__ldcg(src + ((done + t) >> 2)) >> (8u * ((done + t) & 3u)));
}

__device__ __forceinline__ uint32_t block_exclusive_scan_1024(uint32_t *v, uint32_t *scratch, uint32_t t);

/* the last CTA of a launch: member sizes -> offsets (tiles of 1024, running carry), then every member to its place */
__device__ __forceinline__ void fused_compaction(const BgzfCompressArgs &a, uint32_t *v, uint32_t *scratch, uint32_t t)
{
    uint64_t carry = *a.gather_total;
    for (uint32_t start = 0; start < a.nblocks; start += 1024u) {
        const uint32_t i = start + t;
        v[t] = i < a.nblocks ? __ldcg(a.out_len + i) : 0u;
        __syncthreads();
        const uint32_t total = block_exclusive_scan_1024(v, scratch, t);
        if (i < a.nblocks) a.gather_off[i] = carry + v[t];
        carry += total;
        __syncthreads();
    }
    if (t == 0) *a.gather_total = carry;
    __syncthreads();
    const uint32_t grp = t >> 8, gt = t & 255u;
    for (uint32_t b = grp; b < a.nblocks; b += BG_THREADS / 256u) {
        BG_ASSERT(__ldcg(a.out_len + b) <= BG_SLOT_BYTES && a.gather_off[b] + __ldcg(a.out_len + b) <= carry);
        gather_member((const uint32_t *)(a.slots + (size_t)b * BG_SLOT_BYTES), __ldcg(a.out_len + b), a.gather_out + a.gather_off[b], gt, 256u);
    }
}

#define PROF_MARK(i)                                                        \
    do {                                                                    \
        if (prof && t == 0) {                                               \
            long long now_ = clock64();                                     \
            atomicAdd((unsigned long long *)&prof[i], (unsigned long long)(now_ - tprev_)); \
            tprev_ = now_;                                                  \
        }                                                                   \
    } while (0)

/* SPLIT = false: the persistent kernel, CTA i takes blocks i, i + grid, ...
 * SPLIT = true : one block, one cluster (the hook's one-member calls, where latency is everything).  Every CTA of the
 *                cluster stages the payload and hashes it (same inputs, same code: same tables); the equal-hash peers
 *                are found for every size-th tile by each CTA and exchanged through L2, the chains are linked by
 *                everyone, then each CTA searches every size-th tile of positions into the first CTA's match scratch;
 *                after the second cluster barrier the first CTA carries on alone.  The search is half the time of a
 *                block, so a cluster of 4 cuts the latency of a member by about 45 % at the price of three SMs doing
 *                redundant set-up work. */
template <bool SPLIT>
__device__ __forceinline__ void compress_blocks(BgzfCompressArgs &a)
{
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t t = threadIdx.x, T = BG_THREADS;
    uint64_t *mbar = (uint64_t *)(smem + SM_MBAR);
    uint32_t *scan_scratch = (uint32_t *)(smem + SM_SCAN);
    unsigned long long *prof = a.prof;
    long long tprev_ = prof ? clock64() : 0;
    uint32_t *const pscr = scan_scratch;                  /* profiling only: last producer, slowest / fastest pass-1 warp */

    BgCtx c;
    c.dataw = (uint32_t *)(smem + SM_DATA);
    c.prev = (uint16_t *)(smem + SM_REGA);
    c.stepcode = smem + SM_REGA;
    c.jump8 = smem + SM_REGA + 65536u;
    c.offarr = (uint16_t *)(smem + SM_REGA + 65536u);
    c.head = (uint16_t *)(smem + SM_REGB);
    c.regb = smem + SM_REGB;
    c.crctab = (uint32_t *)(smem + SM_CRCTAB);
    c.litflag = smem + SM_LITFLAG;
    c.scal = (uint32_t *)(smem + SM_SCAL);
    const uint32_t crank = SPLIT ? cluster_rank() : 0u, csize = SPLIT ? cluster_size() : 1u;
    const uint32_t unit = SPLIT ? blockIdx.x / csize : blockIdx.x;       /* SPLIT: cluster k of the grid takes block k */
    uint32_t *const unit_scratch = a.scratch + (size_t)unit * (SPLIT ? BGZF_SCRATCH_WORDS + BGZF_SPLIT_EXTRA_WORDS : BGZF_SCRATCH_WORDS);
    c.R = unit_scratch;
    c.cand = a.cand ? a.cand + (size_t)unit * (4u * BG_MAX_BLOCK) : nullptr;
    c.crcpow = a.crcpow;
    c.prm = a.prm;
    c.frame = bg_frame(a.hdr_bytes ? a.hdr_bytes : 18u, 8u, 1u, 0u);
    c.perm = (const uint16_t *)(smem + SM_REGB + BG_B_PERM);

    if (t < 256) c.crctab[t] = a.crctab[t];
    if (t == 0) {
        mbar_init(mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t parity = 0;

    for (uint32_t b = unit; b < a.nblocks; b += SPLIT ? a.nblocks : gridDim.x) {
        const uint8_t *src;
        uint32_t n;
        if (a.in_off) {
            src = a.in + a.in_off[b];
            n = a.in_len[b];
        } else {
            const uint64_t off = (uint64_t)b * a.block_size;
            src = a.in + off;
            const uint64_t rem = a.in_bytes - off;
            n = rem < a.block_size ? (uint32_t)rem : a.block_size;
        }
        c.out = (uint32_t *)(a.slots + (size_t)b * BG_SLOT_BYTES);
        if (a.piece_mode) {
            /* piece b of the call is piece gb of the stream: members are runs of member_blocks pieces (the last one may be short) */
            const uint64_t gb = a.piece_base + b;
            const bool first = gb % a.member_blocks == 0, last = (gb + 1) % a.member_blocks == 0 || gb + 1 == a.piece_total;
            /* dictionary priming: what precedes the piece in its member, as far as the window reaches */
            uint32_t hist = 0;
            if (a.history && !first && !a.in_off) {
                const uint64_t in_member = (gb % a.member_blocks) * a.block_size, in_buffer = (uint64_t)a.lead + (uint64_t)b * a.block_size;
                uint64_t h = in_member < in_buffer ? in_member : in_buffer;
                if (h > a.history) h = a.history;
                hist = (uint32_t)h - (uint32_t)h % BG_HISTORY_STEP;
            }
            src -= hist;
            n += hist;
            c.frame = bg_frame(first ? a.head_gap : 0u, last ? a.tail_gap : 0u, last && !a.no_final ? 1u : 0u, 1u, hist);
        }
        c.n = n;

        /* 1. stage the payload: TMA for the 16-byte-aligned bulk, plain loads for the ragged rest */
        const bool aligned = (((uintptr_t)src) & 15u) == 0;
        const uint32_t bulk = aligned ? (n & ~15u) : 0u;
        if (bulk) {
            if (t == 0) {
                fence_proxy_async();
                mbar_expect_tx(mbar, bulk);
                tma_load_1d(smem + SM_DATA, src, bulk, mbar);
            }
        }
        for (uint32_t i = bulk + t; i < n; i += T)
            smem[SM_DATA + i] = src[i];
        bg_phase_init(c, t, T);
        if (bulk) {
            mbar_wait(mbar, parity);
            parity ^= 1u;
        }
        __syncthreads();
        PROF_MARK(0);

        /* the literal census steers the search; the CRC is needed only by the trailer and runs on the warps the Huffman
         * trees leave idle (below) */
        bg_phase_census(c, t, T);
        __syncthreads();
        bg_phase_count(c, t, T);
        __syncthreads();
        bg_phase_settle_census(c, t, T);
        __syncthreads();
        PROF_MARK(1);
        PROF_MARK(2);
        uint4 *hi = (uint4 *)(c.R + BG_MAX_BLOCK + 32);       /* build commands live behind the match scratch */
        if (SPLIT) {
            /* every CTA has the same hashes; each finds the peers of its share of the tiles, the links travel through L2 */
            uint4 *xprev = (uint4 *)(unit_scratch + BGZF_SCRATCH_WORDS);
            build_peers_phase(c, hi, t & 31u, t >> 5, BG_THREADS / 32u, crank, csize, xprev, nullptr, nullptr, 0);
            cluster_sync();
            import_peer_tiles(c, xprev, t, crank, csize);
            __syncthreads();
            PROF_MARK(3);
            if (t < 32u * BG_LINKERS) build_link_phase(c, hi, t >> 5, t & 31u, &c.scal[BG_S_WLIST], nullptr, nullptr, 0);   /* the other warps wait at the barrier */
        } else {
            /* peers and links at the same time: warps 0..3 are the linking relay, the other 28 find the peers tile by tile
             * and raise a flag per tile; the relay's ordered head-table section hides behind the ballots of the producers */
            volatile uint8_t *ready = (volatile uint8_t *)(smem + SM_READY);
            if (t < 128u) ready[t] = 0;
            if (prof && t == 0) { pscr[0] = 0; pscr[1] = 0; pscr[2] = 0xffffffffu; }
            __syncthreads();
            const long long t0 = prof ? clock64() : 0;
            if (t < 32u * BG_LINKERS) {
                build_link_phase(c, hi, t >> 5, t & 31u, &c.scal[BG_S_WLIST], ready, prof, t0);
            } else {
                build_peers_phase(c, hi, t & 31u, (t >> 5) - BG_LINKERS, BG_THREADS / 32u - BG_LINKERS, 0u, 1u, nullptr, ready, prof, t0);
                if (prof && (t & 31u) == 0) atomicMax(&pscr[0], (uint32_t)(clock64() - t0));
            }
        }
        __syncthreads();
        PROF_MARK(10);
        {
            bg_phase_search_clear(c, t, T);
            if (SPLIT) cluster_sync();                           /* every CTA's bitmap is clear before anyone's marks arrive */
            else __syncthreads();
            const long long t1 = prof ? clock64() : 0;
            search_nearest<SPLIT>(c, t, crank, csize);
            if (!SPLIT && prof && (t & 31u) == 0) {              /* pass 1: when the slowest and the fastest warp finish */
                const uint32_t d = (uint32_t)(clock64() - t1);
                atomicMax(&pscr[1], d);
                atomicMin(&pscr[2], d);
            }
            if (SPLIT) cluster_sync();                           /* ... and complete before it is read */
            else __syncthreads();
            if (!SPLIT && prof && t == 0) {
                atomicAdd(&prof[22], (unsigned long long)pscr[0]);
                atomicAdd(&prof[26], (unsigned long long)pscr[1]);
                atomicAdd(&prof[27], (unsigned long long)pscr[2]);
            }
            PROF_MARK(21);
            if (c.scal[BG_S_DEPTH] > 1) {                        /* (uniform for the CTA) */
                bg_phase_search_todo(c, t, T, crank, csize);
                __syncthreads();
                /* shallow chains (levels 2-7): 32 positions side by side; deep ones: lanes refill themselves */
                const bool h3 = c.scal[BG_S_HBYTES] == 3;        /* (uniform) the 3-byte-window variants carry the free-node rule */
                if (c.scal[BG_S_DEPTH] <= 24u) {
                    if (h3) search_deep_batches<true>(c, t, crank, csize);
                    else search_deep_batches<false>(c, t, crank, csize);
                } else {
                    if (h3) search_deep<true>(c, t, crank, csize);
                    else search_deep<false>(c, t, crank, csize);
                }
            }
        }
        if (SPLIT) {
            cluster_sync();
            if (crank) return;
        }
        __syncthreads();
        PROF_MARK(4);
        for (int pass = 0; pass <= c.prm.opt_passes; pass++) {
            if (pass == 0) {
                bg_phase_accept(c, t, T);
            } else {
                bg_phase_costs(c, t, T);
                __syncthreads();
                dp_segment_warp(c, t >> 5, t & 31u, (uint32_t *)(smem + SM_REGA + 65536u) + (t >> 5) * BG_DP_RING);
            }
            __syncthreads();
            if (bg_f_hist(c)) {                                  /* (uniform) */
                bg_phase_history_steps(c, t, T);
                __syncthreads();
            }
            PROF_MARK(15);
            bg_phase_jump(c, t, T);
            __syncthreads();
            PROF_MARK(5);
            bg_phase_walk_clear(c, t, T);
            bg_phase_clear_freq(c, t, T);
            __syncthreads();
            bg_phase_walk_mark(c, t, T);
            __syncthreads();
            bg_phase_walk_list(c, t, T);
            __syncthreads();
            PROF_MARK(16);
            bg_phase_walk_a(c, t, T);
            __syncthreads();
            PROF_MARK(17);
            bg_phase_walk_b(c, t, T);
            uint32_t ccls, crnk;
            chunk_order_count(c, t, ccls, crnk);             /* (the step codes are final; the counts go where the walk list was) */
            __syncthreads();
            PROF_MARK(18);
            bg_phase_walk_c(c, t, T);
            chunk_order_scan(c, t);
            __syncthreads();
            chunk_order_place(c, t, ccls, crnk);
            __syncthreads();
            PROF_MARK(6);
            bg_phase_tally(c, t, T);
            __syncthreads();
            PROF_MARK(7);
            litlen_keys(c, t);
            if (prof && t == 0) { pscr[3] = 0; pscr[4] = 0; }
            __syncthreads();
            litlen_rank(c, t);
            __syncthreads();
            PROF_MARK(11);
            /* the trees on warps 0..3 (thread 0 merges the litlen tree, thread 32 builds the distance code), the CRC slices
             * on the other 28 warps, once per block; everyone meets at the barrier after the trees */
            const long long t2 = prof ? clock64() : 0;
            if (t < 32u * BG_TREE_WARPS) {
                const uint32_t TT = 32u * BG_TREE_WARPS;
                if (t < 32u) bg_phase_huff(c, t, TT);                /* (thread 0: the litlen merge) */
                else if (t < 64u) dist_tree_warp(c, t - 32u);
                tree_bar();
                bg_phase_huff_depth(c, t, TT);
                tree_bar();
                bg_phase_huff_fix(c, t, TT);
                tree_bar();
                bg_phase_huff_assign(c, t, TT);
                if (prof && pass == 0 && (t & 31u) == 0) atomicMax(&pscr[3], (uint32_t)(clock64() - t2));
            } else if (pass == 0) {
                bg_crc_slices(c, t - 32u * BG_TREE_WARPS, T - 32u * BG_TREE_WARPS);
                if (prof && (t & 31u) == 0) atomicMax(&pscr[4], (uint32_t)(clock64() - t2));
            }
            __syncthreads();
            if (prof && pass == 0 && t == 0 && pscr[4] > pscr[3]) atomicAdd(&prof[28], (unsigned long long)(pscr[4] - pscr[3]));
            PROF_MARK(12);
        }
        if (t == 0) bg_crc_finish(c);                            /* (every slice is in; the trailer is written by the emit) */
        bg_phase_hdr1(c, t, T);
        __syncthreads();
        bg_phase_hdr2(c, t, T);
        __syncthreads();
        bg_phase_hdr3(c, t, T);
        __syncthreads();
        const uint32_t nitems = block_exclusive_scan_1024((uint32_t *)(c.regb + BG_B_CBITS), scan_scratch, t);
        bg_phase_hdr4(c, t, T);
        __syncthreads();
        if (t < 32u) {                                           /* the precode keys and lengths are warp 0's work */
            bg_phase_hdr4b(c, t, 32u);
            __syncwarp();
            precode_hdr_warp(c, t, nitems);
        }
        __syncthreads();
        PROF_MARK(13);
        bg_phase_decide_b(c, t, T);
        __syncthreads();
        bg_phase_codes_a(c, t, T);
        __syncthreads();
        bg_phase_codes_b(c, t, T);
        __syncthreads();
        bg_phase_codes_c(c, t, T);
        __syncthreads();
        bg_phase_tabs(c, t, T);
        __syncthreads();
        PROF_MARK(8);
        bg_phase_hdr_bits(c, t, T);
        bg_phase_sizes(c, t, T);
        __syncthreads();
        PROF_MARK(19);
        block_exclusive_scan_1024((uint32_t *)(c.regb + BG_B_CBITS), scan_scratch, t);
        block_exclusive_scan_1024((uint32_t *)(c.regb + BG_B_IOFF), scan_scratch, t);
        PROF_MARK(20);
        bg_phase_zero_out(c, t, T);
        __syncthreads();
        PROF_MARK(14);
        bg_phase_emit(c, t, T);
        if (t == 0) {
            const uint32_t st = c.scal[BG_S_STATUS];
            a.out_len[b] = st ? 0u : bg_f_hdr(c) + c.scal[BG_S_PAYLOAD] + bg_f_trl(c);
            if (a.crc_out) a.crc_out[b] = c.scal[BG_S_CRC];
            a.status[b] = st;
            if (st) atomicOr(a.err_flag, 1u);
        }
        fence_proxy_async();   /* our generic-proxy accesses to the payload area precede the next TMA write */
        __syncthreads();       /* everyone is done with the payload and the tables before the next block lands */
        PROF_MARK(9);
    }
    if (!SPLIT && a.gather_out) {
        /* whoever finishes last compacts the batch (threadFenceReduction pattern: every CTA's members are out before it counts itself) */
        __threadfence();
        __syncthreads();
        if (t == 0) scan_scratch[35] = atomicAdd(a.done_count, 1u) == gridDim.x - 1u ? 1u : 0u;
        __syncthreads();
        if (scan_scratch[35]) {
            __threadfence();
            fused_compaction(a, (uint32_t *)(smem + SM_REGB), scan_scratch, t);
        }
    }
}

__global__ void __launch_bounds__(BG_THREADS, 1)
bgzf_compress_kernel(BgzfCompressArgs a)
{
    compress_blocks<false>(a);
}

__global__ void __launch_bounds__(BG_THREADS, 1)
bgzf_compress_split_kernel(BgzfCompressArgs a)
{
    compress_blocks<true>(a);
}

/* ---- sizes -> exclusive offsets (single CTA, tiles of 1024 with a running carry).
 * count_dev (optional) overrides the element count, base_dev (optional) seeds the carry: both live on the
 * device so that batches chain without a host round trip. ---- */
__global__ void __launch_bounds__(1024, 1)
bgzf_scan_kernel(const uint32_t *len, uint64_t *off, uint32_t nmax, const uint64_t *count_dev, const uint64_t *base_dev,
                 uint64_t *total_out)
{
    __shared__ uint32_t v[1024];
    __shared__ uint32_t scratch[36];
    const uint32_t t = threadIdx.x;
    uint32_t n = nmax;
    if (count_dev) { const uint64_t cd = *count_dev; n = cd < nmax ? (uint32_t)cd : nmax; }
    uint64_t carry = base_dev ? *base_dev : 0ull;
    __syncthreads();   /* total_out may alias base_dev: everyone has read it before anyone writes */
    for (uint32_t start = 0; start < n; start += 1024) {
        const uint32_t i = start + t;
        v[t] = i < n ? len[i] : 0u;
        __syncthreads();
        const uint32_t total = block_exclusive_scan_1024(v, scratch, t);
        if (i < n) off[i] = carry + v[t];
        carry += total;
        __syncthreads();
    }
    if (t == 0) *total_out = carry;
}

/* ---- slots -> contiguous stream.  One CTA per member; destination may start at any byte. ---- */
__global__ void __launch_bounds__(256)
bgzf_gather_kernel(const uint8_t *slots, const uint32_t *len, const uint64_t *off, uint32_t nblocks, uint8_t *out,
                   const uint64_t *total, int append_eof)
{
    const uint32_t b = blockIdx.x, t = threadIdx.x;
    if (b == nblocks) {
        if (append_eof && t < 28) {
            const uint8_t eof[28] = { 0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0,
                                      0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
            out[*total + t] = eof[t];
        }
        return;
    }
    const uint32_t n = len[b];
    const uint32_t *src = (const uint32_t *)(slots + (size_t)b * BG_SLOT_BYTES);
    uint8_t *dst = out + off[b];
    const uint32_t head = (uint32_t)((4u - ((uintptr_t)dst & 3u)) & 3u);   /* bytes until dst is word aligned */
    if (n <= head + 4) {
        for (uint32_t i = t; i < n; i += blockDim.x) dst[i] = ((const uint8_t *)src)[i];
        return;
    }
    if (t < head) dst[t] = ((const uint8_t *)src)[t];
    const uint32_t words = (n - head) >> 2;
    uint32_t *dw = (uint32_t *)(dst + head);
    const uint32_t sh = head * 8u;
    for (uint32_t i = t; i < words; i += blockDim.x)
        dw[i] = __funnelshift_r(src[i], src[i + 1], sh);       /* src word i+1 stays inside the 64 KiB slot + pad */
    const uint32_t done = head + words * 4u;
    if (t < n - done) dst[done + t] = ((const uint8_t *)src)[done + t];
}

/* ---- the hook combiner's way back: member b of a batch goes from its device slot to the caller's own pinned host buffer
 * (16-byte header: the member size, 0 = did not fit; then the member).  Zero-copy stores over PCIe, 16 bytes per thread:
 * only the member's bytes travel, and no copy call is needed per member. ---- */
__global__ void __launch_bounds__(256)
bgzf_deliver_kernel(const uint8_t *slots, const uint32_t *len, const uint64_t *out_off, uint8_t *host_out, uint32_t n)
{
    const uint32_t b = blockIdx.x, t = threadIdx.x;
    if (b >= n) return;
    const uint32_t nbytes = len[b];
    const uint4 *src = (const uint4 *)(slots + (size_t)b * BG_SLOT_BYTES);
    uint4 *dst = (uint4 *)(host_out + out_off[b]);
    for (uint32_t i = t; i < (nbytes + 15u) / 16u; i += blockDim.x) dst[1u + i] = src[i];
    if (t == 0) dst[0] = make_uint4(nbytes, 0u, 0u, 0u);
}

extern "C" cudaError_t bgzf_launch_deliver(const uint8_t *slots, const uint32_t *len, const uint64_t *out_off, uint8_t *host_out, uint32_t n,
                                           cudaStream_t stream)
{
    bgzf_deliver_kernel<<<n, 256, 0, stream>>>(slots, len, out_off, host_out, n);
    return cudaGetLastError();
}

extern "C" cudaError_t bgzf_launch_compress(const BgzfCompressArgs *a, int grid, cudaStream_t stream)
{
    /* (per device, once: the hook launches this kernel from many threads at a high rate) */
    static std::atomic<unsigned long long> configured{0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!((configured.load() >> dev) & 1ull)) {
        cudaError_t e = cudaFuncSetAttribute(bgzf_compress_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_TOTAL);
        if (e != cudaSuccess) return e;
        configured.fetch_or(1ull << dev);
    }
    bgzf_compress_kernel<<<grid, BG_THREADS, SM_TOTAL, stream>>>(*a);
    return cudaGetLastError();
}

/* a->nblocks blocks, each on its own cluster of `csize` CTAs; a->scratch holds BGZF_SCRATCH_WORDS +
 * BGZF_SPLIT_EXTRA_WORDS words per block (a->cand, if any, 4 * 65536 words per block) */
extern "C" cudaError_t bgzf_launch_compress_split(const BgzfCompressArgs *a, int csize, cudaStream_t stream)
{
    static std::atomic<unsigned long long> configured{0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!((configured.load() >> dev) & 1ull)) {
        cudaError_t e = cudaFuncSetAttribute(bgzf_compress_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM_TOTAL);
        if (e != cudaSuccess) return e;
        configured.fetch_or(1ull << dev);
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3((unsigned)csize * a->nblocks);
    cfg.blockDim = dim3(BG_THREADS);
    cfg.dynamicSmemBytes = SM_TOTAL;
    cfg.stream = stream;
    cudaLaunchAttribute at;
    memset(&at, 0, sizeof at);
    at.id = cudaLaunchAttributeClusterDimension;
    at.val.clusterDim.x = (unsigned)csize;
    at.val.clusterDim.y = 1;
    at.val.clusterDim.z = 1;
    cfg.attrs = &at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, bgzf_compress_split_kernel, *a);
}

extern "C" cudaError_t bgzf_launch_scan(const uint32_t *len, uint64_t *off, uint32_t nmax, const uint64_t *count_dev,
                                        const uint64_t *base_dev, uint64_t *total_out, cudaStream_t stream)
{
    bgzf_scan_kernel<<<1, 1024, 0, stream>>>(len, off, nmax, count_dev, base_dev, total_out);
    return cudaGetLastError();
}

/* total (device) is read as the running base and updated to the new end of the stream */
extern "C" cudaError_t bgzf_launch_compact(const uint8_t *slots, const uint32_t *len, uint64_t *off, uint32_t nblocks,
                                           uint8_t *out, uint64_t *total, int append_eof, cudaStream_t stream)
{
    bgzf_scan_kernel<<<1, 1024, 0, stream>>>(len, off, nblocks, nullptr, total, total);
    bgzf_gather_kernel<<<nblocks + 1, 256, 0, stream>>>(slots, len, off, nblocks, out, total, append_eof);
    return cudaGetLastError();
}
