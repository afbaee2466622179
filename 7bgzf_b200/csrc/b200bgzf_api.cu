/*
 * b200bgzf_api.cu — the C-ABI shim over the sm_100a kernels (see include/b200bgzf.h).
 *
 * Owns, per context: the device tables, a few "lanes" (stream + pinned staging + device workspaces) that the
 * host-buffer paths rotate through so H2D copies, kernels and D2H copies of consecutive batches overlap, and a
 * pool of one-block lanes for the LD_PRELOAD hook so concurrent htslib threads each drive their own SM.
 * No CPU fallback anywhere: a failing CUDA call surfaces as B200BGZF_E_CUDA.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <linux/futex.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <map>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/b200bgzf.h"
#include "bgzf_block.h"
#include "bgzf_gzip_route.h"
#include "bgzf_kernels.h"
#include "bgzf_tables.h"

namespace {

constexpr uint32_t kHostBatchBlocks = 512;      /* 32 MiB of payload per pipelined batch: best of 296 ... 4096 (all within 7 %) */
constexpr uint32_t kDeviceBatchBlocks = 16384;  /* 1 GiB of payload per device-resident batch */
constexpr int kLanes = 8;        /* lanes a host-buffer call may rotate through (it uses the first few) */
constexpr size_t kInflateBatch = 1536;  /* members per pipelined inflate batch (measured: 512 is 15 % slower, 1024-2048 within 3 %) */
constexpr int kInflateLanes = 8;        /* 8 x 1536 members in flight keep the GPU (~4700 resident members) and the D2H engine busy */
constexpr int kHookLanes = 128;
constexpr uint32_t kHookLaneBlocks = 4;

struct Lane {
    cudaStream_t stream = nullptr;
    uint32_t cap_blocks = 0;
    size_t in_cap = 0, out_cap = 0, host_in_cap = 0, host_out_cap = 0, meta_cap = 0;
    uint8_t *d_in = nullptr, *d_slots = nullptr, *d_out = nullptr;
    uint32_t *d_len = nullptr, *d_status = nullptr, *d_scratch = nullptr, *d_cand = nullptr;
    uint64_t *d_off = nullptr, *d_inoff = nullptr, *d_outoff = nullptr;
    uint32_t *d_inlen = nullptr;
    uint64_t *d_total = nullptr;   /* [0] running stream size, [1] error flags, [2..3] spare */
    uint64_t *h_total = nullptr;   /* pinned mirror */
    uint8_t *h_in = nullptr, *h_out = nullptr;   /* pinned staging (hook / block-list paths) */
    uint64_t *h_meta = nullptr;                  /* pinned: offsets / lengths */
    /* bookkeeping of an in-flight host batch */
    bool pending = false;
    size_t pend_out_off = 0;
    uint64_t pend_first = 0;      /* first block and block count of the batch in flight (member offsets) */
    uint32_t pend_nb = 0;
    bool busy = false;
    int scratch_ctas = 0;
    int cand_ctas = 0;            /* CTAs d_cand is sized for (near-optimal levels) */
    cudaEvent_t done = nullptr;   /* hook lanes: the context's completion thread polls it when callers outnumber the host's cores */
    std::atomic<uint32_t> wait_state{0};   /* 0 idle, 1 in flight (the caller sleeps on this word), 2 done */
    cudaError_t wait_result = cudaSuccess;
    volatile uint32_t *h_flag = nullptr;   /* pinned: set by a 4-byte copy queued behind the member's copy (no driver call needed to see it) */
    uint32_t *d_one = nullptr;             /* device word holding 1: the source of that copy */
    uint8_t *one_dev = nullptr, *one_host = nullptr;   /* one-block fast path: everything it needs in one device and one pinned slab */
    uint8_t *d_rdec = nullptr;                  /* range reads: decoded members of a group, then the group's output */
    uint64_t *d_rmeta = nullptr;                /* range reads: the group's gather lists */
    size_t rdec_cap = 0, rmeta_cap = 0;
};

/* ---- the hook's combiner: many synchronous one-block callers, ONE submitter --------------------------------------
 * With more callers than host cores, every caller issuing its own copies and launch serialises on the driver's context
 * lock (measured: 64 callers -> 1.2-1.5 ms per call, 3 GB/s).  Here a caller only copies its payload into its pinned
 * slot, marks it ready and sleeps on the slot's futex word; the context's dispatcher thread gathers the ready slots into
 * a batch — one kernel launch over all of them (the kernel reads the payloads straight from the pinned slots), one copy of
 * the members back, one flag — and wakes each caller when its member is in host memory.  Four driver calls per BATCH. */
constexpr int kCombSlots = 256;
constexpr int kCombBatches = 8;
constexpr int kCombBatchMax = 64;
constexpr size_t kCombInStride = BG_SLOT_BYTES + 64;
constexpr size_t kCombOutStride = BG_SLOT_BYTES + 64;   /* 16-byte header (member size) + the member */

struct CombSlot {
    std::atomic<uint32_t> state{0};     /* 0 free, 1 being filled, 2 ready, 3 in flight, 4 done (the caller sleeps while it is 2 or 3) */
    uint32_t slen = 0, out_len = 0;
    int level = 0, rc = 0;
    int child[4] = { -1, -1, -1, -1 };   /* slots this caller wakes once it is awake itself (the wake-up fans out as a tree) */
};
struct CombBatch {
    cudaStream_t stream = nullptr;
    uint8_t *d_slots = nullptr;
    uint32_t *d_meta = nullptr, *h_meta = nullptr;      /* [0..M) member sizes, [M..2M) status, [2M] error flag, [2M+1] the constant 1 */
    uint64_t *h_inoff = nullptr, *h_outoff = nullptr;   /* pinned, read by the kernels in place */
    uint32_t *h_inlen = nullptr;
    uint32_t *d_scratch = nullptr, *d_cand = nullptr;
    volatile uint32_t *h_flag = nullptr;
    int n = 0, slots[kCombBatchMax];
    bool inflight = false;
};
struct Combiner {
    bool up = false, failed = false;
    uint8_t *h_in = nullptr, *h_out = nullptr;          /* pinned arenas: every caller slot's payload, and where its member comes back */
    CombSlot slots[kCombSlots];
    CombBatch batches[kCombBatches];
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::atomic<int> pending{0};                        /* slots in state 2 or 3 */
    std::atomic<bool> stop{false}, sleeping{false};
};

/* whole-stream gzip: device workspaces of b200bgzf_gzip_inflate_device and the GZIP container reader (grown on demand) */
struct GzWork {
    uint32_t *tile_count = nullptr, *u32 = nullptr, *small32 = nullptr;
    uint64_t *tile_off = nullptr, *u64 = nullptr, *small64 = nullptr, *h = nullptr;
    uint16_t *scratch = nullptr;
    uint8_t *d_in = nullptr, *d_out = nullptr;
    size_t tiles_cap = 0, tileoff_cap = 0, u32_cap = 0, u64_cap = 0, scratch_cap = 0, in_cap = 0, out_cap = 0, h_cap = 0;
    cudaStream_t copy = nullptr;      /* D2H of finished batches (host reader), behind the batch's event */
    cudaEvent_t ev = nullptr;
    /* random access through a checkpoint index: windows, the u8 image of a batch's layout, the window carried over a cut run,
     * per-batch chunk / window / gather lists */
    uint8_t *d_win = nullptr, *d_img = nullptr, *d_rout = nullptr;
    uint16_t *d_carry = nullptr;
    uint64_t *d_meta = nullptr;
    size_t win_cap = 0, img_cap = 0, rout_cap = 0, carry_cap = 0, meta_cap = 0;
};

}  // namespace

struct b200bgzf_ctx {
    int device = 0;
    int sms = 0;
    uint32_t *d_crctab = nullptr, *d_crcpow = nullptr;
    unsigned long long *d_prof = nullptr;
    bool prof_on = false;
    std::mutex mu;                 /* serialises the bulk APIs */
    Lane lanes[kLanes];
    std::mutex hook_mu;
    std::condition_variable hook_cv;
    Lane hook_lanes[kHookLanes];
    /* device-resident inflate index workspaces */
    uint64_t *d_idx_inoff = nullptr, *d_idx_outoff = nullptr, *d_idx_tileoff = nullptr, *d_idx_counts = nullptr;
    uint64_t *d_idx_cand = nullptr, *d_idx_pick = nullptr;
    uint32_t *d_idx_tilecount = nullptr, *d_idx_isize = nullptr, *d_idx_status = nullptr, *d_inf_status = nullptr;
    uint32_t *d_idx_jump = nullptr, *d_idx_jump2 = nullptr, *d_idx_reach = nullptr;
    size_t idx_cap = 0, idx_tiles = 0;
    uint64_t *h_idx = nullptr;
    /* device-resident range reads: per-member and per-range workspaces, the scratch of decoded members, pinned staging */
    uint64_t *d_rng_mem = nullptr, *d_rng_rw = nullptr, *d_rng_counts = nullptr, *h_rng = nullptr, *h_rng_soff = nullptr;
    uint8_t *d_rng_scratch = nullptr;
    size_t rng_mem_cap = 0, rng_rw_cap = 0, rng_scratch_cap = 0, h_rng_cap = 0, h_rng_soff_cap = 0;
    GzWork gz;
    /* Completion thread (hook callers beyond the host's core count): callers neither spin nor poll, they sleep on their
     * lane's futex word; this one thread polls the events of the lanes in flight and wakes each caller as its member is back */
    std::thread waiter;
    std::mutex waiter_mu;
    std::condition_variable waiter_cv;
    std::atomic<int> waiter_inflight{0};
    std::atomic<bool> waiter_stop{false};
    bool waiter_started = false;
    Combiner comb;
    std::atomic<int> one_block_callers{0};         /* threads inside a one-block call right now */
    std::atomic<unsigned long long> launches{0};   /* hook callers bump it concurrently */
    std::atomic<bool> no_clusters{false};          /* set when a cluster launch was refused once */
    char err[256] = { 0 };
};

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

void futex_wait_while(std::atomic<uint32_t> *word, uint32_t value)
{
    while (word->load(std::memory_order_acquire) == value)
        syscall(SYS_futex, (uint32_t *)word, FUTEX_WAIT_PRIVATE, value, nullptr, nullptr, 0);
}
void futex_wake_one(std::atomic<uint32_t> *word) { syscall(SYS_futex, (uint32_t *)word, FUTEX_WAKE_PRIVATE, 1, nullptr, nullptr, 0); }

void waiter_main(b200bgzf_ctx *ctx);
void comb_stop(b200bgzf_ctx *ctx);

int fail(b200bgzf_ctx *c, cudaError_t e, const char *where)
{
    snprintf(c->err, sizeof c->err, "%s: %s", where, cudaGetErrorString(e));
    return B200BGZF_E_CUDA;
}
#define CK(call)                                            \
    do {                                                    \
        cudaError_t e_ = (call);                            \
        if (e_ != cudaSuccess) return fail(ctx, e_, #call); \
    } while (0)

template <typename T>
cudaError_t grow(T **p, size_t *cap, size_t need, bool pinned = false)
{
    if (need <= *cap && *p) return cudaSuccess;
    if (*p) { if (pinned) cudaFreeHost(*p); else cudaFree(*p); *p = nullptr; }
    size_t n = std::max(need, *cap + *cap / 2);
    cudaError_t e = pinned ? cudaMallocHost((void **)p, n * sizeof(T)) : cudaMalloc((void **)p, n * sizeof(T));
    *cap = e == cudaSuccess ? n : 0;
    return e;
}

/* near-optimal levels: four matches per position and CTA; (re)sized for the largest grid the lane launches */
cudaError_t ensure_cand(Lane &l, int ctas)
{
    if (l.d_cand && l.cand_ctas >= ctas) return cudaSuccess;
    if (l.d_cand) { cudaFree(l.d_cand); l.d_cand = nullptr; l.cand_ctas = 0; }
    cudaError_t e = cudaMalloc((void **)&l.d_cand, (size_t)ctas * 4u * BG_MAX_BLOCK * sizeof(uint32_t));
    if (e == cudaSuccess) l.cand_ctas = ctas;
    return e;
}

/* Every exit of a pipelined host call (error exits included) leaves no batch in flight: a stale `pending` lane would be
 * "completed" by the next call with the old batch's sizes. */
struct PendingGuard {
    Lane *lanes;
    int n;
    PendingGuard(Lane *l, int count) : lanes(l), n(count) { settle(); }
    ~PendingGuard() { settle(); }
    void settle()
    {
        for (int i = 0; i < n; i++)
            if (lanes[i].pending) {
                if (lanes[i].stream) cudaStreamSynchronize(lanes[i].stream);
                lanes[i].pending = false;
            }
    }
};

void lane_free(Lane &l)
{
    cudaFree(l.d_in); cudaFree(l.d_slots); cudaFree(l.d_out); cudaFree(l.d_len); cudaFree(l.d_status);
    cudaFree(l.d_scratch); cudaFree(l.d_cand); cudaFree(l.d_off); cudaFree(l.d_inoff); cudaFree(l.d_outoff); cudaFree(l.d_inlen);
    cudaFree(l.d_total);
    if (l.h_total) cudaFreeHost(l.h_total);
    if (l.h_in) cudaFreeHost(l.h_in);
    if (l.h_out) cudaFreeHost(l.h_out);
    if (l.h_meta) cudaFreeHost(l.h_meta);
    if (l.done) cudaEventDestroy(l.done);
    cudaFree(l.one_dev);
    if (l.one_host) cudaFreeHost(l.one_host);
    cudaFree(l.d_rdec); cudaFree(l.d_rmeta);
    if (l.stream) cudaStreamDestroy(l.stream);
    l.~Lane();
    new (&l) Lane();
}

/* make sure a lane can process `blocks` compress blocks (device side); staging is grown on demand elsewhere */
int lane_reserve(b200bgzf_ctx *ctx, Lane &l, uint32_t blocks, size_t in_bytes, size_t out_bytes, bool slots = true, int ctas = 0)
{
    if (!l.stream) CK(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
    if (!l.d_total) {
        CK(cudaMalloc((void **)&l.d_total, 4 * sizeof(uint64_t)));
        CK(cudaMallocHost((void **)&l.h_total, 4 * sizeof(uint64_t)));
    }
    if (slots && !l.d_scratch) {
        l.scratch_ctas = ctas > 0 ? ctas : ctx->sms;
        CK(cudaMalloc((void **)&l.d_scratch, (size_t)l.scratch_ctas * BGZF_SCRATCH_WORDS * sizeof(uint32_t)));
    }
    if (blocks > l.cap_blocks || (slots && !l.d_slots)) {
        cudaFree(l.d_slots); cudaFree(l.d_len); cudaFree(l.d_status); cudaFree(l.d_off);
        cudaFree(l.d_inoff); cudaFree(l.d_outoff); cudaFree(l.d_inlen);
        l.d_slots = nullptr; l.d_len = l.d_status = l.d_inlen = nullptr; l.d_off = l.d_inoff = l.d_outoff = nullptr;
        l.cap_blocks = 0;
        if (slots) CK(cudaMalloc((void **)&l.d_slots, (size_t)blocks * BG_SLOT_BYTES + 64));
        CK(cudaMalloc((void **)&l.d_len, (size_t)blocks * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&l.d_status, (size_t)blocks * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&l.d_inlen, (size_t)blocks * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&l.d_off, (size_t)blocks * sizeof(uint64_t)));
        CK(cudaMalloc((void **)&l.d_inoff, (size_t)blocks * sizeof(uint64_t)));
        CK(cudaMalloc((void **)&l.d_outoff, (size_t)blocks * sizeof(uint64_t)));
        l.cap_blocks = blocks;
    }
    if (in_bytes) CK(grow(&l.d_in, &l.in_cap, in_bytes + 64));
    if (out_bytes) CK(grow(&l.d_out, &l.out_cap, out_bytes + 64));
    return 0;
}

/* one batch: compress kernel into slots, then scan + gather into `d_out` continuing at *d_total */
/* piece mode of a batch (BgzfCompressArgs.piece_mode ...): where the batch sits in the stream of pieces */
struct PieceLaunch {
    b200bgzf_piece_spec spec;
    uint64_t base, total;
    uint32_t *d_crc;
    uint32_t lead;              /* bytes of the stream in the device buffer before the batch's first block (match history) */
};

int launch_compress_batch(b200bgzf_ctx *ctx, Lane &l, const uint8_t *d_in, uint64_t in_bytes, uint32_t block_size,
                          const uint64_t *d_inoff, const uint32_t *d_inlen, uint32_t nblocks, int level, uint8_t *d_out,
                          int append_eof, cudaStream_t stream, bool fused = false, uint32_t hdr_bytes = 18,
                          const PieceLaunch *pl = nullptr)
{
    /* fused: the compress kernel's last CTA compacts the batch itself (l.d_total[2] is its arrival counter, zeroed with
     * l.d_total by the caller).  The pipelined host path uses it: a separate scan + gather launch per 32 MiB batch has to
     * find free SMs among the resident 1024-thread compress CTAs of the neighbouring batches, and every SM it touches
     * keeps a compress CTA waiting (measured: 41.3 -> 36.8 ms per GiB end to end without those launches). */
    if (nblocks) {
        BgzfCompressArgs a;
        memset(&a, 0, sizeof a);
        a.in = d_in;
        a.in_off = d_inoff;
        a.in_len = d_inlen;
        a.in_bytes = in_bytes;
        a.block_size = block_size;
        a.nblocks = nblocks;
        a.hdr_bytes = hdr_bytes;
        a.prm = bg_level_params(level);
        a.slots = l.d_slots;
        a.out_len = l.d_len;
        a.status = l.d_status;
        a.scratch = l.d_scratch;
        if (a.prm.opt_passes > 0) {
            CK(ensure_cand(l, l.scratch_ctas));
            a.cand = l.d_cand;
        }
        a.crctab = ctx->d_crctab;
        a.crcpow = ctx->d_crcpow;
        a.err_flag = (uint32_t *)(l.d_total + 1);
        a.prof = ctx->prof_on ? ctx->d_prof : nullptr;
        if (pl) {
            a.piece_mode = 1;
            a.member_blocks = pl->spec.member_blocks;
            a.head_gap = pl->spec.head_gap;
            a.tail_gap = pl->spec.tail_gap;
            a.no_final = pl->spec.no_final ? 1u : 0u;
            a.piece_base = pl->base;
            a.piece_total = pl->total;
            a.crc_out = pl->d_crc;
            a.history = pl->spec.history;
            a.lead = pl->lead;
        }
        if (fused) {
            a.gather_out = d_out;
            a.gather_off = l.d_off;
            a.gather_total = l.d_total;
            a.done_count = (uint32_t *)(l.d_total + 2);
        }
        const int grid = (int)std::min<uint32_t>(nblocks, (uint32_t)l.scratch_ctas);
        CK(bgzf_launch_compress(&a, grid, stream));
        ctx->launches += 1;
    }
    if (!fused || nblocks == 0) {
        CK(bgzf_launch_compact(l.d_slots, l.d_len, l.d_off, nblocks, d_out, l.d_total, append_eof, stream));
        ctx->launches += 2;
    }
    return 0;
}

bool level_ok(int level) { return level >= 1 && level <= 12; }

}  // namespace

extern "C" const char *b200bgzf_strerror(int code)
{
    switch (code) {
    case B200BGZF_OK: return "ok";
    case B200BGZF_E_NOFIT: return "compressed member does not fit";
    case B200BGZF_E_ARG: return "bad argument";
    case B200BGZF_E_CUDA: return "CUDA failure (no device, out of memory or launch error)";
    case B200BGZF_E_FORMAT: return "not BGZF or corrupt data";
    case B200BGZF_E_NOSPACE: return "output buffer too small";
    case B200BGZF_E_CRC: return "CRC32/ISIZE mismatch";
    default: return "unknown error";
    }
}

extern "C" void *b200bgzf_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void b200bgzf_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

extern "C" const char *b200bgzf_last_error(const b200bgzf_ctx *ctx) { return ctx ? ctx->err : ""; }
extern "C" unsigned long long b200bgzf_launch_count(const b200bgzf_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

extern "C" size_t b200bgzf_compress_bound(size_t in_bytes, uint32_t block_size)
{
    if (block_size == 0 || block_size > B200BGZF_MAX_BLOCK_SIZE) return 0;
    const size_t nb = (in_bytes + block_size - 1) / block_size;
    return in_bytes + nb * 38 + B200BGZF_EOF_BYTES;   /* 18 (BGZF) or 20 (MiGz) + 8 framing + up to two stored-block headers */
}

extern "C" int b200bgzf_create(b200bgzf_ctx **out, int device)
{
    if (!out) return B200BGZF_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return B200BGZF_E_CUDA;
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) return B200BGZF_E_CUDA;
    if (device >= ndev) return B200BGZF_E_ARG;
    b200bgzf_ctx *ctx = new b200bgzf_ctx();
    ctx->device = device;
    DeviceGuard g(device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || (size_t)prop.sharedMemPerBlockOptin < bgzf_compress_smem_bytes()) {
        snprintf(ctx->err, sizeof ctx->err, "device %d lacks the %zu bytes of shared memory per CTA this codec needs", device,
                 bgzf_compress_smem_bytes());
        delete ctx;
        return B200BGZF_E_CUDA;
    }
    ctx->sms = prop.multiProcessorCount;
    uint32_t tab[256];
    std::vector<uint32_t> pw(BG_THREADS);
    bg_make_crc_table(tab);
    bg_make_crc_pow(pw.data(), BG_THREADS);
    bool ok = cudaMalloc((void **)&ctx->d_crctab, sizeof tab) == cudaSuccess &&
              cudaMalloc((void **)&ctx->d_crcpow, pw.size() * 4) == cudaSuccess &&
              cudaMalloc((void **)&ctx->d_prof, BGZF_PROF_SLOTS * 8) == cudaSuccess &&
              cudaMemcpy(ctx->d_crctab, tab, sizeof tab, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(ctx->d_crcpow, pw.data(), pw.size() * 4, cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemset(ctx->d_prof, 0, BGZF_PROF_SLOTS * 8) == cudaSuccess;
    if (!ok) {
        b200bgzf_destroy(ctx);
        return B200BGZF_E_CUDA;
    }
    *out = ctx;
    return B200BGZF_OK;
}

extern "C" void b200bgzf_destroy(b200bgzf_ctx *ctx)
{
    if (!ctx) return;
    if (ctx->waiter_started) {
        {
            std::lock_guard<std::mutex> lk(ctx->waiter_mu);
            ctx->waiter_stop.store(true);
        }
        ctx->waiter_cv.notify_all();
        ctx->waiter.join();
    }
    {
        DeviceGuard g(ctx->device);
        comb_stop(ctx);
        cudaDeviceSynchronize();
        for (auto &l : ctx->lanes) lane_free(l);
        for (auto &l : ctx->hook_lanes) lane_free(l);
        cudaFree(ctx->d_crctab); cudaFree(ctx->d_crcpow); cudaFree(ctx->d_prof);
        cudaFree(ctx->d_idx_inoff); cudaFree(ctx->d_idx_outoff); cudaFree(ctx->d_idx_tileoff); cudaFree(ctx->d_idx_counts);
        cudaFree(ctx->d_idx_tilecount); cudaFree(ctx->d_idx_isize); cudaFree(ctx->d_idx_status); cudaFree(ctx->d_inf_status);
        cudaFree(ctx->d_idx_cand); cudaFree(ctx->d_idx_pick); cudaFree(ctx->d_idx_jump); cudaFree(ctx->d_idx_jump2); cudaFree(ctx->d_idx_reach);
        if (ctx->h_idx) cudaFreeHost(ctx->h_idx);
        cudaFree(ctx->d_rng_mem); cudaFree(ctx->d_rng_rw); cudaFree(ctx->d_rng_counts); cudaFree(ctx->d_rng_scratch);
        if (ctx->h_rng) cudaFreeHost(ctx->h_rng);
        if (ctx->h_rng_soff) cudaFreeHost(ctx->h_rng_soff);
        GzWork &z = ctx->gz;
        cudaFree(z.tile_count); cudaFree(z.u32); cudaFree(z.small32); cudaFree(z.tile_off); cudaFree(z.u64); cudaFree(z.small64);
        cudaFree(z.scratch); cudaFree(z.d_in); cudaFree(z.d_out);
        cudaFree(z.d_win); cudaFree(z.d_img); cudaFree(z.d_rout); cudaFree(z.d_carry); cudaFree(z.d_meta);
        if (z.h) cudaFreeHost(z.h);
        if (z.copy) cudaStreamDestroy(z.copy);
        if (z.ev) cudaEventDestroy(z.ev);
    }
    delete ctx;
}

extern "C" int b200bgzf_profile(b200bgzf_ctx *ctx, int enable, unsigned long long *cycles, int n, int reset)
{
    if (!ctx) return B200BGZF_E_ARG;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->prof_on = enable != 0;
    CK(cudaDeviceSynchronize());
    if (cycles && n > 0) CK(cudaMemcpy(cycles, ctx->d_prof, std::min(n, BGZF_PROF_SLOTS) * 8, cudaMemcpyDeviceToHost));
    if (reset) CK(cudaMemset(ctx->d_prof, 0, BGZF_PROF_SLOTS * 8));
    return 0;
}

/* ------------------------------------------------------------------------------------------------ */
/* compress                                                                                         */

extern "C" int b200bgzf_compress_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, uint32_t block_size, int level,
                                        void *d_out, size_t out_cap, size_t *out_bytes, unsigned flags, void *stream_)
{
    if (!ctx || !d_out || !out_bytes || (!d_in && in_bytes) || block_size == 0 || block_size > B200BGZF_MAX_BLOCK_SIZE || !level_ok(level))
        return B200BGZF_E_ARG;
    if (out_cap < b200bgzf_compress_bound(in_bytes, block_size)) return B200BGZF_E_NOSPACE;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    const uint64_t nb_total = (in_bytes + block_size - 1) / block_size;
    const uint32_t batch = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(nb_total, 1), kDeviceBatchBlocks);
    int r = lane_reserve(ctx, l, batch, 0, 0);
    if (r) return r;
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : l.stream;
    CK(cudaMemsetAsync(l.d_total, 0, 4 * sizeof(uint64_t), stream));
    const uint32_t hdr = (flags & B200BGZF_FRAME_MIGZ) ? 20u : 18u;
    const int eof = (flags & B200BGZF_APPEND_EOF) && hdr == 18u ? 1 : 0;
    uint64_t done = 0;
    do {
        const uint32_t nb = (uint32_t)std::min<uint64_t>(batch, nb_total - done);
        const uint64_t off = done * block_size;
        const bool last = done + nb >= nb_total;
        r = launch_compress_batch(ctx, l, (const uint8_t *)d_in + off, in_bytes - off, block_size, nullptr, nullptr, nb, level,
                                  (uint8_t *)d_out, eof && last, stream, false, hdr);
        if (r) return r;
        done += nb;
    } while (done < nb_total);
    CK(cudaMemcpyAsync(l.h_total, l.d_total, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    *out_bytes = (size_t)l.h_total[0] + (eof ? B200BGZF_EOF_BYTES : 0);
    return l.h_total[1] ? B200BGZF_E_NOFIT : B200BGZF_OK;
}

namespace {
/* the pipelined host-buffer path.  member_off (optional): where every member (piece) starts in `out` — the offsets the
 * device scan computes anyway.  ps (optional): piece mode; piece_crc then receives the CRC-32 of every block's input. */
int compress_host_impl(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level, void *out,
                       size_t out_cap, size_t *out_bytes, unsigned flags, uint64_t *member_off, size_t member_cap,
                       const b200bgzf_piece_spec *ps, uint32_t *piece_crc)
{
    if (!ctx || !out || !out_bytes || (!in && in_bytes) || block_size == 0 || block_size > B200BGZF_MAX_BLOCK_SIZE || !level_ok(level))
        return B200BGZF_E_ARG;
    if (out_cap < b200bgzf_compress_bound(in_bytes, block_size) + (ps ? b200bgzf_pieces_gap_bytes(in_bytes, block_size, ps) : 0)) return B200BGZF_E_NOSPACE;
    if (member_off && member_cap < (in_bytes + block_size - 1) / block_size) return B200BGZF_E_NOSPACE;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    PendingGuard pg(ctx->lanes, kLanes);
    const uint64_t nb_total = (in_bytes + block_size - 1) / block_size;
    /* batches rotate through the lanes (H2D, kernels, D2H on the lane's stream).  Measured: 400-512 blocks per batch is
     * best; multiples of the SM count are 5 % WORSE — when every CTA of a launch finishes at the same moment nothing of the
     * next launch overlaps with the hand-over, while uneven block counts let its CTAs trickle in */
    static const uint32_t host_batch = [] { const char *e = getenv("B200BGZF_HOST_BATCH"); return e && atoi(e) > 0 ? (uint32_t)atoi(e) : kHostBatchBlocks; }();
    static const uint32_t first_batch = [] { const char *e = getenv("B200BGZF_FIRST_BATCH"); return e && atoi(e) > 0 ? (uint32_t)atoi(e) : 0u; }();
    const uint32_t batch = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(nb_total, 1), host_batch);
    const size_t batch_in = (size_t)batch * block_size + (ps ? ps->history : 0u);
    const size_t batch_out = b200bgzf_compress_bound(batch_in, block_size) + (ps ? (size_t)batch * (ps->head_gap + ps->tail_gap) : 0);
    static const int nlanes = [] { const char *e = getenv("B200BGZF_LANES"); return e && atoi(e) > 0 ? std::min(atoi(e), kLanes) : kLanes; }();
    uint32_t cur = first_batch ? std::min(first_batch, batch) : batch;
    size_t host_off = 0;
    bool nofit = false;
    int r;
    auto complete = [&](Lane &l) -> int {
        CK(cudaStreamSynchronize(l.stream));
        const size_t total = (size_t)l.h_total[0];
        if (l.h_total[1]) nofit = true;
        if (member_off)
            for (uint32_t k = 0; k < l.pend_nb; k++) member_off[l.pend_first + k] = host_off + l.h_meta[k];
        if (piece_crc) memcpy(piece_crc + l.pend_first, l.h_meta + batch, l.pend_nb * sizeof(uint32_t));
        CK(cudaMemcpyAsync((uint8_t *)out + host_off, l.d_out, total, cudaMemcpyDeviceToHost, l.stream));
        host_off += total;
        l.pending = false;
        return 0;
    };
    uint64_t done = 0, i = 0;
    while (done < nb_total) {
        Lane &l = ctx->lanes[i % nlanes];
        if (l.pending && (r = complete(l))) return r;
        if ((r = lane_reserve(ctx, l, batch, batch_in, batch_out))) return r;
        const uint32_t nb = (uint32_t)std::min<uint64_t>(cur, nb_total - done);
        cur = std::min<uint32_t>(batch, cur * 2);
        const uint64_t off = done * block_size;
        const size_t bytes = (size_t)std::min<uint64_t>((uint64_t)nb * block_size, in_bytes - off);
        /* primed pieces: the batch's first blocks find their history in front of them in the device buffer */
        uint32_t lead = 0;
        if (ps && ps->history) {
            const uint64_t before = (ps->piece_base + done) * (uint64_t)block_size;      /* bytes of the stream before this batch */
            lead = (uint32_t)std::min<uint64_t>(ps->history, before);
        }
        CK(cudaMemcpyAsync(l.d_in, (const uint8_t *)in + off - lead, bytes + lead, cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemsetAsync(l.d_total, 0, 4 * sizeof(uint64_t), l.stream));
        PieceLaunch pl;
        if (ps) {
            pl.spec = *ps;
            pl.base = ps->piece_base + done;
            pl.total = ps->piece_total ? ps->piece_total : nb_total;
            pl.d_crc = l.d_inlen;                               /* (unused by fixed-size batches) */
            pl.lead = lead;
        }
        if ((r = launch_compress_batch(ctx, l, l.d_in + lead, bytes, block_size, nullptr, nullptr, nb, level, l.d_out, 0, l.stream, true,
                                       (flags & B200BGZF_FRAME_MIGZ) ? 20u : 18u, ps ? &pl : nullptr))) return r;
        CK(cudaMemcpyAsync(l.h_total, l.d_total, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, l.stream));
        if (member_off || piece_crc) {
            /* pinned: u64[batch] member offsets, then u32[batch] CRCs */
            CK(grow(&l.h_meta, &l.meta_cap, (size_t)batch + ((size_t)batch + 1) / 2, true));
            if (member_off) CK(cudaMemcpyAsync(l.h_meta, l.d_off, nb * sizeof(uint64_t), cudaMemcpyDeviceToHost, l.stream));
            if (piece_crc) CK(cudaMemcpyAsync(l.h_meta + batch, l.d_inlen, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, l.stream));
            l.pend_first = done;
            l.pend_nb = nb;
        }
        l.pending = true;
        done += nb;
        i++;
    }
    /* drain in submission order */
    for (uint64_t k = 0; k < (uint64_t)nlanes; k++) {
        Lane &l = ctx->lanes[(i + k) % nlanes];
        if (l.pending && (r = complete(l))) return r;
    }
    for (auto &l : ctx->lanes)
        if (l.stream) CK(cudaStreamSynchronize(l.stream));
    if ((flags & B200BGZF_APPEND_EOF) && !(flags & B200BGZF_FRAME_MIGZ) && !ps) {
        static const uint8_t eof[28] = { 0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0,
                                         0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
        memcpy((uint8_t *)out + host_off, eof, sizeof eof);
        host_off += sizeof eof;
    }
    *out_bytes = host_off;
    return nofit ? B200BGZF_E_NOFIT : B200BGZF_OK;
}
}  // namespace

extern "C" int b200bgzf_compress_host_index(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level, void *out,
                                            size_t out_cap, size_t *out_bytes, unsigned flags, uint64_t *member_off, size_t member_cap)
{
    return compress_host_impl(ctx, in, in_bytes, block_size, level, out, out_cap, out_bytes, flags, member_off, member_cap, nullptr, nullptr);
}

extern "C" size_t b200bgzf_pieces_gap_bytes(size_t in_bytes, uint32_t block_size, const b200bgzf_piece_spec *ps)
{
    if (!ps || !block_size || !ps->member_blocks) return 0;
    const uint64_t nb = (in_bytes + block_size - 1) / block_size, k = ps->member_blocks;
    /* members that begin / end inside the pieces [base, base + nb) of the stream */
    const uint64_t b0 = ps->piece_base, b1 = b0 + nb, total = ps->piece_total ? ps->piece_total : b1;
    const uint64_t firsts = (b1 + k - 1) / k - (b0 + k - 1) / k;
    const uint64_t lasts = b1 / k - b0 / k + (nb && b1 == total && total % k ? 1u : 0u);
    return (size_t)(firsts * ps->head_gap + lasts * ps->tail_gap);
}

extern "C" int b200bgzf_compress_pieces_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level,
                                             const b200bgzf_piece_spec *ps, void *out, size_t out_cap, size_t *out_bytes,
                                             uint64_t *piece_off, uint32_t *piece_crc, size_t piece_cap)
{
    if (!ps || ps->member_blocks == 0 || ps->head_gap > B200BGZF_MAX_GAP || ps->tail_gap > B200BGZF_MAX_GAP) return B200BGZF_E_ARG;
    if (ps->piece_total && ps->piece_base + (in_bytes + block_size - 1) / block_size > ps->piece_total) return B200BGZF_E_ARG;
    if (ps->history % BG_HISTORY_STEP || ps->history > BG_MAX_HISTORY || (ps->history && (uint64_t)block_size + ps->history > BG_MAX_BLOCK))
        return B200BGZF_E_ARG;
    if (piece_crc && piece_cap < (in_bytes + block_size - 1) / block_size) return B200BGZF_E_NOSPACE;
    return compress_host_impl(ctx, in, in_bytes, block_size, level, out, out_cap, out_bytes, 0, piece_off, piece_cap, ps, piece_crc);
}

extern "C" int b200bgzf_compress_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, uint32_t block_size, int level, void *out,
                                      size_t out_cap, size_t *out_bytes, unsigned flags)
{
    return b200bgzf_compress_host_index(ctx, in, in_bytes, block_size, level, out, out_cap, out_bytes, flags, nullptr, 0);
}

/* .gzi as bgzip -i / bgzf_index_dump write it: u64 count, then (compressed offset, uncompressed offset) of every member
 * but the first, all little endian */
extern "C" size_t b200bgzf_gzi_format(const uint64_t *caddr, const uint64_t *uaddr, size_t nmembers, void *dst, size_t cap)
{
    const size_t entries = nmembers ? nmembers - 1 : 0, need = 8 + 16 * entries;
    if (!dst || cap < need || (nmembers && (!caddr || !uaddr))) return 0;
    uint8_t *o = (uint8_t *)dst;
    auto put = [&](uint64_t v) { for (int k = 0; k < 8; k++) *o++ = (uint8_t)(v >> (8 * k)); };
    put(entries);
    for (size_t i = 1; i < nmembers; i++) { put(caddr[i]); put(uaddr[i]); }
    return need;
}

namespace {

/* one staged batch of independent payloads on a given lane (used by the hook and the block-list API) */
int compress_blocks_on_lane(b200bgzf_ctx *ctx, Lane &l, const void *const *src, const uint32_t *slen, void *const *dst, size_t *dlen,
                            int *status, uint32_t nb, int level)
{
    int r = lane_reserve(ctx, l, nb, (size_t)nb * BG_SLOT_BYTES, (size_t)nb * BG_SLOT_BYTES, true, nb <= kHookLaneBlocks ? (int)kHookLaneBlocks : 0);
    if (r) return r;
    CK(grow(&l.h_in, &l.host_in_cap, (size_t)nb * BG_SLOT_BYTES, true));
    CK(grow(&l.h_out, &l.host_out_cap, (size_t)nb * BG_SLOT_BYTES, true));
    size_t meta_need = (size_t)nb * 3;
    CK(grow(&l.h_meta, &l.meta_cap, meta_need, true));
    uint64_t *h_inoff = l.h_meta;
    uint32_t *h_inlen = (uint32_t *)(l.h_meta + nb);
    uint32_t *h_len = (uint32_t *)(l.h_meta + 2 * nb);
    size_t pos = 0;
    for (uint32_t b = 0; b < nb; b++) {
        h_inoff[b] = pos;
        h_inlen[b] = slen[b];
        memcpy(l.h_in + pos, src[b], slen[b]);
        pos += (slen[b] + 15u) & ~(size_t)15u;    /* keep every payload 16-byte aligned for the TMA path */
    }
    CK(cudaMemcpyAsync(l.d_in, l.h_in, pos ? pos : 16, cudaMemcpyHostToDevice, l.stream));
    CK(cudaMemcpyAsync(l.d_inoff, h_inoff, nb * sizeof(uint64_t), cudaMemcpyHostToDevice, l.stream));
    CK(cudaMemcpyAsync(l.d_inlen, h_inlen, nb * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream));
    CK(cudaMemsetAsync(l.d_total, 0, 4 * sizeof(uint64_t), l.stream));
    if ((r = launch_compress_batch(ctx, l, l.d_in, 0, 0, l.d_inoff, l.d_inlen, nb, level, l.d_out, 0, l.stream))) return r;
    CK(cudaMemcpyAsync(l.h_total, l.d_total, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, l.stream));
    CK(cudaMemcpyAsync(h_len, l.d_len, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, l.stream));
    CK(cudaStreamSynchronize(l.stream));
    const size_t total = (size_t)l.h_total[0];
    if (total) {
        CK(cudaMemcpyAsync(l.h_out, l.d_out, total, cudaMemcpyDeviceToHost, l.stream));
        CK(cudaStreamSynchronize(l.stream));
    }
    size_t o = 0;
    int worst = 0;
    for (uint32_t b = 0; b < nb; b++) {
        const uint32_t n = h_len[b];
        int st = 0;
        if (n == 0 || n > dlen[b]) st = B200BGZF_E_NOFIT;
        else { memcpy(dst[b], l.h_out + o, n); dlen[b] = n; }
        o += n;
        if (status) status[b] = st;
        if (st) worst = st;
    }
    return worst;
}

/* One payload, one member: the shape of every call the LD_PRELOAD hook makes.  Latency is everything here (the caller
 * blocks), so the round trip is pared down to: copy in, one kernel, ONE copy out (the whole 64 KiB slot with the member
 * size and status words parked right behind it), one synchronisation.  No scan, no gather, no metadata uploads. */
int compress_one_on_lane(b200bgzf_ctx *ctx, Lane &l, const void *src, uint32_t slen, void *dst, size_t *dlen, int *status, int level,
                         bool sleep_wait, int split)
{
    /* first use of the lane: a stream and two slabs (each allocation is a device-wide synchronisation, and a pool of
     * callers hits this at the same moment) */
    constexpr size_t kIn = BG_SLOT_BYTES + 64, kSlot = BG_SLOT_BYTES + 64,
                     kScratch = ((size_t)BGZF_SCRATCH_WORDS + BGZF_SPLIT_EXTRA_WORDS) * sizeof(uint32_t);
    if (!l.stream) CK(cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking));
    if (!l.one_dev) {
        CK(cudaMalloc((void **)&l.one_dev, kIn + kSlot + kScratch + 64));
        CK(cudaMallocHost((void **)&l.one_host, kIn + kSlot + 64));
        l.d_one = (uint32_t *)(l.one_dev + kIn + kSlot + kScratch);
        l.h_flag = (volatile uint32_t *)(l.one_host + kIn + kSlot);
        const uint32_t one = 1;
        CK(cudaMemcpyAsync(l.d_one, &one, sizeof one, cudaMemcpyHostToDevice, l.stream));
        CK(cudaStreamSynchronize(l.stream));
    }
    uint8_t *d_in = l.one_dev, *d_slot = l.one_dev + kIn, *h_in = l.one_host, *h_out = l.one_host + kIn;
    uint32_t *d_scratch = (uint32_t *)(l.one_dev + kIn + kSlot);
    memcpy(h_in, src, slen);
    const size_t up = ((size_t)slen + 15u) & ~(size_t)15u;
    if (up) CK(cudaMemcpyAsync(d_in, h_in, up, cudaMemcpyHostToDevice, l.stream));
    uint32_t *tail = (uint32_t *)(d_slot + BG_SLOT_BYTES);    /* [0] member size, [1] status, [2] error flag (the slot's pad) */
    BgzfCompressArgs a;
    memset(&a, 0, sizeof a);
    a.in = d_in;
    a.in_bytes = slen;
    a.block_size = B200BGZF_MAX_BLOCK_SIZE;
    a.nblocks = 1;
    a.prm = bg_level_params(level);
    a.slots = d_slot;
    a.out_len = tail;
    a.status = tail + 1;
    a.err_flag = tail + 2;
    a.scratch = d_scratch;
    if (a.prm.opt_passes > 0) {
        if (!l.d_cand) CK(cudaMalloc((void **)&l.d_cand, (size_t)std::max(l.scratch_ctas, 1) * 4u * BG_MAX_BLOCK * sizeof(uint32_t)));
        a.cand = l.d_cand;
    }
    a.crctab = ctx->d_crctab;
    a.crcpow = ctx->d_crcpow;
    a.prof = nullptr;
    /* few callers, many idle SMs: let a cluster of CTAs share the search of this one block (same bytes out) */
    bool launched = false;
    if (split > 1 && slen >= 8192u && !ctx->no_clusters.load(std::memory_order_relaxed)) {
        launched = bgzf_launch_compress_split(&a, split, l.stream) == cudaSuccess;
        if (!launched) {               /* a device or partition that cannot place the cluster: stay on the one-SM kernel */
            cudaGetLastError();
            ctx->no_clusters.store(true, std::memory_order_relaxed);
        }
    }
    if (!launched) CK(bgzf_launch_compress(&a, 1, l.stream));
    ctx->launches += 1;
    CK(cudaMemcpyAsync(h_out, d_slot, (size_t)BG_SLOT_BYTES + 8, cudaMemcpyDeviceToHost, l.stream));
    if (sleep_wait) {
        /* more callers in flight than host cores (samtools -@64 on a 16-core box): a spinning wait would starve the
         * others and a pool of sleep-pollers is at the mercy of the scheduler (1-5 GB/s run to run), so the caller sleeps
         * on its lane's futex word and the context's ONE completion thread wakes it (a blocking-sync event costs about a
         * millisecond per wake-up here: not used) */
        if (!l.done) CK(cudaEventCreateWithFlags(&l.done, cudaEventDisableTiming));
        *l.h_flag = 0;
        CK(cudaMemcpyAsync((void *)l.h_flag, l.d_one, sizeof(uint32_t), cudaMemcpyDeviceToHost, l.stream));
        CK(cudaEventRecord(l.done, l.stream));
        {
            std::lock_guard<std::mutex> lk(ctx->waiter_mu);
            if (!ctx->waiter_started) {
                ctx->waiter = std::thread(waiter_main, ctx);
                ctx->waiter_started = true;
            }
            l.wait_state.store(1, std::memory_order_release);
            ctx->waiter_inflight.fetch_add(1);
        }
        ctx->waiter_cv.notify_one();
        futex_wait_while(&l.wait_state, 1u);
        l.wait_state.store(0, std::memory_order_relaxed);
        CK(l.wait_result);
    } else {
        CK(cudaStreamSynchronize(l.stream));
    }
    const uint32_t n = *(const uint32_t *)(h_out + BG_SLOT_BYTES);
    int st = 0;
    if (n == 0 || n > *dlen) st = B200BGZF_E_NOFIT;
    else { memcpy(dst, h_out, n); *dlen = n; }
    if (status) *status = st;
    return st;
}

void waiter_main(b200bgzf_ctx *ctx)
{
    cudaSetDevice(ctx->device);
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(ctx->waiter_mu);
            ctx->waiter_cv.wait(lk, [&] { return ctx->waiter_stop.load() || ctx->waiter_inflight.load() > 0; });
            if (ctx->waiter_stop.load()) return;
        }
        /* the lanes' flags are plain pinned memory: polling them takes no driver lock away from the callers that are
         * launching at the same time; the event is only asked now and then, to notice a failed stream */
        unsigned spins = 0;
        while (ctx->waiter_inflight.load(std::memory_order_acquire) > 0 && !ctx->waiter_stop.load(std::memory_order_relaxed)) {
            const bool ask = (++spins & 0x3fffu) == 0;
            for (auto &h : ctx->hook_lanes) {
                if (h.wait_state.load(std::memory_order_acquire) != 1u) continue;
                cudaError_t q = cudaSuccess;
                if (!*h.h_flag) {
                    if (!ask) continue;
                    q = cudaEventQuery(h.done);
                    if (q == cudaErrorNotReady) continue;
                }
                h.wait_result = q;
                ctx->waiter_inflight.fetch_sub(1);
                h.wait_state.store(2u, std::memory_order_release);
                futex_wake_one(&h.wait_state);
            }
        }
    }
}

/* ---- combiner ---- */
int comb_start(b200bgzf_ctx *ctx);

void comb_fail_batch(b200bgzf_ctx *ctx, CombBatch &b, int rc)
{
    Combiner &cb = ctx->comb;
    for (int k = 0; k < b.n; k++) {
        CombSlot &sl = cb.slots[b.slots[k]];
        sl.rc = rc;
        sl.out_len = 0;
        for (int j = 0; j < 4; j++) sl.child[j] = -1;
        cb.pending.fetch_sub(1);
        sl.state.store(4u, std::memory_order_release);
        futex_wake_one(&sl.state);
    }
    b.n = 0;
    b.inflight = false;
}

void comb_main(b200bgzf_ctx *ctx)
{
    Combiner &cb = ctx->comb;
    cudaSetDevice(ctx->device);
    uint64_t first_seen = 0;
    unsigned spins = 0;
    for (;;) {
        if (cb.pending.load(std::memory_order_acquire) == 0) {
            std::unique_lock<std::mutex> lk(cb.mu);
            cb.sleeping.store(true);
            cb.cv.wait(lk, [&] { return cb.stop.load() || cb.pending.load() > 0; });
            cb.sleeping.store(false);
        }
        if (cb.stop.load()) return;
        /* members that have arrived (the flags are plain pinned memory; the stream is only asked now and then, to notice a failure) */
        const bool ask = (++spins & 0xffffu) == 0;
        for (int bi = 0; bi < kCombBatches; bi++) {
            CombBatch &b = cb.batches[bi];
            if (!b.inflight) continue;
            if (!*b.h_flag) {
                if (ask) {
                    const cudaError_t q = cudaStreamQuery(b.stream);
                    if (q != cudaSuccess && q != cudaErrorNotReady) {
                        snprintf(ctx->err, sizeof ctx->err, "hook combiner: %s", cudaGetErrorString(q));
                        comb_fail_batch(ctx, b, B200BGZF_E_CUDA);
                    }
                }
                continue;
            }
            /* waking a sleeper is a system call of several microseconds: the dispatcher wakes four callers of the batch, each
             * of them four more, and so on, instead of paying for all of them itself while new payloads wait */
            for (int k = 0; k < b.n; k++) {
                CombSlot &sl = cb.slots[b.slots[k]];
                sl.rc = 0;
                for (int j = 0; j < 4; j++) sl.child[j] = 4 * (k + 1) + j < b.n ? b.slots[4 * (k + 1) + j] : -1;
            }
            cb.pending.fetch_sub(b.n);
            for (int k = 0; k < b.n; k++) cb.slots[b.slots[k]].state.store(4u, std::memory_order_release);
            for (int k = 0; k < b.n && k < 4; k++) futex_wake_one(&cb.slots[b.slots[k]].state);
            b.inflight = false;
        }
        /* ready payloads -> one batch */
        CombBatch *nb = nullptr;
        int busy = 0;
        for (auto &b : cb.batches) {
            if (b.inflight) busy++;
            else if (!nb) nb = &b;
        }
        if (!nb) continue;
        int n = 0, level = 0;
        for (int i = 0; i < kCombSlots && n < kCombBatchMax; i++) {
            CombSlot &sl = cb.slots[i];
            if (sl.state.load(std::memory_order_acquire) != 2u) continue;
            if (n == 0) level = sl.level;
            else if (sl.level != level) continue;
            nb->slots[n] = i;
            nb->h_inoff[n] = (uint64_t)i * kCombInStride;
            nb->h_outoff[n] = (uint64_t)i * kCombOutStride;
            nb->h_inlen[n] = sl.slen;
            n++;
        }
        if (n == 0) { first_seen = 0; continue; }
        /* Fewer payloads than a batch is worth while other batches are still running: wait for the callers that are about to
         * arrive (up to 120 us).  A batch costs this thread about 60 us of driver calls and wake-ups whatever its size; with
         * payloads trickling in one by one it would otherwise spend all its time launching batches of two or three. */
        const int want = std::min(32, std::max(1, ctx->one_block_callers.load(std::memory_order_relaxed) / 4));
        if (n < want && busy > 0) {
            struct timespec ts;
            clock_gettime(CLOCK_MONOTONIC, &ts);
            const uint64_t now = (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec;
            if (first_seen == 0) first_seen = now;
            if (now - first_seen < 120000ull) continue;
        }
        first_seen = 0;
        for (int k = 0; k < n; k++) cb.slots[nb->slots[k]].state.store(3u, std::memory_order_relaxed);
        nb->n = n;
        nb->inflight = true;
        *nb->h_flag = 0;
        BgzfCompressArgs a;
        memset(&a, 0, sizeof a);
        a.in = cb.h_in;
        a.in_off = nb->h_inoff;
        a.in_len = nb->h_inlen;
        a.nblocks = (uint32_t)n;
        a.prm = bg_level_params(level);
        a.slots = nb->d_slots;
        a.out_len = nb->d_meta;
        a.status = nb->d_meta + kCombBatchMax;
        a.err_flag = nb->d_meta + 2 * kCombBatchMax;
        a.scratch = nb->d_scratch;
        a.crctab = ctx->d_crctab;
        a.crcpow = ctx->d_crcpow;
        cudaError_t e = cudaSuccess;
        if (a.prm.opt_passes > 0) {
            if (!nb->d_cand) e = cudaMalloc((void **)&nb->d_cand, (size_t)kCombBatchMax * 4u * BG_MAX_BLOCK * sizeof(uint32_t));
            a.cand = nb->d_cand;
        }
        /* (B200BGZF_COMB_SPLIT=1: let every block of a batch have a cluster of 2, 4 or 8 of the SMs the blocks in flight leave
         * over.  Measured and left off: many clusters from several streams place badly — 64 callers fell from 5 to 1-2.6 GB/s,
         * 16 callers from 490 to 707 us per call.) */
        static const bool comb_split = [] { const char *e = getenv("B200BGZF_COMB_SPLIT"); return e && atoi(e) > 0; }();
        int flying = n, split = 1;
        bool small = false;
        for (auto &b : cb.batches)
            if (b.inflight && &b != nb) flying += b.n;
        for (int k = 0; k < n; k++) small = small || nb->h_inlen[k] < 8192u;
        if (comb_split && !small && !ctx->no_clusters.load(std::memory_order_relaxed)) split = flying <= 18 ? 8 : flying <= 37 ? 4 : flying <= 74 ? 2 : 1;
        if (e == cudaSuccess && split > 1) {
            e = bgzf_launch_compress_split(&a, split, nb->stream);
            if (e != cudaSuccess) {
                cudaGetLastError();
                ctx->no_clusters.store(true, std::memory_order_relaxed);
                e = bgzf_launch_compress(&a, n, nb->stream);
            }
        } else if (e == cudaSuccess) {
            e = bgzf_launch_compress(&a, n, nb->stream);
        }
        if (e == cudaSuccess) e = bgzf_launch_deliver(nb->d_slots, nb->d_meta, nb->h_outoff, cb.h_out, (uint32_t)n, nb->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync((void *)nb->h_flag, nb->d_meta + 2 * kCombBatchMax + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, nb->stream);
        ctx->launches += 2;
        if (e != cudaSuccess) {
            snprintf(ctx->err, sizeof ctx->err, "hook combiner: %s", cudaGetErrorString(e));
            comb_fail_batch(ctx, *nb, B200BGZF_E_CUDA);
        }
    }
}

int comb_start(b200bgzf_ctx *ctx)
{
    Combiner &cb = ctx->comb;
    std::lock_guard<std::mutex> lk(cb.mu);
    if (cb.up) return 0;
    if (cb.failed) return B200BGZF_E_CUDA;
    cb.failed = true;                                   /* until everything below has worked */
    CK(cudaMallocHost((void **)&cb.h_in, (size_t)kCombSlots * kCombInStride));
    CK(cudaMallocHost((void **)&cb.h_out, (size_t)kCombSlots * kCombOutStride));
    for (auto &b : cb.batches) {
        CK(cudaStreamCreateWithFlags(&b.stream, cudaStreamNonBlocking));
        CK(cudaMalloc((void **)&b.d_slots, (size_t)kCombBatchMax * BG_SLOT_BYTES + 64));
        CK(cudaMalloc((void **)&b.d_meta, (2 * kCombBatchMax + 8) * sizeof(uint32_t)));
        CK(cudaMallocHost((void **)&b.h_meta, (2 * kCombBatchMax + 8) * sizeof(uint32_t)));
        CK(cudaMallocHost((void **)&b.h_inoff, 2 * kCombBatchMax * sizeof(uint64_t)));
        b.h_outoff = b.h_inoff + kCombBatchMax;
        CK(cudaMallocHost((void **)&b.h_inlen, kCombBatchMax * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&b.d_scratch, (size_t)kCombBatchMax * (BGZF_SCRATCH_WORDS + BGZF_SPLIT_EXTRA_WORDS) * sizeof(uint32_t)));
        b.h_flag = b.h_meta + 2 * kCombBatchMax + 4;
        const uint32_t one = 1;
        CK(cudaMemcpy(b.d_meta + 2 * kCombBatchMax + 1, &one, sizeof one, cudaMemcpyHostToDevice));
    }
    cb.th = std::thread(comb_main, ctx);
    cb.up = true;
    cb.failed = false;
    return 0;
}

void comb_stop(b200bgzf_ctx *ctx)
{
    Combiner &cb = ctx->comb;
    if (cb.up) {
        {
            std::lock_guard<std::mutex> lk(cb.mu);
            cb.stop.store(true);
        }
        cb.cv.notify_all();
        cb.th.join();
    }
    if (cb.h_in) cudaFreeHost(cb.h_in);
    if (cb.h_out) cudaFreeHost(cb.h_out);
    for (auto &b : cb.batches) {
        cudaFree(b.d_slots); cudaFree(b.d_meta); cudaFree(b.d_scratch); cudaFree(b.d_cand);
        if (b.h_meta) cudaFreeHost(b.h_meta);
        if (b.h_inoff) cudaFreeHost(b.h_inoff);
        if (b.h_inlen) cudaFreeHost(b.h_inlen);
        if (b.stream) cudaStreamDestroy(b.stream);
    }
}

/* one payload through the combiner; returns 2 if it cannot take the call (no free slot, set-up failed): use a lane */
int compress_one_combined(b200bgzf_ctx *ctx, const void *src, uint32_t slen, void *dst, size_t *dlen, int *status, int level)
{
    Combiner &cb = ctx->comb;
    if (!cb.up && comb_start(ctx) != 0) return 2;
    static thread_local int hint = -1;
    int si = -1;
    for (int k = 0; k < kCombSlots; k++) {
        const int i = hint >= 0 ? (hint + k) % kCombSlots : (int)((std::hash<std::thread::id>()(std::this_thread::get_id()) + k) % kCombSlots);
        uint32_t expect = 0;
        if (cb.slots[i].state.compare_exchange_strong(expect, 1u, std::memory_order_acquire)) { si = i; break; }
    }
    if (si < 0) return 2;
    hint = si;
    CombSlot &sl = cb.slots[si];
    memcpy(cb.h_in + (size_t)si * kCombInStride, src, slen);
    sl.slen = slen;
    sl.level = level;
    cb.pending.fetch_add(1);
    sl.state.store(2u, std::memory_order_release);
    if (cb.sleeping.load(std::memory_order_acquire)) {
        std::lock_guard<std::mutex> lk(cb.mu);
        cb.cv.notify_one();
    }
    for (;;) {
        const uint32_t st = sl.state.load(std::memory_order_acquire);
        if (st == 4u) break;
        syscall(SYS_futex, (uint32_t *)&sl.state, FUTEX_WAIT_PRIVATE, st, nullptr, nullptr, 0);
    }
    for (int j = 0; j < 4; j++)
        if (sl.child[j] >= 0) futex_wake_one(&cb.slots[sl.child[j]].state);
    int rc = sl.rc;
    if (rc == 0) {
        const uint8_t *mine = cb.h_out + (size_t)si * kCombOutStride;
        const uint32_t n = *(const volatile uint32_t *)mine;
        if (n == 0 || n > *dlen) rc = B200BGZF_E_NOFIT;
        else { memcpy(dst, mine + 16, n); *dlen = n; }
    }
    sl.state.store(0u, std::memory_order_release);
    if (status) *status = rc > 0 ? rc : 0;
    return rc;
}

}  // namespace

extern "C" int b200bgzf_compress_blocks_host(b200bgzf_ctx *ctx, const void *const *src, const uint32_t *slen, void *const *dst,
                                             size_t *dlen, int *status, uint32_t nblocks, int level)
{
    if (!ctx || !src || !slen || !dst || !dlen || !level_ok(level)) return B200BGZF_E_ARG;
    for (uint32_t b = 0; b < nblocks; b++)
        if (slen[b] > B200BGZF_MAX_BLOCK_SIZE || dlen[b] < 26) return B200BGZF_E_ARG;
    if (nblocks == 0) return 0;
    DeviceGuard g(ctx->device);
    if (nblocks == 1) {
        /* many concurrent one-block callers (htslib's pool with more threads than this host has cores): hand the payload to the
         * combiner instead of driving the GPU from every caller (B200BGZF_HOOK_BATCH=0 / 1 forces the choice; for measurements) */
        struct Count { std::atomic<int> &c; int now; explicit Count(std::atomic<int> &x) : c(x), now(x.fetch_add(1) + 1) {} ~Count() { c.fetch_sub(1); } } count(ctx->one_block_callers);
        static const int forced_batch = [] { const char *e = getenv("B200BGZF_HOOK_BATCH"); return e && *e ? atoi(e) : -1; }();
        if (forced_batch == 1 || (forced_batch < 0 && count.now > 36)) {
            const int r = compress_one_combined(ctx, src[0], slen[0], dst[0], dlen, status, level);
            if (r != 2) return r;
        }
    }
    if (nblocks <= kHookLaneBlocks) {
        /* small calls (the hook): grab any free one-block lane so concurrent callers run on different SMs */
        Lane *l = nullptr;
        int in_flight = 0;
        {
            std::unique_lock<std::mutex> lk(ctx->hook_mu);
            for (;;) {
                in_flight = 0;
                for (auto &h : ctx->hook_lanes) {
                    if (h.busy) in_flight++;
                    else if (!l) l = &h;
                }
                if (l) break;
                ctx->hook_cv.wait(lk);
            }
            l->busy = true;
        }
        static const int cores = (int)std::max(1u, std::thread::hardware_concurrency());
        /* one-member calls share the GPU between the callers in flight: up to 18 of them get a cluster of 8 SMs each (144
         * of the 148 SMs), up to 36 a cluster of 4, beyond that one SM each (B200BGZF_SPLIT=1/2/4/8 forces a size; for
         * measurements).  Measured, MB/s with 1 / 8 / 16 callers: one SM 130 / 1020 / 2000, clusters of 8: 291 / 2130 / 3500 */
        static const int forced = [] { const char *e = getenv("B200BGZF_SPLIT"); return e && *e ? atoi(e) : 0; }();
        const int callers = in_flight + 1;
        int split = forced > 0 ? std::min(forced, BGZF_SPLIT_MAX) : callers <= 18 ? 8 : callers <= 36 ? 4 : 1;
        if (split == 3) split = 2;
        if (split > 4 && split < 8) split = 4;
        int r = nblocks == 1 ? compress_one_on_lane(ctx, *l, src[0], slen[0], dst[0], dlen, status, level, in_flight + 1 > cores, split)
                             : compress_blocks_on_lane(ctx, *l, src, slen, dst, dlen, status, nblocks, level);
        {
            std::lock_guard<std::mutex> lk(ctx->hook_mu);
            l->busy = false;
        }
        ctx->hook_cv.notify_one();
        return r;
    }
    std::lock_guard<std::mutex> lk(ctx->mu);
    int worst = 0;
    for (uint32_t done = 0; done < nblocks; done += kHostBatchBlocks) {
        const uint32_t nb = std::min(kHostBatchBlocks, nblocks - done);
        int r = compress_blocks_on_lane(ctx, ctx->lanes[0], src + done, slen + done, dst + done, dlen + done,
                                        status ? status + done : nullptr, nb, level);
        if (r < 0) return r;
        if (r) worst = r;
    }
    return worst;
}

/* ------------------------------------------------------------------------------------------------ */
/* inflate                                                                                          */

namespace {

uint32_t rd16(const uint8_t *p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
uint32_t rd32(const uint8_t *p) { return rd16(p) | (rd16(p + 2) << 16); }

/* The member header parser of the applet's decompress loop (applet/7bgzf.c:81-131), all its flavours: BGZF
 * ("BC", BSIZE), MiGz ("MZ", compressed size), mgzip v1/v2 ("IG"), jerodsanto's mgzip; optional name / comment /
 * header-CRC fields are skipped.  Returns the header length (offset of the DEFLATE data) and the whole member size,
 * or 0 if `p` does not start such a member or the member is cut short by `avail`. */
uint32_t member_parse(const uint8_t *p, size_t avail, uint64_t *member_bytes)
{
    if (avail < 4 || p[0] != 0x1f || p[1] != 0x8b) return 0;
    const uint32_t flags = p[3];
    if (p[2] != 8 || (flags & 0xE0u)) return 0;
    size_t n = 10, xoff = 12, xlen = 0;
    if (flags & 0x04u) {
        if (avail < n + 2) return 0;
        xlen = rd16(p + n);
        n += 2;
        xoff = n;
        if (avail < n + xlen) return 0;
        n += xlen;
    }
    if (flags & 0x08u) while (n < avail && p[n++]) {}
    if (flags & 0x10u) while (n < avail && p[n++]) {}
    if (flags & 0x02u) {
        if (n + 2 > avail) return 0;
        n += 2;
    }
    const uint8_t *x = p + xoff;
    uint64_t sz;
    if (xlen == 6 && !memcmp(x, "BC\x02\x00", 4)) sz = (uint64_t)rd16(x + 4) + 1;
    else if (xlen == 8 && !memcmp(x, "MZ\x04\x00", 4)) sz = (uint64_t)rd32(x + 4) + n + 8;
    else if (xlen == 20 && !memcmp(x, "IG\x10\x00", 4)) sz = rd32(x + 4);   /* (64-bit field; the reference keeps its low half: `int`) */
    else if (xlen == 8 && !memcmp(x, "IG\x04\x00", 4)) sz = rd32(x + 4);
    else if (xlen == 4 && x[3] == 0x7d) sz = rd32(x) & 0xffffffu;
    else return 0;
    if (sz < n + 8 || sz > avail || sz > 0xffffffffull || n > 0xffff) return 0;
    *member_bytes = sz;
    return (uint32_t)n;
}

int inflate_status_to_code(uint32_t st) { return st == 0 ? B200BGZF_OK : B200BGZF_E_FORMAT; }

}  // namespace

extern "C" uint32_t b200bgzf_member_header(const void *p, size_t avail, uint64_t *member_bytes)
{
    uint64_t sz = 0;
    const uint32_t n = p ? member_parse((const uint8_t *)p, avail, &sz) : 0;
    if (member_bytes) *member_bytes = n ? sz : 0;
    return n;
}

extern "C" int b200bgzf_inflate_size_host(const void *in, size_t in_bytes, size_t *out_bytes, size_t *nmembers)
{
    if (!in && in_bytes) return B200BGZF_E_ARG;
    const uint8_t *p = (const uint8_t *)in;
    size_t off = 0, total = 0, n = 0;
    while (off < in_bytes) {
        uint64_t sz = 0;
        if (!member_parse(p + off, in_bytes - off, &sz)) return B200BGZF_E_FORMAT;
        total += rd32(p + off + sz - 4);
        off += (size_t)sz;
        n++;
    }
    if (out_bytes) *out_bytes = total;
    if (nmembers) *nmembers = n;
    return B200BGZF_OK;
}

namespace {
/* the member index of a device-resident BGZF stream (ctx->d_idx_*): member count and decoded size to the host */
int device_index(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, cudaStream_t stream, uint64_t *nmembers, uint64_t *total)
{
    const size_t tiles = bgzf_index_tiles(in_bytes);
    if (!ctx->h_idx) CK(cudaMallocHost((void **)&ctx->h_idx, 8 * sizeof(uint64_t)));
    if (!ctx->d_idx_counts) {
        CK(cudaMalloc((void **)&ctx->d_idx_counts, 4 * sizeof(uint64_t)));
        CK(cudaMalloc((void **)&ctx->d_idx_status, 4 * sizeof(uint32_t)));
    }
    if (tiles > ctx->idx_tiles) {
        cudaFree(ctx->d_idx_tilecount); cudaFree(ctx->d_idx_tileoff);
        CK(cudaMalloc((void **)&ctx->d_idx_tilecount, tiles * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&ctx->d_idx_tileoff, tiles * sizeof(uint64_t)));
        ctx->idx_tiles = tiles;
    }
    /* first guess: signature hits average >= 1 KiB apart; retry with the 28-byte worst case if there are more */
    size_t guess = in_bytes / 1024 + 4096;
    for (int attempt = 0; attempt < 2; attempt++) {
        if (guess > ctx->idx_cap) {
            cudaFree(ctx->d_idx_inoff); cudaFree(ctx->d_idx_outoff); cudaFree(ctx->d_idx_isize); cudaFree(ctx->d_inf_status);
            cudaFree(ctx->d_idx_cand); cudaFree(ctx->d_idx_pick); cudaFree(ctx->d_idx_jump); cudaFree(ctx->d_idx_jump2); cudaFree(ctx->d_idx_reach);
            ctx->d_idx_inoff = ctx->d_idx_outoff = ctx->d_idx_cand = ctx->d_idx_pick = nullptr;
            ctx->d_idx_isize = ctx->d_inf_status = ctx->d_idx_jump = ctx->d_idx_jump2 = ctx->d_idx_reach = nullptr;
            ctx->idx_cap = 0;
            CK(cudaMalloc((void **)&ctx->d_idx_inoff, guess * sizeof(uint64_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_outoff, guess * sizeof(uint64_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_cand, guess * sizeof(uint64_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_pick, guess * sizeof(uint64_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_isize, guess * sizeof(uint32_t)));
            CK(cudaMalloc((void **)&ctx->d_inf_status, guess * sizeof(uint32_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_jump, (guess + 2) * sizeof(uint32_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_jump2, (guess + 2) * sizeof(uint32_t)));
            CK(cudaMalloc((void **)&ctx->d_idx_reach, (guess + 2) * sizeof(uint32_t)));
            ctx->idx_cap = guess;
        }
        CK(cudaMemsetAsync(ctx->d_idx_status, 0, 4 * sizeof(uint32_t), stream));
        BgzfIndexWork w;
        w.max_blocks = (uint32_t)std::min<size_t>(ctx->idx_cap, 0xfffffff0u);
        w.tile_count = ctx->d_idx_tilecount; w.tile_off = ctx->d_idx_tileoff; w.cand_off = ctx->d_idx_cand;
        w.jump = ctx->d_idx_jump; w.jump2 = ctx->d_idx_jump2; w.reach = ctx->d_idx_reach; w.pick_idx = ctx->d_idx_pick;
        w.in_off = ctx->d_idx_inoff; w.out_off = ctx->d_idx_outoff; w.isize = ctx->d_idx_isize;
        w.ncand = ctx->d_idx_counts + 2; w.nmembers = ctx->d_idx_counts; w.out_bytes = ctx->d_idx_counts + 1;
        w.status = ctx->d_idx_status;
        CK(bgzf_launch_index((const uint8_t *)d_in, in_bytes, &w, stream));
        ctx->launches += BGZF_INDEX_LAUNCHES;
        CK(cudaMemcpyAsync(ctx->h_idx, ctx->d_idx_counts, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaMemcpyAsync(ctx->h_idx + 2, ctx->d_idx_status, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        const uint32_t st = (uint32_t)ctx->h_idx[2];
        if ((st & 2u) && attempt == 0) { guess = in_bytes / 28 + 1; continue; }
        if (st) return B200BGZF_E_FORMAT;
        break;
    }
    if ((uint32_t)ctx->h_idx[2]) return B200BGZF_E_FORMAT;
    *nmembers = ctx->h_idx[0];
    *total = ctx->h_idx[1];
    return B200BGZF_OK;
}
}  // namespace

extern "C" int b200bgzf_inflate_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, void *d_out, size_t out_cap,
                                       size_t *out_bytes, unsigned flags, void *stream_)
{
    if (!ctx || !d_in || !out_bytes || in_bytes < 28) return B200BGZF_E_ARG;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    int r = lane_reserve(ctx, l, 1, 0, 0, false);
    if (r) return r;
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : l.stream;
    uint64_t nm = 0, total = 0;
    if ((r = device_index(ctx, d_in, in_bytes, stream, &nm, &total))) return r;
    *out_bytes = (size_t)total;
    if (total > out_cap || (!d_out && total)) return B200BGZF_E_NOSPACE;
    BgzfInflateArgs a;
    memset(&a, 0, sizeof a);
    a.in = (const uint8_t *)d_in;
    a.in_off = ctx->d_idx_inoff;
    a.out_off = ctx->d_idx_outoff;
    a.nblocks = (uint32_t)nm;
    a.out = (uint8_t *)d_out;
    a.status = ctx->d_inf_status;
    a.err_flag = ctx->d_idx_status + 1;
    a.crctab = ctx->d_crctab;
    a.crcpow = ctx->d_crcpow;
    a.verify_crc = (flags & B200BGZF_VERIFY) ? 1 : 0;
    CK(bgzf_launch_inflate(&a, stream));
    ctx->launches += 1 + a.verify_crc;
    CK(cudaMemcpyAsync(ctx->h_idx + 3, ctx->d_idx_status + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    const uint32_t ef = (uint32_t)ctx->h_idx[3];
    return (ef & 1u) ? B200BGZF_E_FORMAT : (ef & 2u) ? B200BGZF_E_CRC : B200BGZF_OK;
}

namespace {
/* units == nullptr: the members are found by walking their headers; else: the caller's list (members and raw pieces) */
int inflate_host_impl(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, const b200bgzf_unit *units, size_t nunits, void *out,
                      size_t out_cap, size_t *out_bytes, unsigned flags, uint32_t *unit_crc = nullptr)
{
    if (!ctx || !in || !out_bytes) return B200BGZF_E_ARG;
    const uint8_t *p = (const uint8_t *)in;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    PendingGuard pg(ctx->lanes, kLanes);
    /* Batches of members rotate through the lanes (H2D, kernel, D2H on the lane's stream).  The host walk of the
     * member headers (applet/7bgzf.c:306-330) is done batch by batch, between submissions, so the GPU starts on the
     * first members while the host is still finding the later ones; the first batches are small so that the D2H
     * copies — the longest leg — start early, then kInflateBatch members each over kInflateLanes lanes. */
    static const size_t xp_batch = [] { const char *e = getenv("B200BGZF_INF_BATCH"); return e && atoi(e) > 0 ? (size_t)atoi(e) : kInflateBatch; }();
    static const int xp_lanes = [] { const char *e = getenv("B200BGZF_INF_LANES"); return e && atoi(e) > 0 ? std::min(atoi(e), kLanes) : kInflateLanes; }();
    static const size_t xp_first = [] { const char *e = getenv("B200BGZF_INF_FIRST"); return e && atoi(e) > 0 ? (size_t)atoi(e) : (size_t)256; }();
    const size_t kBatchMax = xp_batch;
    const int nlanes = xp_lanes;
    size_t batch = kBatchMax < xp_first ? kBatchMax : xp_first;
    int r;
    bool bad = false, badcrc = false;
    size_t off = 0, total = 0, i = 0;
    *out_bytes = 0;
    auto complete = [&](Lane &l) -> int {
        CK(cudaStreamSynchronize(l.stream));
        if (l.h_total[1] & 1u) bad = true;
        if (l.h_total[1] & 2u) badcrc = true;
        if (unit_crc) memcpy(unit_crc + l.pend_first, (const uint32_t *)(l.h_meta + 2 * kBatchMax) + 3 * kBatchMax, l.pend_nb * sizeof(uint32_t));
        l.pending = false;
        return 0;
    };
    auto drain = [&]() -> int {
        for (auto &l : ctx->lanes)
            if (l.pending && (r = complete(l))) return r;
        return 0;
    };
    size_t u = 0;                                       /* next unit of the caller's list */
    while (units ? u < nunits : off < in_bytes) {
        Lane &l = ctx->lanes[i % nlanes];
        if (l.pending && (r = complete(l))) return r;
        if ((r = lane_reserve(ctx, l, (uint32_t)kBatchMax, 0, 0, false))) return r;
        CK(grow(&l.h_meta, &l.meta_cap, 4 * kBatchMax, true));
        uint32_t *h_hdr = (uint32_t *)(l.h_meta + 2 * kBatchMax), *h_msz = h_hdr + kBatchMax, *h_isz = h_msz + kBatchMax;
        /* walk the next `batch` members */
        size_t in0 = off;
        const size_t out0 = total;
        size_t nb = 0;
        const size_t u0 = u;
        if (units) {
            in0 = off = (size_t)units[u].in_off;
            while (nb < batch && u < nunits) {
                const b200bgzf_unit &un = units[u];
                /* ascending, inside the input, and a member has room for its trailer */
                if (un.in_off < off || un.in_off + un.in_len > in_bytes || un.hdr_len > un.in_len || (!un.piece && un.in_len < un.hdr_len + 8u) ||
                    un.in_len == 0 || un.hdr_len > 0xffffu) { drain(); return B200BGZF_E_FORMAT; }
                l.h_meta[nb] = un.in_off - in0;
                l.h_meta[kBatchMax + nb] = total - out0;
                h_hdr[nb] = un.hdr_len;
                h_msz[nb] = un.in_len;
                h_isz[nb] = un.piece ? un.out_len : 0xffffffffu;
                const uint32_t unit_out = un.piece ? un.out_len : rd32(p + un.in_off + un.in_len - 4);
                /* (the kernel's positions are 32-bit; DEFLATE cannot expand its input more than 1032 times) */
                if (unit_out > 0x7fffffffu || unit_out > 1032ull * (un.in_len - un.hdr_len) + 1032u) { drain(); return B200BGZF_E_FORMAT; }
                total += unit_out;
                off = (size_t)(un.in_off + un.in_len);
                nb++;
                u++;
            }
        }
        while (!units && nb < batch && off < in_bytes) {
            uint64_t sz = 0;
            const uint32_t hlen = member_parse(p + off, in_bytes - off, &sz);
            if (!hlen) { drain(); return B200BGZF_E_FORMAT; }
            l.h_meta[nb] = off - in0;
            l.h_meta[kBatchMax + nb] = total - out0;
            h_hdr[nb] = hlen;
            h_msz[nb] = (uint32_t)sz;
            const uint32_t isz = rd32(p + off + sz - 4);   /* ISIZE: the member's share of the output */
            if (isz > 1032ull * (sz - hlen) + 1032u) { drain(); return B200BGZF_E_FORMAT; }   /* (more than DEFLATE can expand its input) */
            total += isz;
            off += (size_t)sz;
            nb++;
        }
        *out_bytes = total;
        if (total > out_cap || (!out && total)) { drain(); return B200BGZF_E_NOSPACE; }
        const size_t cbytes = off - in0, obytes = total - out0;
        if ((r = lane_reserve(ctx, l, (uint32_t)kBatchMax, cbytes + 256, obytes + 256, false))) return r;
        CK(cudaMemcpyAsync(l.d_in, p + in0, cbytes, cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_inoff, l.h_meta, nb * sizeof(uint64_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_outoff, l.h_meta + kBatchMax, nb * sizeof(uint64_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_inlen, h_hdr, nb * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_len, h_msz, nb * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream));
        if (units) CK(cudaMemcpyAsync(l.d_off, h_isz, nb * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream));   /* (d_off: unused by inflate batches) */
        CK(cudaMemsetAsync(l.d_total, 0, 4 * sizeof(uint64_t), l.stream));
        BgzfInflateArgs a;
        memset(&a, 0, sizeof a);
        a.unit_isize = units ? (const uint32_t *)l.d_off : nullptr;
        a.in = l.d_in;
        a.in_off = l.d_inoff;
        a.out_off = l.d_outoff;
        a.hdr_len = l.d_inlen;                          /* headers were parsed here: any flavour the applet's loop accepts */
        a.msize = l.d_len;
        a.nblocks = (uint32_t)nb;
        a.out = l.d_out;
        a.status = l.d_status;
        a.err_flag = (uint32_t *)(l.d_total + 1);
        a.crctab = ctx->d_crctab;
        a.crcpow = ctx->d_crcpow;
        a.verify_crc = ((flags & B200BGZF_VERIFY) || unit_crc) ? 1 : 0;
        if (unit_crc) a.unit_crc = (uint32_t *)l.d_off + kBatchMax;       /* (second half of the u64 array whose first half holds unit_isize) */
        CK(bgzf_launch_inflate(&a, l.stream));
        ctx->launches += 1 + a.verify_crc;
        if (unit_crc) {
            CK(cudaMemcpyAsync((uint32_t *)(l.h_meta + 2 * kBatchMax) + 3 * kBatchMax, a.unit_crc, nb * sizeof(uint32_t), cudaMemcpyDeviceToHost, l.stream));
            l.pend_first = u0;
            l.pend_nb = (uint32_t)nb;
        }
        if (obytes) CK(cudaMemcpyAsync((uint8_t *)out + out0, l.d_out, obytes, cudaMemcpyDeviceToHost, l.stream));
        CK(cudaMemcpyAsync(l.h_total, l.d_total, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, l.stream));
        l.pending = true;
        i++;
        batch = batch * 2 < kBatchMax ? batch * 2 : kBatchMax;
    }
    if ((r = drain())) return r;
    return bad ? B200BGZF_E_FORMAT : badcrc ? B200BGZF_E_CRC : B200BGZF_OK;
}
}  // namespace

extern "C" int b200bgzf_inflate_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, void *out, size_t out_cap, size_t *out_bytes,
                                     unsigned flags)
{
    return inflate_host_impl(ctx, in, in_bytes, nullptr, 0, out, out_cap, out_bytes, flags);
}

extern "C" int b200bgzf_inflate_units_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, const b200bgzf_unit *units, size_t nunits,
                                           void *out, size_t out_cap, size_t *out_bytes, unsigned flags, uint32_t *unit_crc)
{
    if (!units && nunits) return B200BGZF_E_ARG;
    if (nunits == 0) {
        if (out_bytes) *out_bytes = 0;
        return out_bytes ? B200BGZF_OK : B200BGZF_E_ARG;
    }
    return inflate_host_impl(ctx, in, in_bytes, units, nunits, out, out_cap, out_bytes, flags, unit_crc);
}

/* ------------------------------------------------------------------------------------------------ */
/* whole-stream gzip: one member, inflated in parallel between its byte-aligned flush points (bgzf_gzip.cu)               */

namespace {

/* Scratch (2 bytes per output byte of the chunks in flight) stays under this; B200BGZF_GZIP_BUDGET (bytes, at least 1 MiB)
 * lowers it, so that the multi-batch path can be exercised on small inputs. */
uint64_t gzip_budget()
{
    static const uint64_t b = [] {
        const char *e = getenv("B200BGZF_GZIP_BUDGET");
        const unsigned long long v = e && *e ? strtoull(e, nullptr, 10) : 0ull;
        return v >= (1ull << 20) && v < (1ull << 30) ? (uint64_t)v : (uint64_t)1 << 30;
    }();
    return b;
}

constexpr uint64_t kGzMaxChunkIn = 4ull << 20;   /* compressed bytes one chunk may span: bounds a false candidate's garbage decode */
constexpr uint32_t kGzCrcPiece = 1u << 20;       /* B200BGZF_VERIFY: output bytes per CRC unit of bgzf_verify_kernel */

/* Decodes the member d_in[0, in_bytes) (header of hlen bytes, trailer isize / want_crc) into d_out through its flush-point chain.
 * Returns BGZF_GZIP_FALLBACK when the member has no complete chain (no flush point, a chunk over the caps, a chain that ends
 * anywhere but at the trailer, a decode that differs from the boundary pass): the one-warp path then gives the outcome.
 * on_batch(base, bytes) is called after the launches that write output [base, base + bytes). */
/* the chain the index builder keeps: the chunk arrays of BgzfGzipArgs (c_start, c_off, c_len), valid until the next gzip call */
struct GzChain {
    BgzfGzipArgs a;
    uint64_t nchunks;
};

template <typename F>
int gzip_batches(b200bgzf_ctx *ctx, BgzfGzipArgs a, uint64_t nchunks, uint64_t total, uint32_t want_crc, unsigned flags,
                 cudaStream_t stream, F on_batch, const uint64_t *bit_end);

template <typename F>
int gzip_chain_inflate(b200bgzf_ctx *ctx, const uint8_t *d_in, size_t in_bytes, uint32_t hlen, uint32_t isize, uint32_t want_crc,
                       uint8_t *d_out, size_t out_cap, size_t *total_out, unsigned flags, cudaStream_t stream, F on_batch,
                       GzChain *keep = nullptr)
{
    GzWork &z = ctx->gz;
    const uint64_t data_len = in_bytes - hlen - 8;
    if (data_len == 0) return BGZF_GZIP_FALLBACK;
    const size_t tiles = bgzf_gzip_tiles(data_len);
    CK(grow(&z.tile_count, &z.tiles_cap, tiles));
    CK(grow(&z.tile_off, &z.tileoff_cap, tiles));
    size_t c64 = z.small64 ? 8 : 0, c32 = z.small32 ? 8 : 0, hc = z.h_cap;
    CK(grow(&z.small64, &c64, 8));
    CK(grow(&z.small32, &c32, 8));
    CK(grow(&z.h, &hc, 8, true));
    z.h_cap = hc;
    BgzfGzipArgs a;
    memset(&a, 0, sizeof a);
    a.data = d_in + hlen;
    a.data_len = data_len;
    a.max_in = kGzMaxChunkIn;
    a.tile_count = z.tile_count;
    a.tile_off = z.tile_off;
    a.counts = z.small64;
    a.ncand = z.small64 + 1;
    a.nchunks = z.small64 + 2;
    a.total = z.small64 + 3;
    a.chain_status = z.small32;
    a.err = z.small32 + 1;
    a.out = d_out;
    CK(cudaMemsetAsync(z.small64, 0, 8 * sizeof(uint64_t), stream));
    CK(cudaMemsetAsync(z.small32, 0, 8 * sizeof(uint32_t), stream));
    /* 1. flush points: count, then size the candidate arrays by it */
    CK(bgzf_launch_gzip_count(&a, stream));
    ctx->launches += 3;
    CK(cudaMemcpyAsync(z.h, z.small64, sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    const uint64_t nc = z.h[0] + 1;
    /* (the index builder takes a member without flush points as one chunk when its data is within the chunk cap) */
    if ((nc < 2 && !(keep && data_len <= kGzMaxChunkIn)) || nc > 0xfffffff0ull) return BGZF_GZIP_FALLBACK;
    /* u64: cand, end, pick, c_start, c_off; u32: olen, status, c_len, lastm, anchor, jump, jump2, reach */
    CK(grow(&z.u64, &z.u64_cap, 5 * nc));
    CK(grow(&z.u32, &z.u32_cap, 8 * (nc + 2)));
    a.cand = z.u64; a.end = z.u64 + nc; a.pick = z.u64 + 2 * nc; a.c_start = z.u64 + 3 * nc; a.c_off = z.u64 + 4 * nc;
    uint32_t *q = z.u32;
    a.olen = q; a.status = q + nc; a.c_len = q + 2 * nc; a.lastm = q + 3 * nc; a.anchor = q + 4 * nc;
    a.jump = q + 5 * nc; a.jump2 = q + 6 * nc + 2; a.reach = q + 7 * nc + 4;
    /* 2. boundary pass, chain from the data start, chunk offsets */
    CK(bgzf_launch_gzip_chain(&a, (uint32_t)nc, stream));
    ctx->launches += BGZF_GZIP_CHAIN_LAUNCHES;
    CK(cudaMemcpyAsync(z.h, z.small64, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaMemcpyAsync(z.h + 4, z.small32, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if ((uint32_t)z.h[4] & 1u) return BGZF_GZIP_FALLBACK;
    const uint64_t nchunks = z.h[2], total = z.h[3];
    if (nchunks == 0 || nchunks > nc) return BGZF_GZIP_FALLBACK;
    /* the chain is the sequential decoder's exact bit path: its length is what that decoder would produce */
    *total_out = (size_t)total;
    if ((uint32_t)total != isize) return B200BGZF_E_FORMAT;
    if (total > out_cap || (!d_out && total)) return B200BGZF_E_NOSPACE;
    if (keep) *keep = { a, nchunks };
    return gzip_batches(ctx, a, nchunks, total, want_crc, flags, stream, on_batch, nullptr);
}

/* Steps 3 and 4 of both parallel routes: the chained chunks of `a` (c_start, c_len, c_off; nchunks of them, total bytes) are
 * decoded in batches under the scratch budget, then checked (B200BGZF_VERIFY).  bit_end: NULL for flush-point chunks, else
 * the searched route's chunk ends (c_start in bits). */
template <typename F>
int gzip_batches(b200bgzf_ctx *ctx, BgzfGzipArgs a, uint64_t nchunks, uint64_t total, uint32_t want_crc, unsigned flags,
                 cudaStream_t stream, F on_batch, const uint64_t *bit_end)
{
    GzWork &z = ctx->gz;
    /* 3. batches of chained chunks whose scratch fits the budget */
    const uint64_t win = bgzf_gzip_window(), budget = gzip_budget();
    std::vector<uint64_t> cut;                      /* batch boundaries (chunk indices) */
    if (2 * (win + total) <= budget) {
        cut = { 0, nchunks };
    } else {
        std::vector<uint64_t> off(nchunks + 1);
        CK(cudaMemcpyAsync(off.data(), a.c_off, nchunks * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        off[nchunks] = total;
        cut.push_back(0);
        uint64_t j = 0;
        while (j < nchunks) {
            uint64_t j1 = j + 1;
            if (2 * (win + off[j1] - off[j]) > budget) return BGZF_GZIP_FALLBACK;   /* one chunk alone is over the budget */
            while (j1 < nchunks && 2 * (win + off[j1 + 1] - off[j]) <= budget) j1++;
            cut.push_back(j1);
            j = j1;
        }
    }
    uint64_t most = 0;
    std::vector<uint64_t> base(cut.size());
    {
        std::vector<uint64_t> off0(cut.size());
        for (size_t i = 0; i < cut.size(); i++) {
            if (cut[i] == nchunks) { off0[i] = total; continue; }
            CK(cudaMemcpyAsync(&off0[i], a.c_off + cut[i], sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        }
        CK(cudaStreamSynchronize(stream));
        for (size_t i = 0; i + 1 < cut.size(); i++) most = std::max(most, off0[i + 1] - off0[i]);
        base = off0;
    }
    CK(grow(&z.scratch, &z.scratch_cap, win + most + 16));
    a.scratch = z.scratch;
    for (size_t i = 0; i + 1 < cut.size(); i++) {
        CK(bgzf_launch_gzip_batch(&a, (uint32_t)cut[i], (uint32_t)cut[i + 1], base[i], base[i + 1] - base[i], bit_end, stream));
        ctx->launches += BGZF_GZIP_BATCH_LAUNCHES;
        if (int r = on_batch(base[i], base[i + 1] - base[i])) return r;
    }
    /* 4. B200BGZF_VERIFY: CRC-32 of 1 MiB units of the output (bgzf_verify_kernel's tiles), combined here */
    const bool verify = (flags & B200BGZF_VERIFY) != 0;
    const uint64_t nu = verify ? (total + kGzCrcPiece - 1) / kGzCrcPiece : 0;
    std::vector<uint32_t> hcrc(nu);
    if (nu) {
        /* u64: in_off (0), out_off; u32: hdr_len (0), msize (0), unit_isize, status (0), unit_crc */
        size_t un64 = 0, un32 = 0;
        uint64_t *d64 = nullptr;
        uint32_t *d32 = nullptr;
        CK(grow(&d64, &un64, 2 * nu));
        if (cudaError_t e = grow(&d32, &un32, 5 * nu)) { cudaFree(d64); return fail(ctx, e, "grow"); }
        std::vector<uint64_t> h64(2 * nu, 0);
        std::vector<uint32_t> h32(5 * nu, 0);
        for (uint64_t u = 0; u < nu; u++) {
            h64[nu + u] = u * kGzCrcPiece;
            h32[2 * nu + u] = (uint32_t)std::min<uint64_t>(kGzCrcPiece, total - u * kGzCrcPiece);
        }
        cudaError_t e = cudaMemcpyAsync(d64, h64.data(), h64.size() * 8, cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d32, h32.data(), h32.size() * 4, cudaMemcpyHostToDevice, stream);
        BgzfInflateArgs v;
        memset(&v, 0, sizeof v);
        v.in = a.out;
        v.in_off = d64;
        v.out_off = d64 + nu;
        v.hdr_len = d32;
        v.msize = d32 + nu;
        v.unit_isize = d32 + 2 * nu;
        v.status = d32 + 3 * nu;
        v.unit_crc = d32 + 4 * nu;
        v.nblocks = (uint32_t)nu;
        v.out = a.out;
        v.err_flag = a.err + 2;
        v.verify_crc = 1;
        v.crctab = ctx->d_crctab;
        v.crcpow = ctx->d_crcpow;
        if (e == cudaSuccess) e = bgzf_launch_verify(&v, stream);
        ctx->launches += 1;
        if (e == cudaSuccess) e = cudaMemcpyAsync(hcrc.data(), v.unit_crc, nu * 4, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        cudaFree(d64);
        cudaFree(d32);
        if (e != cudaSuccess) return fail(ctx, e, "gzip verify");
    }
    CK(cudaMemcpyAsync(z.h + 5, a.err, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if ((uint32_t)z.h[5]) return BGZF_GZIP_FALLBACK;    /* (a back-reference before the member start: the one-warp path reports it) */
    if (verify) {
        uint32_t crc = 0;
        for (uint64_t u = 0; u < nu; u++) crc = u ? b200bgzf_crc32_combine(crc, hcrc[u], std::min<uint64_t>(kGzCrcPiece, total - u * kGzCrcPiece)) : hcrc[u];
        if (crc != want_crc) return B200BGZF_E_CRC;
    }
    return B200BGZF_OK;
}

constexpr int kGzRepairRounds = 8;   /* searched route: chain repairs before the member goes to one warp */

/* The searched route (DESIGN §6g), for a member whose flush-point chain is unusable: chunk starts at bit offsets proposed by
 * gz_search_kernel (one per region after the first), a boundary pass from each up to the next proposal, and a chain walk
 * here from the data start.  A chunk on the walk ends at a true block boundary; when that end is no candidate, it becomes
 * one, and the boundary pass runs again on the new candidates only.  The chained chunks are the sequential decoder's exact
 * bit path, decoded by gzip_batches.  Returns BGZF_GZIP_FALLBACK for a member within one region, a chain that breaks (a
 * failed chunk: an error, a reference before the member start, over the caps) or does not end 8 bytes before the input end,
 * or more than kGzRepairRounds repairs: the one-warp path then gives the outcome. */
template <typename F>
int gzip_search_inflate(b200bgzf_ctx *ctx, const uint8_t *d_in, size_t in_bytes, uint32_t hlen, uint32_t isize, uint32_t want_crc,
                        uint8_t *d_out, size_t out_cap, size_t *total_out, unsigned flags, cudaStream_t stream, F on_batch)
{
    GzWork &z = ctx->gz;
    const uint64_t data_len = in_bytes - hlen - 8, region = bgzf_gzip_region();
    const uint64_t nreg = (data_len + region - 1) / region;
    if (nreg < 2) return BGZF_GZIP_FALLBACK;
    size_t c32 = z.small32 ? 8 : 0, hc = z.h_cap;
    CK(grow(&z.small32, &c32, 8));
    CK(grow(&z.h, &hc, 8, true));
    z.h_cap = hc;
    CK(cudaMemsetAsync(z.small32, 0, 8 * sizeof(uint32_t), stream));
    BgzfGzipArgs a;
    memset(&a, 0, sizeof a);
    a.data = d_in + hlen;
    a.data_len = data_len;
    a.max_in = kGzMaxChunkIn;
    a.err = z.small32 + 1;
    a.out = d_out;
    /* 1. candidates (bit offsets, ascending): the data start, then what the search proposes */
    std::vector<uint64_t> cand{ 0 };
    {
        CK(grow(&z.u64, &z.u64_cap, nreg));
        CK(bgzf_launch_gzip_search(&a, (uint32_t)nreg, z.u64, stream));
        ctx->launches += 1;
        std::vector<uint64_t> found(nreg - 1);
        CK(cudaMemcpyAsync(found.data(), z.u64, found.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        for (uint64_t f : found)
            if (f != ~0ull) cand.push_back(f);
    }
    /* 2. rounds of the boundary pass over the new candidates and the walk from the data start */
    struct Bound {
        uint64_t end;
        uint32_t olen, status;
    };
    std::map<uint64_t, Bound> bound;              /* every candidate's chunk, by its start */
    std::vector<uint64_t> todo = cand, chain;
    for (int round = 0;; round++) {
        const size_t n = todo.size();
        CK(grow(&z.u64, &z.u64_cap, 3 * n));
        CK(grow(&z.u32, &z.u32_cap, 2 * n));
        std::vector<uint64_t> h64(2 * n);         /* start, stop (the next candidate; none: decode up to the final block) */
        for (size_t k = 0; k < n; k++) {
            const auto next = std::upper_bound(cand.begin(), cand.end(), todo[k]);
            h64[k] = todo[k];
            h64[n + k] = next == cand.end() ? ~0ull : *next;
        }
        a.cand = z.u64;
        a.end = z.u64 + 2 * n;
        a.olen = z.u32;
        a.status = z.u32 + n;
        CK(cudaMemcpyAsync(z.u64, h64.data(), h64.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
        CK(bgzf_launch_gzip_bit_bound(&a, z.u64 + n, (uint32_t)n, stream));
        ctx->launches += 1;
        std::vector<uint64_t> end(n);
        std::vector<uint32_t> h32(2 * n);
        CK(cudaMemcpyAsync(end.data(), a.end, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaMemcpyAsync(h32.data(), a.olen, 2 * n * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        for (size_t k = 0; k < n; k++) bound[todo[k]] = { end[k], h32[k], h32[n + k] };
        chain.clear();
        bool done = false;
        for (uint64_t at = 0;;) {
            const Bound &c = bound.at(at);
            if (c.status == GZ_FAIL) return BGZF_GZIP_FALLBACK;
            chain.push_back(at);
            if (c.status == GZ_END_FINAL) {
                if ((c.end + 7) / 8 != data_len) return BGZF_GZIP_FALLBACK;
                done = true;
                break;
            }
            if (!bound.count(c.end)) break;       /* a true block boundary the search did not propose */
            at = c.end;
        }
        if (done) break;
        if (round == kGzRepairRounds) return BGZF_GZIP_FALLBACK;
        /* repair: the unmatched ends of all chunks become candidates (those of chunks from false starts cost a warp each) */
        todo.clear();
        for (const auto &kv : bound)
            if (kv.second.status == GZ_END_FLUSH && !bound.count(kv.second.end)) todo.push_back(kv.second.end);
        std::sort(todo.begin(), todo.end());
        todo.erase(std::unique(todo.begin(), todo.end()), todo.end());
        std::vector<uint64_t> merged(cand.size() + todo.size());
        std::merge(cand.begin(), cand.end(), todo.begin(), todo.end(), merged.begin());
        cand.swap(merged);
    }
    /* 3. the chained chunks: start and end (bits), output offset and length */
    const uint64_t nchunks = chain.size();
    std::vector<uint64_t> h64(3 * nchunks);
    std::vector<uint32_t> h32(nchunks);
    uint64_t total = 0;
    for (uint64_t j = 0; j < nchunks; j++) {
        const Bound &c = bound.at(chain[j]);
        h64[j] = chain[j];
        h64[nchunks + j] = total;
        h64[2 * nchunks + j] = c.end;
        h32[j] = c.olen;
        total += c.olen;
    }
    *total_out = (size_t)total;
    if ((uint32_t)total != isize) return B200BGZF_E_FORMAT;
    if (total > out_cap || (!d_out && total)) return B200BGZF_E_NOSPACE;
    CK(grow(&z.u64, &z.u64_cap, 3 * nchunks));
    CK(grow(&z.u32, &z.u32_cap, 3 * nchunks));
    a.c_start = z.u64;
    a.c_off = z.u64 + nchunks;
    a.c_len = z.u32;
    a.lastm = z.u32 + nchunks;
    a.anchor = z.u32 + 2 * nchunks;
    CK(cudaMemcpyAsync(z.u64, h64.data(), h64.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    CK(cudaMemcpyAsync(z.u32, h32.data(), h32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    return gzip_batches(ctx, a, nchunks, total, want_crc, flags, stream, on_batch, z.u64 + 2 * nchunks);
}

/* the checks the one-warp path makes of a member before decoding it (inflate_host_impl): 0 or B200BGZF_E_FORMAT */
int gzip_member_check(size_t in_bytes, uint32_t hlen, uint32_t isize)
{
    if (!hlen || in_bytes < (size_t)hlen + 10 || in_bytes > 0xffffffffull || hlen > 0xffffu) return B200BGZF_E_FORMAT;
    if (isize > 0x7fffffffu || isize > 1032ull * (in_bytes - hlen) + 1032u) return B200BGZF_E_FORMAT;
    return 0;
}

/* the header (FEXTRA, FNAME, FCOMMENT, FHCRC) of a member in device memory, in small reads that grow while a field runs past
 * what was read (*hlen = 0: not a gzip header); the trailer */
int gzip_device_header(b200bgzf_ctx *ctx, const uint8_t *in, size_t in_bytes, cudaStream_t stream, size_t *hlen, uint8_t tr[8])
{
    std::vector<uint8_t> head;
    size_t xoff, xlen;
    for (size_t want = std::min<size_t>(in_bytes, 4096);; want = std::min(in_bytes, want * 4)) {
        head.resize(want);
        CK(cudaMemcpyAsync(head.data(), in, want, cudaMemcpyDeviceToHost, stream));
        CK(cudaMemcpyAsync(tr, in + in_bytes - 8, 8, cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        *hlen = bgzf_gz_header(head.data(), want, &xoff, &xlen);
        if (*hlen || want == in_bytes || head.size() < 10 || head[0] != 0x1f || head[1] != 0x8b) break;
    }
    return B200BGZF_OK;
}

}  // namespace

extern "C" int b200bgzf_gzip_inflate_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, void *d_out, size_t out_cap,
                                            size_t *out_bytes, unsigned flags, void *stream_)
{
    if (!ctx || !d_in || !out_bytes) return B200BGZF_E_ARG;
    *out_bytes = 0;
    if (in_bytes < 18) return B200BGZF_E_FORMAT;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    int r = lane_reserve(ctx, l, 1, 0, 0, false);
    if (r) return r;
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : l.stream;
    GzWork &z = ctx->gz;
    const uint8_t *in = (const uint8_t *)d_in;
    uint8_t tr[8];
    size_t hlen = 0;
    if ((r = gzip_device_header(ctx, in, in_bytes, stream, &hlen, tr))) return r;
    const uint32_t want_crc = rd32(tr), isize = rd32(tr + 4);
    if ((r = gzip_member_check(in_bytes, (uint32_t)hlen, isize))) return r;
    size_t total = isize;
    bool batched = false;                   /* (a fallback after the flush-point route decoded a batch goes to one warp) */
    const auto on_batch = [&](uint64_t, uint64_t) { batched = true; return 0; };
    r = gzip_chain_inflate(ctx, in, in_bytes, (uint32_t)hlen, isize, want_crc, (uint8_t *)d_out, d_out ? out_cap : 0, &total, flags, stream,
                           on_batch);
    *out_bytes = total;
    if (r != BGZF_GZIP_FALLBACK) return r;
    *out_bytes = isize;
    if (isize > out_cap || (!d_out && isize)) return B200BGZF_E_NOSPACE;
    /* no usable flush points: chunks from a search for block headers, else one warp, as b200bgzf_inflate_units_host decodes */
    if (!batched) {
        total = isize;
        r = gzip_search_inflate(ctx, in, in_bytes, (uint32_t)hlen, isize, want_crc, (uint8_t *)d_out, out_cap, &total, flags, stream,
                                on_batch);
        *out_bytes = total;
        if (r != BGZF_GZIP_FALLBACK) return r;
        *out_bytes = isize;
    }
    size_t c64 = z.small64 ? 8 : 0, c32 = z.small32 ? 8 : 0, hc = z.h_cap;
    CK(grow(&z.small64, &c64, 8));
    CK(grow(&z.small32, &c32, 8));
    CK(grow(&z.h, &hc, 8, true));
    z.h_cap = hc;
    uint32_t *h32 = (uint32_t *)z.h;
    z.h[0] = 0;                                          /* in_off, out_off */
    z.h[1] = 0;
    h32[4] = (uint32_t)hlen;                             /* hdr_len, msize, status, err_flag */
    h32[5] = (uint32_t)in_bytes;
    h32[6] = 0;
    h32[7] = 0;
    CK(cudaMemcpyAsync(z.small64, z.h, 2 * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    CK(cudaMemcpyAsync(z.small32, h32 + 4, 4 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    BgzfInflateArgs a;
    memset(&a, 0, sizeof a);
    a.in = in;
    a.in_off = z.small64;
    a.out_off = z.small64 + 1;
    a.hdr_len = z.small32;
    a.msize = z.small32 + 1;
    a.status = z.small32 + 2;
    a.err_flag = z.small32 + 3;
    a.nblocks = 1;
    a.out = (uint8_t *)d_out;
    a.crctab = ctx->d_crctab;
    a.crcpow = ctx->d_crcpow;
    a.verify_crc = (flags & B200BGZF_VERIFY) ? 1 : 0;
    CK(bgzf_launch_inflate(&a, stream));
    ctx->launches += 1 + a.verify_crc;
    CK(cudaMemcpyAsync(z.h + 2, a.err_flag, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    const uint32_t ef = (uint32_t)z.h[2];
    return (ef & 1u) ? B200BGZF_E_FORMAT : (ef & 2u) ? B200BGZF_E_CRC : B200BGZF_OK;
}

/* the GZIP container reader's route (host/containers.c): the member goes to the device, finished batches come back while the
 * next ones decode; BGZF_GZIP_FALLBACK hands the member to the one-warp path */
extern "C" int bgzf_gzip_inflate_host(b200bgzf_ctx *ctx, const void *in_, size_t in_bytes, uint32_t hlen, void *out, size_t out_cap,
                                      size_t *out_bytes, unsigned flags)
{
    const uint8_t *in = (const uint8_t *)in_;
    if (!ctx || !in || !out_bytes || in_bytes < (size_t)hlen + 10) return BGZF_GZIP_FALLBACK;
    const uint32_t want_crc = rd32(in + in_bytes - 8), isize = rd32(in + in_bytes - 4);
    if (gzip_member_check(in_bytes, hlen, isize) || isize > out_cap || (!out && isize)) return BGZF_GZIP_FALLBACK;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    int r = lane_reserve(ctx, l, 1, 0, 0, false);
    if (r) return r;
    GzWork &z = ctx->gz;
    if (!z.copy) CK(cudaStreamCreateWithFlags(&z.copy, cudaStreamNonBlocking));
    if (!z.ev) CK(cudaEventCreateWithFlags(&z.ev, cudaEventDisableTiming));
    CK(grow(&z.d_in, &z.in_cap, in_bytes + 64));
    CK(grow(&z.d_out, &z.out_cap, (size_t)isize + 64));
    CK(cudaMemcpyAsync(z.d_in, in, in_bytes, cudaMemcpyHostToDevice, l.stream));
    size_t total = isize;
    bool batched = false;
    const auto on_batch = [&](uint64_t base, uint64_t bytes) -> int {
        batched = true;
        if (!bytes) return 0;
        CK(cudaEventRecord(z.ev, l.stream));
        CK(cudaStreamWaitEvent(z.copy, z.ev, 0));
        CK(cudaMemcpyAsync((uint8_t *)out + base, z.d_out + base, bytes, cudaMemcpyDeviceToHost, z.copy));
        return 0;
    };
    r = gzip_chain_inflate(ctx, z.d_in, in_bytes, hlen, isize, want_crc, z.d_out, isize, &total, flags, l.stream, on_batch);
    if (r == BGZF_GZIP_FALLBACK && !batched) {
        total = isize;
        r = gzip_search_inflate(ctx, z.d_in, in_bytes, hlen, isize, want_crc, z.d_out, isize, &total, flags, l.stream, on_batch);
    }
    const cudaError_t e = cudaStreamSynchronize(z.copy);
    if (r == B200BGZF_E_NOSPACE) r = B200BGZF_E_FORMAT;   /* (more output than ISIZE: the one-warp path's overrun) */
    if (r == B200BGZF_OK || r == B200BGZF_E_CRC) *out_bytes = isize;
    if (e != cudaSuccess && r != BGZF_GZIP_FALLBACK) return fail(ctx, e, "gzip copy");
    return r;
}

/* ------------------------------------------------------------------------------------------------ */
/* random access                                                                                    */

namespace {

/* Device bytes a range call may hold for decoded members: the device variant's scratch; a host-variant group (decoded
 * members + output) takes a quarter, and a range is cut into pieces of a sixteenth.  B200BGZF_RANGE_BUDGET (bytes, at least
 * 1 MiB) lowers it, so that the multi-pass paths can be exercised on small inputs. */
uint64_t range_budget()
{
    static const uint64_t b = [] {
        const char *e = getenv("B200BGZF_RANGE_BUDGET");
        const unsigned long long v = e && *e ? strtoull(e, nullptr, 10) : 0ull;
        return v >= (1ull << 20) ? (uint64_t)v : (uint64_t)1 << 30;
    }();
    return b;
}

/* largest i in [0, n) with a[i] <= x (a ascending, a[0] <= x) */
size_t last_le(const uint64_t *a, size_t n, uint64_t x) { return (size_t)(std::upper_bound(a, a + n, x) - a) - 1; }

/* every member start (EOF marker included) by a header walk */
int walk_index(const uint8_t *p, size_t in_bytes, std::vector<uint64_t> &c, std::vector<uint64_t> &u)
{
    uint64_t off = 0, pos = 0;
    while (off < in_bytes) {
        uint64_t sz = 0;
        if (!member_parse(p + off, in_bytes - off, &sz)) return B200BGZF_E_FORMAT;
        c.push_back(off);
        u.push_back(pos);
        pos += rd32(p + off + sz - 4);
        off += sz;
    }
    return B200BGZF_OK;
}

}  // namespace

extern "C" int b200bgzf_index_host(const void *in, size_t in_bytes, uint64_t *caddr, uint64_t *uaddr, size_t cap, size_t *nmembers)
{
    if ((!in && in_bytes) || !nmembers || (cap && (!caddr || !uaddr))) return B200BGZF_E_ARG;
    std::vector<uint64_t> c, u;
    const int r = walk_index((const uint8_t *)in, in_bytes, c, u);
    if (r) return r;
    *nmembers = c.size();
    const size_t n = std::min(cap, c.size());
    if (n) { memcpy(caddr, c.data(), n * 8); memcpy(uaddr, u.data(), n * 8); }
    return c.size() > cap ? B200BGZF_E_NOSPACE : B200BGZF_OK;
}

extern "C" int b200bgzf_gzi_parse(const void *gzi, size_t gzi_bytes, uint64_t *caddr, uint64_t *uaddr, size_t cap, size_t *nmembers)
{
    if (!gzi || !nmembers || (cap && (!caddr || !uaddr))) return B200BGZF_E_ARG;
    const uint8_t *p = (const uint8_t *)gzi;
    auto get = [&](size_t at) { uint64_t v = 0; for (int k = 7; k >= 0; k--) v = v << 8 | p[at + k]; return v; };
    if (gzi_bytes < 8) return B200BGZF_E_FORMAT;
    const uint64_t entries = get(0);
    if (entries > (gzi_bytes - 8) / 16 || gzi_bytes != 8 + 16 * entries) return B200BGZF_E_FORMAT;
    uint64_t pc = 0, pu = 0;
    for (uint64_t i = 0; i < entries; i++) {
        const uint64_t c = get(8 + 16 * i), u = get(16 + 16 * i);
        if (c <= pc || u < pu) return B200BGZF_E_FORMAT;
        pc = c;
        pu = u;
    }
    *nmembers = (size_t)entries + 1;
    const size_t n = std::min<size_t>(cap, entries + 1);
    for (size_t i = 0; i < n; i++) {
        caddr[i] = i ? get(8 + 16 * (i - 1)) : 0;
        uaddr[i] = i ? get(16 + 16 * (i - 1)) : 0;
    }
    return entries + 1 > cap ? B200BGZF_E_NOSPACE : B200BGZF_OK;
}

extern "C" int b200bgzf_inflate_ranges_host(b200bgzf_ctx *ctx, const void *in, size_t in_bytes, const uint64_t *caddr, const uint64_t *uaddr,
                                            size_t nindex, const b200bgzf_range *ranges, size_t nranges, void *out, size_t out_cap,
                                            size_t *out_bytes, uint64_t *range_off, unsigned flags)
{
    if (!ctx || !out_bytes || (!in && in_bytes) || (!ranges && nranges) || (!caddr != !uaddr) || (caddr && !nindex)) return B200BGZF_E_ARG;
    const uint8_t *p = (const uint8_t *)in;
    /* ---- plan on the host: the index, every range as [beg, end) of the decoded stream, the output layout ---- */
    std::vector<uint64_t> wc, wu;
    if (!caddr) {
        const int r = walk_index(p, in_bytes, wc, wu);
        if (r) return r;
        caddr = wc.data();
        uaddr = wu.data();
        nindex = wc.size();
    }
    const size_t n = nindex;
    for (size_t m = 0; m < n; m++)
        if (caddr[m] >= in_bytes || (m && (caddr[m] <= caddr[m - 1] || uaddr[m] < uaddr[m - 1])) || (m == 0 && uaddr[0] != 0)) return B200BGZF_E_ARG;
    uint64_t total = 0;
    if (n) {                                            /* the decoded size: the last listed member's ISIZE */
        uint64_t sz = 0;
        if (!member_parse(p + caddr[n - 1], in_bytes - caddr[n - 1], &sz)) return B200BGZF_E_FORMAT;
        total = uaddr[n - 1] + rd32(p + caddr[n - 1] + sz - 4);
    }
    auto uend = [&](size_t m) { return m + 1 < n ? uaddr[m + 1] : total; };
    auto cend = [&](size_t m) { return m + 1 < n ? caddr[m + 1] : (uint64_t)in_bytes; };
    auto resolve = [&](uint64_t v, uint64_t *pos) {
        const uint64_t c = v >> 16, u = v & 0xffffu;
        if (c == in_bytes) { *pos = total; return u == 0; }
        if (!n || c < caddr[0]) return false;
        const size_t m = last_le(caddr, n, c);
        if (caddr[m] != c || u > uend(m) - uaddr[m]) return false;
        *pos = uaddr[m] + u;
        return true;
    };
    std::vector<uint64_t> rb(nranges), re(nranges);
    uint64_t out_total = 0;
    for (size_t i = 0; i < nranges; i++) {
        uint64_t b = ranges[i].beg, e = ranges[i].end;
        if ((flags & B200BGZF_RANGE_VOFFSET) && !(resolve(b, &b) && resolve(e, &e))) return B200BGZF_E_ARG;
        if (b > e || e > total) return B200BGZF_E_ARG;
        rb[i] = b;
        re[i] = e;
        if (range_off) range_off[i] = out_total;
        out_total += e - b;
    }
    *out_bytes = (size_t)out_total;
    if (out_total > out_cap || (!out && out_total)) return B200BGZF_E_NOSPACE;
    if (out_total == 0) return B200BGZF_OK;

    /* ---- groups of consecutive pieces of ranges, pipelined over the lanes ---- */
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    PendingGuard pg(ctx->lanes, kLanes);
    const uint64_t group_cap = range_budget() / 4, piece_cap = range_budget() / 16;
    const bool verify = (flags & B200BGZF_VERIFY) != 0;
    struct Piece { uint64_t beg, len, out; size_t first; };
    std::vector<uint64_t> stamp(n, ~0ull), msoff(n);
    std::vector<size_t> gm;                             /* the group's touched members */
    std::vector<Piece> gp;
    uint64_t gdec = 0, gout = 0, gout0 = 0, out_pos = 0, gid = 0;
    bool bad = false, badcrc = false;
    int r, lane_i = 0;
    auto complete = [&](Lane &l) -> int {
        CK(cudaStreamSynchronize(l.stream));
        if (l.h_total[1] & 1u) bad = true;
        if (l.h_total[1] & 2u) badcrc = true;
        l.pending = false;
        return 0;
    };
    auto submit = [&]() -> int {
        Lane &l = ctx->lanes[lane_i++ % kInflateLanes];
        if (l.pending && (r = complete(l))) return r;
        std::sort(gm.begin(), gm.end());
        const size_t M = gm.size(), P = gp.size();
        uint64_t cbytes = 0;
        for (size_t k = 0; k < M; k++)
            if (k + 1 == M || gm[k + 1] != gm[k] + 1) {                       /* end of a run of consecutive members */
                size_t k0 = k;
                while (k0 > 0 && gm[k0 - 1] + 1 == gm[k0]) k0--;
                cbytes += cend(gm[k]) - caddr[gm[k0]];
            }
        if ((r = lane_reserve(ctx, l, (uint32_t)std::max<size_t>(M, kInflateBatch), cbytes + 256, 0, false))) return r;
        const uint64_t obase = (gdec + 64 + 255) & ~(uint64_t)255;             /* the group's output behind its decoded members */
        CK(grow(&l.d_rdec, &l.rdec_cap, obase + gout + 64));
        CK(grow(&l.d_rmeta, &l.rmeta_cap, 4 * P));
        CK(grow(&l.h_in, &l.host_in_cap, cbytes + 16, true));
        CK(grow(&l.h_meta, &l.meta_cap, 3 * M + 4 * P, true));
        uint64_t *h_inoff = l.h_meta, *h_outoff = l.h_meta + M, *h_rm = l.h_meta + 3 * M;
        uint32_t *h_hdr = (uint32_t *)(l.h_meta + 2 * M), *h_msz = h_hdr + M;
        /* the compressed bytes of every run of touched members, packed; nothing else of the input is read */
        uint64_t pos = 0, soff = 0;
        for (size_t k0 = 0; k0 < M;) {
            size_t k1 = k0 + 1;
            while (k1 < M && gm[k1] == gm[k1 - 1] + 1) k1++;
            const uint64_t cs = caddr[gm[k0]], ce = cend(gm[k1 - 1]);
            memcpy(l.h_in + pos, p + cs, ce - cs);
            for (size_t k = k0; k < k1; k++) {
                const size_t m = gm[k];
                uint64_t sz = 0;
                const uint32_t hl = member_parse(p + caddr[m], cend(m) - caddr[m], &sz);
                if (!hl) return B200BGZF_E_FORMAT;
                const uint32_t isz = rd32(p + caddr[m] + sz - 4);
                if (isz != uend(m) - uaddr[m] || isz > 1032ull * (sz - hl) + 1032u) return B200BGZF_E_FORMAT;   /* (index and stream disagree) */
                h_inoff[k] = pos + (caddr[m] - cs);
                h_outoff[k] = soff;
                h_hdr[k] = hl;
                h_msz[k] = (uint32_t)sz;
                msoff[m] = soff;
                soff += isz;
            }
            pos += ce - cs;
            k0 = k1;
        }
        /* gather lists: where each piece starts in the decoded members and in the group's output, its length, first tile */
        uint64_t tiles = 0;
        for (size_t j = 0; j < P; j++) {
            const Piece &q = gp[j];
            h_rm[j] = msoff[q.first] + (q.beg - uaddr[q.first]);
            h_rm[P + j] = q.out - gout0;
            h_rm[2 * P + j] = q.len;
            h_rm[3 * P + j] = tiles;
            tiles += (q.len + BGZF_GATHER_TILE - 1) / BGZF_GATHER_TILE;
        }
        CK(cudaMemcpyAsync(l.d_in, l.h_in, pos, cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_inoff, h_inoff, M * sizeof(uint64_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_outoff, h_outoff, M * sizeof(uint64_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_inlen, h_hdr, M * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_len, h_msz, M * sizeof(uint32_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemcpyAsync(l.d_rmeta, h_rm, 4 * P * sizeof(uint64_t), cudaMemcpyHostToDevice, l.stream));
        CK(cudaMemsetAsync(l.d_total, 0, 4 * sizeof(uint64_t), l.stream));
        BgzfInflateArgs a;
        memset(&a, 0, sizeof a);
        a.in = l.d_in;
        a.in_off = l.d_inoff;
        a.out_off = l.d_outoff;
        a.hdr_len = l.d_inlen;
        a.msize = l.d_len;
        a.nblocks = (uint32_t)M;
        a.out = l.d_rdec;
        a.status = l.d_status;
        a.err_flag = (uint32_t *)(l.d_total + 1);
        a.crctab = ctx->d_crctab;
        a.crcpow = ctx->d_crcpow;
        a.verify_crc = verify ? 1 : 0;
        CK(bgzf_launch_inflate(&a, l.stream));
        BgzfRangeGatherArgs ga;
        ga.scratch = l.d_rdec;
        ga.win_lo = 0;
        ga.win_hi = ~0ull;
        ga.out = l.d_rdec + obase;
        ga.src = l.d_rmeta;
        ga.range_off = l.d_rmeta + P;
        ga.len = l.d_rmeta + 2 * P;
        ga.tile_off = l.d_rmeta + 3 * P;
        ga.nranges = (uint32_t)P;
        CK(bgzf_launch_range_gather(&ga, tiles, l.stream));
        ctx->launches += 2 + a.verify_crc;
        CK(cudaMemcpyAsync((uint8_t *)out + gout0, l.d_rdec + obase, gout, cudaMemcpyDeviceToHost, l.stream));
        CK(cudaMemcpyAsync(l.h_total, l.d_total, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, l.stream));
        l.pending = true;
        gid++;
        gm.clear();
        gp.clear();
        gout0 += gout;
        gdec = gout = 0;
        return 0;
    };
    for (size_t i = 0; i < nranges; i++) {
        for (uint64_t b = rb[i]; b < re[i];) {
            const uint64_t len = std::min(piece_cap, re[i] - b);
            const size_t f = last_le(uaddr, n, b), l = last_le(uaddr, n, b + len - 1);
            uint64_t add = 0;
            for (size_t m = f; m <= l; m++)
                if (stamp[m] != gid) add += uend(m) - uaddr[m];
            if (!gp.empty() && gdec + add + gout + len > group_cap) {
                if ((r = submit())) return r;
                add = uaddr[l] - uaddr[f] + (uend(l) - uaddr[l]);
            }
            if (gp.size() >= 0xffffffffu) return B200BGZF_E_ARG;
            for (size_t m = f; m <= l; m++)
                if (stamp[m] != gid) { stamp[m] = gid; gm.push_back(m); }
            gdec += add;
            gout += len;
            gp.push_back({ b, len, out_pos, f });
            out_pos += len;
            b += len;
        }
    }
    if (!gp.empty() && (r = submit())) return r;
    for (auto &l : ctx->lanes)
        if (l.pending && (r = complete(l))) return r;
    return bad ? B200BGZF_E_FORMAT : badcrc ? B200BGZF_E_CRC : B200BGZF_OK;
}

extern "C" int b200bgzf_inflate_ranges_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, const b200bgzf_range *ranges, size_t nranges,
                                              void *d_out, size_t out_cap, size_t *out_bytes, uint64_t *range_off, unsigned flags, void *stream_)
{
    if (!ctx || !d_in || !out_bytes || in_bytes < 28 || (!ranges && nranges) || nranges > 0x7fffffffu) return B200BGZF_E_ARG;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    int r = lane_reserve(ctx, l, 1, 0, 0, false);
    if (r) return r;
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : l.stream;
    uint64_t nm = 0, total = 0;
    if ((r = device_index(ctx, d_in, in_bytes, stream, &nm, &total))) return r;
    *out_bytes = 0;
    if (nranges == 0) return B200BGZF_OK;
    const size_t R = nranges;
    /* workspaces: per member diff (i32, nm + 1), m_soff, t_in_off, t_soff; per range 2 (beg, end) + delta, len, src, range_off,
     * tile_off + first (u32); pinned: 8 words of counts, the ranges, range_off */
    CK(grow(&ctx->d_rng_mem, &ctx->rng_mem_cap, 3 * (size_t)ctx->idx_cap + ctx->idx_cap / 2 + 2));
    CK(grow(&ctx->d_rng_rw, &ctx->rng_rw_cap, 7 * R + R / 2 + 1));
    CK(grow(&ctx->h_rng, &ctx->h_rng_cap, 8 + 3 * R, true));
    if (!ctx->d_rng_counts) CK(cudaMalloc((void **)&ctx->d_rng_counts, 8 * sizeof(uint64_t)));
    uint64_t *m_soff = ctx->d_rng_mem, *t_in_off = m_soff + nm, *t_soff = t_in_off + nm;
    int32_t *diff = (int32_t *)(t_soff + nm);
    uint64_t *d_rng = ctx->d_rng_rw, *delta = d_rng + 2 * R, *len = delta + R, *src = len + R, *roff = src + R, *toff = roff + R;
    uint32_t *first = (uint32_t *)(toff + R);
    uint64_t *h_counts = ctx->h_rng, *h_rng = ctx->h_rng + 8, *h_roff = h_rng + 2 * R;
    for (size_t i = 0; i < R; i++) { h_rng[2 * i] = ranges[i].beg; h_rng[2 * i + 1] = ranges[i].end; }
    CK(cudaMemcpyAsync(d_rng, h_rng, 2 * R * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    CK(cudaMemsetAsync(diff, 0, (nm + 1) * sizeof(int32_t), stream));
    CK(cudaMemsetAsync(ctx->d_rng_counts, 0, 8 * sizeof(uint64_t), stream));
    BgzfRangePlanArgs pa;
    pa.ranges = d_rng;
    pa.nranges = (uint32_t)R;
    pa.voffsets = (flags & B200BGZF_RANGE_VOFFSET) ? 1 : 0;
    pa.in_bytes = in_bytes;
    pa.in_off = ctx->d_idx_inoff;
    pa.out_off = ctx->d_idx_outoff;
    pa.isize = ctx->d_idx_isize;
    pa.nmembers = ctx->d_idx_counts;
    pa.total = ctx->d_idx_counts + 1;
    pa.diff = diff;
    pa.first = first;
    pa.delta = delta;
    pa.len = len;
    pa.status = (uint32_t *)(ctx->d_rng_counts + 4);
    CK(bgzf_launch_range_plan(&pa, stream));
    BgzfRangeTouchArgs ta;
    ta.nmembers = (uint32_t)nm;
    ta.nranges = (uint32_t)R;
    ta.diff = diff;
    ta.in_off = ctx->d_idx_inoff;
    ta.isize = ctx->d_idx_isize;
    ta.t_in_off = t_in_off;
    ta.t_soff = t_soff;
    ta.m_soff = m_soff;
    ta.first = first;
    ta.delta = delta;
    ta.len = len;
    ta.src = src;
    ta.range_off = roff;
    ta.tile_off = toff;
    ta.counts = ctx->d_rng_counts;
    CK(bgzf_launch_range_touch(&ta, stream));
    ctx->launches += 2;
    CK(cudaMemcpyAsync(h_counts, ctx->d_rng_counts, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaMemcpyAsync(h_roff, roff, R * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if ((uint32_t)h_counts[4]) return B200BGZF_E_ARG;
    const uint64_t nt = h_counts[0], sbytes = h_counts[1], obytes = h_counts[2], ntiles = h_counts[3];
    *out_bytes = (size_t)obytes;
    if (range_off) memcpy(range_off, h_roff, R * sizeof(uint64_t));
    if (obytes > out_cap || (!d_out && obytes)) return B200BGZF_E_NOSPACE;
    if (obytes == 0) return B200BGZF_OK;
    /* passes over consecutive touched members whose decoded bytes fit the scratch (one pass unless they exceed the budget) */
    const uint64_t budget = range_budget();
    std::vector<uint64_t> cut{ 0 }, base{ 0 };          /* pass k: touched members [cut[k], cut[k+1]), scratch coordinates from base[k] */
    if (sbytes <= budget) {
        cut.push_back(nt);
    } else {
        CK(grow(&ctx->h_rng_soff, &ctx->h_rng_soff_cap, (size_t)nt, true));
        uint64_t *h_soff = ctx->h_rng_soff;
        CK(cudaMemcpyAsync(h_soff, t_soff, nt * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
        CK(cudaStreamSynchronize(stream));
        for (uint64_t k0 = 0; k0 < nt;) {
            uint64_t k1 = k0 + 1;
            while (k1 < nt && (k1 + 1 < nt ? h_soff[k1 + 1] : sbytes) - h_soff[k0] <= budget) k1++;
            cut.push_back(k1);
            base.push_back(k1 < nt ? h_soff[k1] : sbytes);
            k0 = k1;
        }
        base.pop_back();
        for (size_t k = 0; k + 1 < cut.size(); k++)       /* scratch offsets relative to their pass */
            for (uint64_t j = cut[k]; j < cut[k + 1]; j++) h_soff[j] -= base[k];
        CK(cudaMemcpyAsync(t_soff, h_soff, nt * sizeof(uint64_t), cudaMemcpyHostToDevice, stream));
    }
    uint64_t widest = 0;
    for (size_t k = 0; k + 1 < cut.size(); k++) {
        const uint64_t hi = k + 2 < cut.size() ? base[k + 1] : sbytes;
        widest = std::max(widest, hi - base[k]);
    }
    CK(grow(&ctx->d_rng_scratch, &ctx->rng_scratch_cap, (size_t)widest + 64));
    for (size_t k = 0; k + 1 < cut.size(); k++) {
        BgzfInflateArgs a;
        memset(&a, 0, sizeof a);
        a.in = (const uint8_t *)d_in;
        a.in_off = t_in_off + cut[k];
        a.out_off = t_soff + cut[k];
        a.nblocks = (uint32_t)(cut[k + 1] - cut[k]);
        a.out = ctx->d_rng_scratch;
        a.status = ctx->d_inf_status + cut[k];
        a.err_flag = ctx->d_idx_status + 1;
        a.crctab = ctx->d_crctab;
        a.crcpow = ctx->d_crcpow;
        a.verify_crc = (flags & B200BGZF_VERIFY) ? 1 : 0;
        CK(bgzf_launch_inflate(&a, stream));
        BgzfRangeGatherArgs ga;
        ga.scratch = ctx->d_rng_scratch;
        ga.win_lo = base[k];
        ga.win_hi = k + 2 < cut.size() ? base[k + 1] : sbytes;
        ga.out = (uint8_t *)d_out;
        ga.src = src;
        ga.range_off = roff;
        ga.len = len;
        ga.tile_off = toff;
        ga.nranges = (uint32_t)R;
        CK(bgzf_launch_range_gather(&ga, ntiles, stream));
        ctx->launches += 2 + a.verify_crc;
    }
    CK(cudaMemcpyAsync(ctx->h_idx + 3, ctx->d_idx_status + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    const uint32_t ef = (uint32_t)ctx->h_idx[3];
    return (ef & 1u) ? B200BGZF_E_FORMAT : (ef & 2u) ? B200BGZF_E_CRC : B200BGZF_OK;
}

/* ------------------------------------------------------------------------------------------------ */
/* whole-stream gzip: random access through a checkpoint index (the format: include/b200bgzf.h)    */

namespace {

constexpr size_t kGzIxHead = 48;                 /* magic, in_bytes, hdr_len, crc32, isize, out_bytes, span, nchunks, npoints */
constexpr uint64_t kGzIxChunk = 20, kGzIxPoint = 8;
constexpr uint32_t kGzIxSpan = 1u << 20;         /* span 0 */

uint64_t rd64(const uint8_t *p) { return (uint64_t)rd32(p) | (uint64_t)rd32(p + 4) << 32; }
void wr32(uint8_t *p, uint32_t v) { for (int k = 0; k < 4; k++) p[k] = (uint8_t)(v >> (8 * k)); }
void wr64(uint8_t *p, uint64_t v) { wr32(p, (uint32_t)v); wr32(p + 4, (uint32_t)(v >> 32)); }

/* CRC-32 on the host, eight bytes per step (an index carries up to 32 KiB of window per access point) */
uint32_t host_crc32(const uint8_t *p, size_t n)
{
    static const std::vector<uint32_t> tab = [] {
        std::vector<uint32_t> t(8 * 256);
        bg_make_crc_table(t.data());
        for (int k = 1; k < 8; k++)
            for (int i = 0; i < 256; i++) t[k * 256 + i] = (t[(k - 1) * 256 + i] >> 8) ^ t[t[(k - 1) * 256 + i] & 0xffu];
        return t;
    }();
    const uint32_t *t = tab.data();
    uint32_t c = 0xffffffffu;
    for (; n >= 8; p += 8, n -= 8) {
        const uint32_t a = rd32(p) ^ c, b = rd32(p + 4);
        c = t[7 * 256 + (a & 0xffu)] ^ t[6 * 256 + ((a >> 8) & 0xffu)] ^ t[5 * 256 + ((a >> 16) & 0xffu)] ^ t[4 * 256 + (a >> 24)] ^
            t[3 * 256 + (b & 0xffu)] ^ t[2 * 256 + ((b >> 8) & 0xffu)] ^ t[256 + ((b >> 16) & 0xffu)] ^ t[b >> 24];
    }
    while (n--) c = t[(c ^ *p++) & 0xffu] ^ (c >> 8);
    return ~c;
}

/* a parsed index: every field checked, the windows left in place */
struct GzIx {
    uint64_t in_bytes = 0, out_bytes = 0;
    uint32_t hdr_len = 0, crc = 0, isize = 0, span = 0;
    std::vector<uint64_t> cs, uo;        /* per chunk: file offset, output offset */
    std::vector<uint32_t> ccrc;          /* per chunk: CRC-32 of its output */
    std::vector<uint32_t> pchunk, wlen;  /* per access point: its chunk, its window's length */
    std::vector<uint64_t> woff;          /* per access point: where its window starts in `win` */
    const uint8_t *win = nullptr;
    size_t n() const { return cs.size(); }
    uint64_t uend(size_t k) const { return k + 1 < cs.size() ? uo[k + 1] : out_bytes; }
    uint64_t cend(size_t k) const { return k + 1 < cs.size() ? cs[k + 1] : in_bytes - 8; }
};

int gz_index_parse(const void *index, size_t bytes, GzIx &ix)
{
    const uint8_t *x = (const uint8_t *)index;
    if (bytes < kGzIxHead + 4 || memcmp(x, "B2GZIX01", 8) || rd32(x + bytes - 4) != host_crc32(x, bytes - 4)) return B200BGZF_E_FORMAT;
    ix.in_bytes = rd64(x + 8);
    ix.hdr_len = rd32(x + 16);
    ix.crc = rd32(x + 20);
    ix.isize = rd32(x + 24);
    ix.out_bytes = rd64(x + 28);
    ix.span = rd32(x + 36);
    const uint64_t n = rd32(x + 40), np = rd32(x + 44);
    if (!n || !np || np > n || ix.span < 32768 || ix.hdr_len < 10 || ix.in_bytes < (uint64_t)ix.hdr_len + 10 ||
        ix.out_bytes > 0x7fffffffu || (uint32_t)ix.out_bytes != ix.isize)
        return B200BGZF_E_FORMAT;
    const uint64_t fixed = kGzIxHead + kGzIxChunk * n + kGzIxPoint * np + 4;
    if (fixed > bytes) return B200BGZF_E_FORMAT;
    ix.cs.resize(n);
    ix.uo.resize(n);
    ix.ccrc.resize(n);
    for (uint64_t k = 0; k < n; k++) {
        const uint8_t *c = x + kGzIxHead + kGzIxChunk * k;
        const uint64_t s = rd64(c), u = rd64(c + 8);
        if (k == 0 ? (s != ix.hdr_len || u != 0) : (s <= ix.cs[k - 1] || u < ix.uo[k - 1])) return B200BGZF_E_FORMAT;
        if (s >= ix.in_bytes - 8 || u > ix.out_bytes) return B200BGZF_E_FORMAT;
        ix.cs[k] = s;
        ix.uo[k] = u;
        ix.ccrc[k] = rd32(c + 16);
    }
    uint64_t wsum = 0;
    for (uint64_t p = 0; p < np; p++) {
        const uint8_t *q = x + kGzIxHead + kGzIxChunk * n + kGzIxPoint * p;
        const uint32_t k = rd32(q), w = rd32(q + 4);
        if (p == 0 ? k != 0 : k <= ix.pchunk.back()) return B200BGZF_E_FORMAT;
        if (k >= n || w != std::min<uint64_t>(32768, ix.uo[k])) return B200BGZF_E_FORMAT;
        ix.pchunk.push_back(k);
        ix.wlen.push_back(w);
        ix.woff.push_back(wsum);
        wsum += w;
    }
    if (fixed + wsum != bytes) return B200BGZF_E_FORMAT;
    ix.win = x + kGzIxHead + kGzIxChunk * n + kGzIxPoint * np;
    return B200BGZF_OK;
}

/* Builds the index of the member d_in[0, in_bytes) (header of hlen bytes, trailer tr): its flush-point chain decoded once into
 * the context's output buffer, the chunks' CRC-32 (bgzf_verify_kernel, one unit per chunk), the access points' windows
 * (gathered on the device, copied back in one piece). */
int gzip_index_build(b200bgzf_ctx *ctx, const uint8_t *d_in, size_t in_bytes, uint32_t hlen, const uint8_t tr[8], uint32_t span,
                     void *index, size_t index_cap, size_t *index_bytes, cudaStream_t stream)
{
    const uint32_t want_crc = rd32(tr), isize = rd32(tr + 4);
    int r = gzip_member_check(in_bytes, hlen, isize);
    if (r) return r;
    GzWork &z = ctx->gz;
    CK(grow(&z.d_out, &z.out_cap, (size_t)isize + 64));
    size_t total = isize;
    GzChain ch;
    r = gzip_chain_inflate(ctx, d_in, in_bytes, hlen, isize, want_crc, z.d_out, isize, &total, 0, stream,
                           [](uint64_t, uint64_t) { return 0; }, &ch);
    if (r == BGZF_GZIP_FALLBACK || r == B200BGZF_E_NOSPACE) return B200BGZF_E_FORMAT;   /* not indexable */
    if (r) return r;
    const uint64_t n = ch.nchunks;
    std::vector<uint64_t> cs(n), uo(n);
    CK(cudaMemcpyAsync(uo.data(), ch.a.c_off, n * 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaMemcpyAsync(cs.data(), ch.a.c_start, n * 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    /* access points: chunk 0, then every chunk at least `span` bytes of output past the previous point */
    std::vector<uint32_t> pts{ 0 };
    for (uint64_t k = 1; k < n; k++)
        if (uo[k] - uo[pts.back()] >= span) pts.push_back((uint32_t)k);
    const uint64_t np = pts.size();
    std::vector<uint64_t> wl(np), wo(np);
    uint64_t wsum = 0;
    for (uint64_t p = 0; p < np; p++) {
        wl[p] = std::min<uint64_t>(32768, uo[pts[p]]);
        wo[p] = wsum;
        wsum += wl[p];
    }
    const uint64_t size = kGzIxHead + kGzIxChunk * n + kGzIxPoint * np + wsum + 4;
    *index_bytes = (size_t)size;
    if (!index || index_cap < size) return B200BGZF_E_NOSPACE;
    /* chunk CRCs: bgzf_verify_kernel over pieces of the output (in_off / hdr_len / msize / status unused: zeros) */
    uint32_t *zero = ch.a.olen, *ucrc = ch.a.status;     /* (per-candidate arrays the chain no longer needs, >= n entries) */
    CK(cudaMemsetAsync(zero, 0, n * 4, stream));
    BgzfInflateArgs v;
    memset(&v, 0, sizeof v);
    v.in = z.d_out;
    v.in_off = ch.a.c_off;
    v.out_off = ch.a.c_off;
    v.hdr_len = zero;
    v.msize = zero;
    v.unit_isize = ch.a.c_len;
    v.status = zero;
    v.unit_crc = ucrc;
    v.nblocks = (uint32_t)n;
    v.out = z.d_out;
    v.err_flag = ch.a.err + 2;
    v.verify_crc = 1;
    v.crctab = ctx->d_crctab;
    v.crcpow = ctx->d_crcpow;
    CK(bgzf_launch_verify(&v, stream));
    ctx->launches += 1;
    /* windows: bgzf_range_gather_kernel cuts them out of the output, back to back */
    std::vector<uint8_t> out(size);
    if (wsum) {
        std::vector<uint64_t> g(4 * np);
        uint64_t tiles = 0;
        for (uint64_t p = 0; p < np; p++) {
            g[p] = uo[pts[p]] - wl[p];
            g[np + p] = wo[p];
            g[2 * np + p] = wl[p];
            g[3 * np + p] = tiles;
            tiles += (wl[p] + BGZF_GATHER_TILE - 1) / BGZF_GATHER_TILE;
        }
        CK(grow(&z.d_meta, &z.meta_cap, 4 * np));
        CK(grow(&z.d_win, &z.win_cap, wsum + 64));
        CK(cudaMemcpyAsync(z.d_meta, g.data(), g.size() * 8, cudaMemcpyHostToDevice, stream));
        BgzfRangeGatherArgs ga;
        ga.scratch = z.d_out;
        ga.win_lo = 0;
        ga.win_hi = ~0ull;
        ga.out = z.d_win;
        ga.src = z.d_meta;
        ga.range_off = z.d_meta + np;
        ga.len = z.d_meta + 2 * np;
        ga.tile_off = z.d_meta + 3 * np;
        ga.nranges = (uint32_t)np;
        CK(bgzf_launch_range_gather(&ga, tiles, stream));
        ctx->launches += 1;
        CK(cudaMemcpyAsync(out.data() + kGzIxHead + kGzIxChunk * n + kGzIxPoint * np, z.d_win, wsum, cudaMemcpyDeviceToHost, stream));
    }
    std::vector<uint32_t> crc(n);
    CK(cudaMemcpyAsync(crc.data(), ucrc, n * 4, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    uint8_t *x = out.data();
    memcpy(x, "B2GZIX01", 8);
    wr64(x + 8, in_bytes);
    wr32(x + 16, hlen);
    wr32(x + 20, want_crc);
    wr32(x + 24, isize);
    wr64(x + 28, total);
    wr32(x + 36, span);
    wr32(x + 40, (uint32_t)n);
    wr32(x + 44, (uint32_t)np);
    for (uint64_t k = 0; k < n; k++) {
        uint8_t *c = x + kGzIxHead + kGzIxChunk * k;
        wr64(c, cs[k] + hlen);
        wr64(c + 8, uo[k]);
        wr32(c + 16, crc[k]);
    }
    for (uint64_t p = 0; p < np; p++) {
        uint8_t *q = x + kGzIxHead + kGzIxChunk * n + kGzIxPoint * p;
        wr32(q, pts[p]);
        wr32(q + 4, (uint32_t)wl[p]);
    }
    wr32(x + size - 4, host_crc32(x, size - 4));
    memcpy(index, x, size);
    return B200BGZF_OK;
}

int gzip_span(uint32_t *span)
{
    if (*span == 0) *span = kGzIxSpan;
    return *span < 32768 ? B200BGZF_E_ARG : B200BGZF_OK;
}

/* a run: chunks [s, e] decoded from the access point s */
struct GzRun {
    uint32_t s, e;
};

/* Checks the index against the file (size, trailer) and the ranges against the index; the merged runs the ranges touch, in
 * order, range_off and the output size.  Returns E_FORMAT / E_ARG / E_NOSPACE as the public calls do. */
int gz_ranges_plan(const GzIx &ix, size_t in_bytes, const uint8_t tr[8], const b200bgzf_range *ranges, size_t nranges, size_t out_cap,
                   bool have_out, size_t *out_bytes, uint64_t *range_off, std::vector<GzRun> &runs)
{
    if (ix.in_bytes != in_bytes || ix.crc != rd32(tr) || ix.isize != rd32(tr + 4)) return B200BGZF_E_FORMAT;
    uint64_t out_total = 0;
    for (size_t i = 0; i < nranges; i++) {
        const uint64_t b = ranges[i].beg, e = ranges[i].end;
        if (b > e || e > ix.out_bytes) return B200BGZF_E_ARG;
        if (range_off) range_off[i] = out_total;
        out_total += e - b;
        if (b == e) continue;
        const uint32_t f = (uint32_t)last_le(ix.uo.data(), ix.n(), b), l = (uint32_t)last_le(ix.uo.data(), ix.n(), e - 1);
        const size_t p = (size_t)(std::upper_bound(ix.pchunk.begin(), ix.pchunk.end(), f) - ix.pchunk.begin()) - 1;
        runs.push_back({ ix.pchunk[p], l });
    }
    *out_bytes = (size_t)out_total;
    if (out_total > out_cap || (!have_out && out_total)) return B200BGZF_E_NOSPACE;
    std::sort(runs.begin(), runs.end(), [](const GzRun &a, const GzRun &b) { return a.s < b.s || (a.s == b.s && a.e > b.e); });
    size_t m = 0;
    for (size_t i = 0; i < runs.size(); i++) {
        if (m && runs[i].s <= runs[m - 1].e + 1) runs[m - 1].e = std::max(runs[m - 1].e, runs[i].e);
        else runs[m++] = runs[i];
    }
    runs.resize(m);
    return B200BGZF_OK;
}

/* Decodes the runs and cuts the ranges out of them into d_out.  The compressed bytes are in d_data[0, data_len), chunk k at
 * cstart[k] (indexed by chunk number, only touched chunks are read).  A batch holds consecutive runs (or parts of one run cut at
 * a chunk boundary) whose u16 layout fits the budget: per part 32 KiB of window, then its chunks.  A part that continues a run
 * takes its window from the last 32 KiB of the batch before it, resolved in scratch (as gzip_chain_inflate's prefix does). */
int gz_ranges_decode(b200bgzf_ctx *ctx, const GzIx &ix, const uint8_t *d_data, uint64_t data_len, const std::vector<uint64_t> &cstart,
                     const std::vector<GzRun> &runs, const b200bgzf_range *ranges, size_t nranges, const uint64_t *range_off,
                     uint8_t *d_out, unsigned flags, cudaStream_t stream)
{
    GzWork &z = ctx->gz;
    const uint64_t win = bgzf_gzip_window(), half = gzip_budget() / 2;
    struct Part { uint32_t run, k0, k1; bool cont; uint64_t pos; };    /* chunks [k0, k1); pos: its window's place in the layout */
    std::vector<std::vector<Part>> batches(1);
    std::vector<uint64_t> bytes_of;                                    /* per batch: image bytes (layout after the first window) */
    uint64_t used = 0;
    auto close = [&]() { bytes_of.push_back(used - win); batches.emplace_back(); used = 0; };
    for (uint32_t r = 0; r < runs.size(); r++) {
        bool cont = false;
        for (uint32_t k = runs[r].s; k <= runs[r].e;) {
            if (win + ix.uend(k) - ix.uo[k] > half - used) {
                if (!used) return B200BGZF_E_FORMAT;                   /* one chunk alone is over the budget */
                close();
                continue;
            }
            uint32_t k1 = k + 1;
            while (k1 <= runs[r].e && win + ix.uend(k1) - ix.uo[k] <= half - used) k1++;
            batches.back().push_back({ r, k, k1, cont, used });
            used += win + ix.uo[k1 - 1] - ix.uo[k] + (ix.uend(k1 - 1) - ix.uo[k1 - 1]);
            if (k1 <= runs[r].e) { close(); cont = true; }
            k = k1;
        }
    }
    if (used) close();
    batches.pop_back();
    /* image coordinates of every touched chunk over all batches, then the gather lists of the ranges */
    std::vector<uint64_t> gbase(batches.size()), gpos(ix.n());
    uint64_t g = 0, most = 0;
    for (size_t b = 0; b < batches.size(); b++) {
        gbase[b] = g;
        for (const Part &p : batches[b])
            for (uint32_t k = p.k0; k < p.k1; k++) gpos[k] = g + p.pos + ix.uo[k] - ix.uo[p.k0];
        g += bytes_of[b];
        most = std::max(most, bytes_of[b]);
    }
    const uint64_t R = nranges;
    std::vector<uint64_t> rl(4 * R);
    uint64_t tiles = 0;
    for (uint64_t i = 0; i < R; i++) {
        const uint64_t b = ranges[i].beg, len = ranges[i].end - b;
        rl[i] = len ? gpos[last_le(ix.uo.data(), ix.n(), b)] + b - ix.uo[last_le(ix.uo.data(), ix.n(), b)] : 0;
        rl[R + i] = range_off[i];
        rl[2 * R + i] = len;
        rl[3 * R + i] = tiles;
        tiles += (len + BGZF_GATHER_TILE - 1) / BGZF_GATHER_TILE;
    }
    size_t maxj = 0, maxw = 0;
    for (auto &parts : batches) {
        size_t j = 0;
        for (const Part &p : parts) j += p.k1 - p.k0;
        maxj = std::max(maxj, j);
        maxw = std::max(maxw, parts.size());
    }
    /* u64 meta: the gather lists [4R], then per batch c_start, c_off, m_off [J], win_src, win_dst [W]; u32 after it: c_len,
     * lastm, anchor, zero, unit_crc [J], win_len [W], err */
    const size_t m64 = 4 * R + 3 * maxj + 2 * maxw, m32 = 5 * maxj + maxw + 4;
    CK(grow(&z.d_meta, &z.meta_cap, m64 + (m32 + 1) / 2));
    CK(grow(&z.scratch, &z.scratch_cap, win + most + 16));
    CK(grow(&z.d_img, &z.img_cap, most + 64));
    CK(grow(&z.d_carry, &z.carry_cap, win));
    size_t wcap = 0;
    for (auto &parts : batches) {
        size_t w = 0;
        for (const Part &p : parts) w += p.cont ? 0 : 32768;
        wcap = std::max(wcap, w);
    }
    CK(grow(&z.d_win, &z.win_cap, wcap + 64));
    uint64_t *d_rl = z.d_meta, *d64 = z.d_meta + 4 * R;
    uint32_t *d32 = (uint32_t *)(z.d_meta + m64);
    uint32_t *d_err = d32 + 5 * maxj + maxw;
    CK(cudaMemcpyAsync(d_rl, rl.data(), rl.size() * 8, cudaMemcpyHostToDevice, stream));
    CK(cudaMemsetAsync(d_err, 0, 4, stream));
    const bool verify = (flags & B200BGZF_VERIFY) != 0;
    bool badcrc = false;
    std::vector<uint64_t> h64;
    std::vector<uint32_t> h32, hcrc, want;
    std::vector<uint8_t> hwin;
    for (size_t b = 0; b < batches.size(); b++) {
        const std::vector<Part> &parts = batches[b];
        size_t J = 0, W = 0;
        for (const Part &p : parts) { J += p.k1 - p.k0; W += p.cont ? 0 : 1; }
        h64.assign(3 * J + 2 * W, 0);
        h32.assign(J + W, 0);
        hwin.clear();
        want.clear();
        uint64_t *c_start = h64.data(), *c_off = c_start + J, *m_off = c_off + J, *wsrc = m_off + J, *wdst = wsrc + W;
        uint32_t *c_len = h32.data(), *wlen = c_len + J;
        size_t j = 0, w = 0;
        for (const Part &p : parts) {
            for (uint32_t k = p.k0; k < p.k1; k++, j++) {
                c_start[j] = cstart[k];
                c_off[j] = p.pos + ix.uo[k] - ix.uo[p.k0];
                m_off[j] = ix.uo[k];
                c_len[j] = (uint32_t)(ix.uend(k) - ix.uo[k]);
                want.push_back(ix.ccrc[k]);
            }
            if (p.cont) continue;
            const size_t pt = (size_t)(std::lower_bound(ix.pchunk.begin(), ix.pchunk.end(), p.k0) - ix.pchunk.begin());
            wsrc[w] = hwin.size();
            wdst[w] = p.pos;
            wlen[w] = ix.wlen[pt];
            hwin.insert(hwin.end(), ix.win + ix.woff[pt], ix.win + ix.woff[pt] + ix.wlen[pt]);
            w++;
        }
        CK(cudaMemcpyAsync(d64, h64.data(), h64.size() * 8, cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(d32, h32.data(), J * 4, cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(d32 + 5 * maxj, wlen, W * 4, cudaMemcpyHostToDevice, stream));
        if (!hwin.empty()) CK(cudaMemcpyAsync(z.d_win, hwin.data(), hwin.size(), cudaMemcpyHostToDevice, stream));
        if (parts[0].cont) CK(cudaMemcpyAsync(z.scratch, z.d_carry, win * 2, cudaMemcpyDeviceToDevice, stream));
        BgzfGzipArgs a;
        memset(&a, 0, sizeof a);
        a.data = d_data;
        a.data_len = data_len;
        a.max_in = kGzMaxChunkIn;
        a.c_start = d64;
        a.c_off = d64 + J;
        a.c_len = d32;
        a.lastm = d32 + maxj;
        a.anchor = d32 + 2 * maxj;
        a.scratch = z.scratch;
        a.out = z.d_img;
        a.err = d_err;
        BgzfGzipRunArgs ra;
        ra.nchunks = (uint32_t)J;
        ra.m_off = d64 + 2 * J;
        ra.nwin = (uint32_t)W;
        ra.win = z.d_win;
        ra.win_src = d64 + 3 * J;
        ra.win_len = d32 + 5 * maxj;
        ra.win_dst = d64 + 3 * J + W;
        CK(bgzf_launch_gzip_runs(&a, &ra, bytes_of[b], stream));
        ctx->launches += 4 + (W ? 1 : 0) + (bytes_of[b] ? 1 : 0);
        if (verify) {
            uint32_t *zero = d32 + 3 * maxj, *ucrc = d32 + 4 * maxj;
            CK(cudaMemsetAsync(zero, 0, J * 4, stream));
            BgzfInflateArgs v;
            memset(&v, 0, sizeof v);
            v.in = z.d_img;
            v.in_off = a.c_off;
            v.out_off = a.c_off;
            v.hdr_len = zero;
            v.msize = zero;
            v.unit_isize = a.c_len;
            v.status = zero;
            v.unit_crc = ucrc;
            v.nblocks = (uint32_t)J;
            v.out = z.d_img;
            v.err_flag = d_err + 1;
            v.verify_crc = 1;
            v.crctab = ctx->d_crctab;
            v.crcpow = ctx->d_crcpow;
            CK(bgzf_launch_verify(&v, stream));
            ctx->launches += 1;
            hcrc.resize(J);
            CK(cudaMemcpyAsync(hcrc.data(), ucrc, J * 4, cudaMemcpyDeviceToHost, stream));
        }
        BgzfRangeGatherArgs ga;
        ga.scratch = z.d_img;
        ga.win_lo = gbase[b];
        ga.win_hi = gbase[b] + bytes_of[b];
        ga.out = d_out;
        ga.src = d_rl;
        ga.range_off = d_rl + R;
        ga.len = d_rl + 2 * R;
        ga.tile_off = d_rl + 3 * R;
        ga.nranges = (uint32_t)R;
        CK(bgzf_launch_range_gather(&ga, tiles, stream));
        ctx->launches += 1;
        if (parts.back().k1 <= runs[parts.back().run].e)   /* the last run goes on in the next batch: its window */
            CK(cudaMemcpyAsync(z.d_carry, z.scratch + bytes_of[b], win * 2, cudaMemcpyDeviceToDevice, stream));
        if (verify) {
            CK(cudaStreamSynchronize(stream));
            if (hcrc != want) badcrc = true;
        }
    }
    uint32_t err = 0;
    CK(cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    return err ? B200BGZF_E_FORMAT : badcrc ? B200BGZF_E_CRC : B200BGZF_OK;
}

}  // namespace

extern "C" int b200bgzf_gzip_index_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, uint32_t span, void *index,
                                          size_t index_cap, size_t *index_bytes, void *stream_)
{
    if (!ctx || !d_in || !index_bytes || gzip_span(&span)) return B200BGZF_E_ARG;
    *index_bytes = 0;
    if (in_bytes < 18) return B200BGZF_E_FORMAT;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    int r = lane_reserve(ctx, l, 1, 0, 0, false);
    if (r) return r;
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : l.stream;
    uint8_t tr[8];
    size_t hlen = 0;
    if ((r = gzip_device_header(ctx, (const uint8_t *)d_in, in_bytes, stream, &hlen, tr))) return r;
    return gzip_index_build(ctx, (const uint8_t *)d_in, in_bytes, (uint32_t)hlen, tr, span, index, index_cap, index_bytes, stream);
}

extern "C" int b200bgzf_gzip_index_host(b200bgzf_ctx *ctx, const void *in_, size_t in_bytes, uint32_t span, void *index, size_t index_cap,
                                        size_t *index_bytes)
{
    const uint8_t *in = (const uint8_t *)in_;
    if (!ctx || !in || !index_bytes || gzip_span(&span)) return B200BGZF_E_ARG;
    *index_bytes = 0;
    if (in_bytes < 18) return B200BGZF_E_FORMAT;
    size_t xoff, xlen;
    const size_t hlen = bgzf_gz_header(in, in_bytes, &xoff, &xlen);
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    int r = lane_reserve(ctx, l, 1, 0, 0, false);
    if (r) return r;
    GzWork &z = ctx->gz;
    CK(grow(&z.d_in, &z.in_cap, in_bytes + 64));
    CK(cudaMemcpyAsync(z.d_in, in, in_bytes, cudaMemcpyHostToDevice, l.stream));
    return gzip_index_build(ctx, z.d_in, in_bytes, (uint32_t)hlen, in + in_bytes - 8, span, index, index_cap, index_bytes, l.stream);
}

extern "C" int b200bgzf_gzip_inflate_ranges_device(b200bgzf_ctx *ctx, const void *d_in, size_t in_bytes, const void *index, size_t index_bytes,
                                                   const b200bgzf_range *ranges, size_t nranges, void *d_out, size_t out_cap,
                                                   size_t *out_bytes, uint64_t *range_off, unsigned flags, void *stream_)
{
    if (!ctx || !d_in || !index || !out_bytes || (!ranges && nranges) || nranges > 0x7fffffffu || (flags & B200BGZF_RANGE_VOFFSET))
        return B200BGZF_E_ARG;
    *out_bytes = 0;
    GzIx ix;
    int r = gz_index_parse(index, index_bytes, ix);
    if (r) return r;
    if (in_bytes != ix.in_bytes) return B200BGZF_E_FORMAT;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    if ((r = lane_reserve(ctx, l, 1, 0, 0, false))) return r;
    cudaStream_t stream = stream_ ? (cudaStream_t)stream_ : l.stream;
    uint8_t tr[8];
    CK(cudaMemcpyAsync(tr, (const uint8_t *)d_in + in_bytes - 8, 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    std::vector<uint64_t> roff(nranges);
    std::vector<GzRun> runs;
    r = gz_ranges_plan(ix, in_bytes, tr, ranges, nranges, out_cap, d_out != nullptr, out_bytes, roff.data(), runs);
    if (range_off && (r == B200BGZF_OK || r == B200BGZF_E_NOSPACE)) memcpy(range_off, roff.data(), nranges * 8);
    if (r || runs.empty()) return r;
    return gz_ranges_decode(ctx, ix, (const uint8_t *)d_in, in_bytes - 8, ix.cs, runs, ranges, nranges, roff.data(), (uint8_t *)d_out,
                            flags, stream);
}

extern "C" int b200bgzf_gzip_inflate_ranges_host(b200bgzf_ctx *ctx, const void *in_, size_t in_bytes, const void *index, size_t index_bytes,
                                                 const b200bgzf_range *ranges, size_t nranges, void *out, size_t out_cap,
                                                 size_t *out_bytes, uint64_t *range_off, unsigned flags)
{
    const uint8_t *in = (const uint8_t *)in_;
    if (!ctx || !in || !index || !out_bytes || (!ranges && nranges) || nranges > 0x7fffffffu || (flags & B200BGZF_RANGE_VOFFSET))
        return B200BGZF_E_ARG;
    *out_bytes = 0;
    GzIx ix;
    int r = gz_index_parse(index, index_bytes, ix);
    if (r) return r;
    if (in_bytes != ix.in_bytes) return B200BGZF_E_FORMAT;
    std::vector<uint64_t> roff(nranges);
    std::vector<GzRun> runs;
    r = gz_ranges_plan(ix, in_bytes, in + in_bytes - 8, ranges, nranges, out_cap, out != nullptr, out_bytes, roff.data(), runs);
    if (range_off && (r == B200BGZF_OK || r == B200BGZF_E_NOSPACE)) memcpy(range_off, roff.data(), nranges * 8);
    if (r || runs.empty()) return r;
    DeviceGuard g(ctx->device);
    std::lock_guard<std::mutex> lk(ctx->mu);
    Lane &l = ctx->lanes[0];
    if ((r = lane_reserve(ctx, l, 1, 0, 0, false))) return r;
    GzWork &z = ctx->gz;
    /* only the compressed bytes of the touched runs are read: packed back to back on the device */
    std::vector<uint64_t> cstart(ix.n());
    uint64_t packed = 0;
    for (const GzRun &u : runs) {
        for (uint32_t k = u.s; k <= u.e; k++) cstart[k] = packed + ix.cs[k] - ix.cs[u.s];
        packed += ix.cend(u.e) - ix.cs[u.s];
    }
    CK(grow(&z.d_in, &z.in_cap, packed + 64));
    CK(grow(&z.d_rout, &z.rout_cap, *out_bytes + 64));
    for (const GzRun &u : runs)
        CK(cudaMemcpyAsync(z.d_in + cstart[u.s], in + ix.cs[u.s], ix.cend(u.e) - ix.cs[u.s], cudaMemcpyHostToDevice, l.stream));
    r = gz_ranges_decode(ctx, ix, z.d_in, packed, cstart, runs, ranges, nranges, roff.data(), z.d_rout, flags, l.stream);
    if (r) return r;
    CK(cudaMemcpyAsync(out, z.d_rout, *out_bytes, cudaMemcpyDeviceToHost, l.stream));
    CK(cudaStreamSynchronize(l.stream));
    return B200BGZF_OK;
}
