// garage_ec.cu -- C ABI (include/garage_ec.h) over the sm_100a kernels in rs_kernels.cuh.
//
// Product code: no CPU fallback, nothing from oracle/.  Every entry point returns a status
// code and never throws/aborts across the boundary, mirroring the reference's
// Result<_, Error> convention (src/util/error.rs:14-82; SURVEY.md section 8(b)).
#include "../../include/garage_ec.h"

#if defined(__x86_64__)
#include <emmintrin.h>
#include <immintrin.h>
#endif
#include <cuda_runtime.h>

#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cctype>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <utility>
#include <vector>

#include "rs_kernels.cuh"

using namespace garage_ec;

static_assert(GARAGE_EC_MAX_K == kMaxK && GARAGE_EC_MAX_M == kMaxM, "header/kernels limits differ");
static_assert(GARAGE_EC_MAX_K == GARAGE_EC_MAX_K_HOST && GARAGE_EC_MAX_M == GARAGE_EC_MAX_M_HOST,
              "header/gf256 limits differ");

namespace {

constexpr int kHostLanes = 3;                       // H2D / kernel / D2H overlap across chunks
constexpr size_t kHostChunkBytes = 48ull << 20;     // target source bytes per pipeline chunk

struct HostLane {
    cudaStream_t stream = nullptr;
    uint8_t *d_buf = nullptr;  // chunk of shards (sources + outputs)
    size_t d_cap = 0;
    uint8_t *d_small = nullptr;  // shard_len / present / want / status / mismatch / plan
    size_t small_cap = 0;
    cudaEvent_t done = nullptr;  // blocking-sync event (garage_ec_set_wait_mode)
};
// One HOST-mode call owns one set of lanes for its duration; concurrent callers (tokio
// spawn_blocking threads, src/block/block.rs:86) get different sets, up to kMaxLaneSets.
struct LaneSet {
    HostLane lanes[kHostLanes];
};
constexpr int kMaxLaneSets = 4;

}  // namespace

struct garage_ec_ctx {
    int device = 0, k = 0, m = 0;
    uint8_t P[kMaxM * kMaxK] = {0};
    int sm_count = 0;
    size_t smem_optin = 0;
    std::mutex pool_mu;  // lane-set pool of the HOST-mode calls
    std::condition_variable pool_cv;
    std::vector<LaneSet *> free_sets;
    int n_sets = 0;
    // NUMA placement of the GPU (from sysfs): host memory for DMA should live on this node
    // stream-ordered scratch (decode plans of DEVICE-mode calls) comes from a pool of our own that KEEPS freed memory:
    // the default pool hands memory back to the driver at every synchronisation, and re-mapping it on the next call
    // cost 10-40 ms of host time at random whenever the GPU work ahead of it was short (config-5 sweep with adler8 tags)
    cudaMemPool_t pool = nullptr;
    std::atomic<int> sum_kind{GARAGE_EC_SUM_BLAKE2};  // per-shard integrity tag (garage_ec_set_sum_kind)
    int numa_node = -1;
    bool have_node_cpus = false;
    cpu_set_t node_cpus;
    int last_alloc_node = -1;                 // node the last garage_ec_host_alloc landed on (-1 unknown)
    std::atomic<long> fault_countdown{-1};
    // GARAGE_EC_TRACE=1: host-side time per phase of the block-level encode call, printed at destroy (tuning aid)
    bool trace = false;
    // how a HOST-mode call waits for its lanes: 0 = cudaStreamSynchronize (the driver spins: lowest latency, one CPU
    // per waiting caller), 1 = block on an event (garage_ec_set_wait_mode)
    std::atomic<int> wait_blocking{0};
    // HOST-mode calls on pinned (device-addressable) buffers: let the kernel read and write the host memory directly
    // over PCIe instead of staging chunks through device buffers.  Measured on one B200 (profiles/r02_summary.md):
    // reconstruct, whose staged form moves ~130 scattered 100 KB pieces per chunk in each direction, goes from
    // 39.7 + 15.9 GB/s (up + down) to 49.9 + 20.0 GB/s; encode, one contiguous copy per chunk, is faster staged
    // (53.3 vs 49.9 GB/s).  Default: reconstruct only.  GARAGE_EC_ZEROCOPY=0 turns it off, =1 also applies it to encode.
    bool zero_copy_rec = true, zero_copy_enc = false;
    std::atomic<uint64_t> tr_calls{0}, tr_blocks{0}, tr_prep_us{0}, tr_issue_us{0}, tr_sync_us{0};
    std::atomic<uint64_t> tr_gpu_ns[4] = {};  // device time of the first chunk: H2D | split+encode | parity D2H | tags + D2H
    // test hook: fail the n-th staged operation (see garage_ec_debug_fail_after)
    std::mutex misc_mu;  // timing list, last_error
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    std::vector<cudaEvent_t> free_events;
    std::atomic<uint64_t> launches{0};
    std::atomic<int> batch_copy_ok{1};  // cudaMemcpyBatchAsync usable (cleared on first failure)
    // generalized-RS structure of P (garage_ec_correct): log of locator X_r and of column multiplier v_r
    bool grs_ok = false;
    uint8_t grs_logx[kMaxK + kMaxM] = {0}, grs_logv[kMaxK + kMaxM] = {0};
    char last_error[256] = {0};
};

namespace {

int set_cuda_error(garage_ec_ctx *ctx, cudaError_t e, const char *what)
{
    if (ctx) {
        std::lock_guard<std::mutex> g(ctx->misc_mu);
        snprintf(ctx->last_error, sizeof(ctx->last_error), "%s: %s", what, cudaGetErrorString(e));
    }
    (void)cudaGetLastError();  // clear sticky-less errors
    return e == cudaErrorMemoryAllocation ? GARAGE_EC_E_NOMEM : GARAGE_EC_E_CUDA;
}

// test hook (garage_ec_debug_fail_after): the n-th checked runtime call from now fails
inline bool fault_hit(garage_ec_ctx *ctx)
{
    if (!ctx || ctx->fault_countdown.load(std::memory_order_relaxed) < 0) return false;
    return ctx->fault_countdown.fetch_sub(1, std::memory_order_relaxed) == 0;
}

#define CU_TRY(ctx, expr)                                                                          \
    do {                                                                                           \
        if (fault_hit(ctx)) return set_cuda_error(ctx, cudaErrorUnknown, "injected fault at " #expr); \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess) return set_cuda_error(ctx, e__, #expr);                            \
    } while (0)

// wait for everything queued on a lane (see garage_ec_ctx::wait_blocking)
inline cudaError_t lane_wait(garage_ec_ctx *ctx, HostLane &L)
{
    if (!ctx->wait_blocking.load(std::memory_order_relaxed)) return cudaStreamSynchronize(L.stream);
    cudaError_t e = cudaSuccess;
    if (!L.done) e = cudaEventCreateWithFlags(&L.done, cudaEventBlockingSync | cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventRecord(L.done, L.stream);
    if (e == cudaSuccess) e = cudaEventSynchronize(L.done);
    return e;
}

// Lease of one lane set for the duration of a HOST-mode call.  The destructor waits for every
// lane stream BEFORE the set goes back to the pool -- and therefore before the entry point
// returns, on every path including the early error returns: no DMA touches the caller's buffers
// after a HOST call has returned ("the library keeps no pointer", include/garage_ec.h).
struct LaneLease {
    garage_ec_ctx *ctx;
    LaneSet *set = nullptr;
    explicit LaneLease(garage_ec_ctx *c) : ctx(c)
    {
        std::unique_lock<std::mutex> lk(ctx->pool_mu);
        ctx->pool_cv.wait(lk, [&] { return !ctx->free_sets.empty() || ctx->n_sets < kMaxLaneSets; });
        if (!ctx->free_sets.empty()) {
            set = ctx->free_sets.back();
            ctx->free_sets.pop_back();
        } else {
            set = new (std::nothrow) LaneSet();
            if (set) ctx->n_sets++;
        }
    }
    ~LaneLease()
    {
        if (!set) return;
        for (HostLane &L : set->lanes)
            if (L.stream) (void)cudaStreamSynchronize(L.stream);
        (void)cudaGetLastError();
        {
            std::lock_guard<std::mutex> lk(ctx->pool_mu);
            ctx->free_sets.push_back(set);
        }
        ctx->pool_cv.notify_one();
    }
    LaneLease(const LaneLease &) = delete;
    LaneLease &operator=(const LaneLease &) = delete;
    HostLane &operator[](size_t i) { return set->lanes[i]; }
};
#define LEASE_LANES(ctx, name)  \
    LaneLease name(ctx);        \
    if (!name.set) return GARAGE_EC_E_NOMEM

// ---- NUMA placement of the GPU ------------------------------------------------------------
// 8-GPU hosts hang 4 GPUs off each socket; pinned buffers that land on the other socket cross
// the inter-socket link on every DMA (round 1: e2e weak scaling 0.65 at 8 GPUs with unplaced
// buffers).  The node comes from sysfs, the CPU list of the node likewise; no libnuma.
#ifndef MPOL_PREFERRED
#define MPOL_DEFAULT 0
#define MPOL_PREFERRED 1
#endif
bool read_small_file(const char *path, char *buf, size_t cap)
{
    FILE *f = fopen(path, "r");
    if (!f) return false;
    const size_t n = fread(buf, 1, cap - 1, f);
    fclose(f);
    buf[n] = 0;
    return n > 0;
}
bool parse_cpulist(const char *s, cpu_set_t *out)
{
    CPU_ZERO(out);
    bool any = false;
    while (*s) {
        while (*s == ',' || isspace((unsigned char)*s)) s++;
        if (!isdigit((unsigned char)*s)) break;
        char *e;
        long a = strtol(s, &e, 10), b = a;
        if (*e == '-') b = strtol(e + 1, &e, 10);
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) {
            CPU_SET((int)c, out);
            any = true;
        }
        s = e;
    }
    return any;
}
void probe_numa(garage_ec_ctx *ctx)
{
    char busid[64] = {0}, path[160], buf[4096];
    if (cudaDeviceGetPCIBusId(busid, sizeof(busid), ctx->device) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    for (char *c = busid; *c; c++) *c = (char)tolower((unsigned char)*c);
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", busid);
    if (!read_small_file(path, buf, sizeof(buf))) return;
    const int node = atoi(buf);
    if (node < 0) return;
    ctx->numa_node = node;
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
    if (read_small_file(path, buf, sizeof(buf))) ctx->have_node_cpus = parse_cpulist(buf, &ctx->node_cpus);
}
// node a page lives on (move_pages with nodes == NULL only queries), -1 if unknown
int node_of_page(void *p)
{
    int status = -1;
    void *pages[1] = {p};
    if (syscall(SYS_move_pages, 0, 1ul, pages, nullptr, &status, 0) != 0) return -1;
    return status;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

int check_geometry(const garage_ec_ctx *ctx, size_t stride, size_t n, int shards_per_stripe)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    if (stride == 0 || (stride & 15)) return GARAGE_EC_E_ALIGN;
    if ((unsigned long long)stride * (unsigned long long)shards_per_stripe >= (1ull << 32))
        return GARAGE_EC_E_INVALID;
    if (n > 0xffffffffull) return GARAGE_EC_E_INVALID;
    return GARAGE_EC_OK;
}

// ---- timing ---------------------------------------------------------------------------
struct TimedLaunch {
    garage_ec_ctx *ctx;
    cudaStream_t st;
    cudaEvent_t a = nullptr, b = nullptr;
    TimedLaunch(garage_ec_ctx *c, cudaStream_t s) : ctx(c), st(s)
    {
        if (!ctx->timing) return;
        std::lock_guard<std::mutex> g(ctx->misc_mu);
        for (cudaEvent_t *e : {&a, &b}) {
            if (!ctx->free_events.empty()) {
                *e = ctx->free_events.back();
                ctx->free_events.pop_back();
            } else if (cudaEventCreate(e) != cudaSuccess) {
                *e = nullptr;
            }
        }
        if (a && b) cudaEventRecord(a, st);
    }
    ~TimedLaunch()
    {
        if (!a || !b) return;
        cudaEventRecord(b, st);
        std::lock_guard<std::mutex> g(ctx->misc_mu);
        ctx->pending.emplace_back(a, b);
    }
};

// ---- kernel dispatch --------------------------------------------------------------------
// Launch shape, table layout and shared-memory carve-up are compile-time functions of (k, mode):
// StreamCfg in rs_kernels.cuh.
template <int K, int MODE>
cudaError_t launch_apply_t(const garage_ec_ctx *ctx, const ApplyParams &p, cudaStream_t st)
{
    static std::atomic<int> configured_for_device{-1};  // per instantiation
    using CFG = StreamCfg<K, MODE>;
    auto kern = rs_apply_kernel<K, MODE>;
    if ((size_t)CFG::kSmem > ctx->smem_optin) return cudaErrorInvalidConfiguration;
    // opt-in shared memory size is a per-function, per-device attribute; setting it is cheap
    // but not free, so remember the last device it was set for.
    if (configured_for_device.load(std::memory_order_acquire) != ctx->device) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CFG::kSmem);
        if (e != cudaSuccess) return e;
        configured_for_device.store(ctx->device, std::memory_order_release);
    }
    kern<<<ctx->sm_count, CFG::kThreads, CFG::kSmem, st>>>(p);
    return cudaGetLastError();
}

template <int MODE>
cudaError_t launch_apply(garage_ec_ctx *ctx, const ApplyParams &p, cudaStream_t st)
{
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    switch (p.k) {
#define GEC_CASE(KK) case KK: return launch_apply_t<KK, MODE>(ctx, p, st);
#ifndef GEC_FAST_BUILD
        GEC_CASE(1) GEC_CASE(2) GEC_CASE(3) GEC_CASE(4) GEC_CASE(5) GEC_CASE(6) GEC_CASE(7) GEC_CASE(8)
        GEC_CASE(9) GEC_CASE(11) GEC_CASE(12) GEC_CASE(13) GEC_CASE(14) GEC_CASE(15) GEC_CASE(16)
        GEC_CASE(17) GEC_CASE(18) GEC_CASE(19) GEC_CASE(20) GEC_CASE(21) GEC_CASE(22) GEC_CASE(23) GEC_CASE(24)
        GEC_CASE(25) GEC_CASE(26) GEC_CASE(27) GEC_CASE(28) GEC_CASE(29) GEC_CASE(30) GEC_CASE(31) GEC_CASE(32)
#endif
        GEC_CASE(10)
#if defined(GEC_FAST_BUILD) && GEC_FAST_BUILD != 10
        GEC_CASE(GEC_FAST_BUILD)
#endif
#undef GEC_CASE
    default: return cudaErrorInvalidConfiguration;
    }
}

uint32_t items_per_stripe(size_t stride) { return (uint32_t)((stride / 16 + 31) / 32); }

// cuTensorMapEncodeTiled through the runtime (no link against libcuda)
using TensorMapEncodeFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                       const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TensorMapEncodeFn tensor_map_encoder()
{
    static std::atomic<void *> cached{nullptr};
    static std::atomic<int> tried{0};
    if (!tried.load(std::memory_order_acquire)) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            fn = nullptr;
        (void)cudaGetLastError();
        cached.store(fn, std::memory_order_release);
        tried.store(1, std::memory_order_release);
    }
    return reinterpret_cast<TensorMapEncodeFn>(cached.load(std::memory_order_acquire));
}
// 2-D view of a shard array for the TMA path of the uniform kernels: dim0 = stride/4 uint32, dim1 = rows shards.
// false = no tensor map (the kernel then issues one 1-D bulk copy per row)
bool make_src_tensor_map(CUtensorMap *tm, const uint8_t *src, size_t stride, size_t rows, int box_rows)
{
#if GEC_TMAP
    TensorMapEncodeFn enc = tensor_map_encoder();
    if (!enc || stride < kStageRowBytes || rows == 0 || rows > 0xffffffffull || box_rows > 256) return false;
    const cuuint64_t gdim[2] = {(cuuint64_t)(stride / 4), (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)stride};
    const cuuint32_t box[2] = {kStageRowBytes / 4, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<uint8_t *>(src), gdim, gstride, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
#else
    (void)tm, (void)src, (void)stride, (void)rows, (void)box_rows;
    return false;
#endif
}

// Device-resident encode (mode 0) / verify (mode 2) of n stripes, split so that
// n * items_per_stripe stays below 2^32 and m > 4 runs in passes of 4 rows.
int run_uniform(garage_ec_ctx *ctx, int mode, const uint8_t *src, size_t src_pitch, uint8_t *dst,
                size_t dst_pitch, uint32_t *mismatch, const uint32_t *shard_len, size_t stride,
                size_t n, cudaStream_t st, bool allow_tmap = true)
{
    const uint32_t ips = items_per_stripe(stride);
    const size_t max_n = 0xffffffffull / ips;
    TimedLaunch tl(ctx, st);
    for (size_t s0 = 0; s0 < n; s0 += max_n) {
        const size_t cnt = n - s0 < max_n ? n - s0 : max_n;
        for (int r0 = 0; r0 < ctx->m; r0 += kRowsPerPass) {
            ApplyParams p;
            memset(&p, 0, sizeof(p));
            p.src = src + s0 * src_pitch;
            p.src_pitch = src_pitch;
            p.dst = dst ? dst + s0 * dst_pitch + (size_t)r0 * stride : nullptr;
            p.dst_pitch = dst_pitch;
            p.shard_len = shard_len ? shard_len + s0 : nullptr;
            p.mismatch = mismatch ? mismatch + s0 : nullptr;
            p.stride = (uint32_t)stride;
            p.n = (uint32_t)cnt;
            p.k = (uint32_t)ctx->k;
            p.rows = (uint32_t)(ctx->m - r0 < kRowsPerPass ? ctx->m - r0 : kRowsPerPass);
            p.row_off = (uint32_t)r0;
            p.items_per_stripe = ips;
            p.row_bytes = 128;
            p.rows_per_stripe = (uint32_t)(src_pitch / stride);
            p.use_tmap = (allow_tmap && GEC_TMAP && ctx->k >= GEC_TMAP_FROM_K && make_src_tensor_map(&p.tmap, p.src, stride, cnt * p.rows_per_stripe,
                                              (GEC_SPLIT_STAGE && ctx->k > 16) ? 16 : ctx->k)) ? 1u : 0u;  // box rows: StreamCfg::kSrcRows
            for (uint32_t i = 0; i < p.rows; i++)
                memcpy(p.coef + i * ctx->k, ctx->P + (r0 + i) * ctx->k, ctx->k);
            cudaError_t e = mode == kModeEncode ? launch_apply<kModeEncode>(ctx, p, st)
                                                : launch_apply<kModeVerify>(ctx, p, st);
            if (e != cudaSuccess) return set_cuda_error(ctx, e, "rs_apply_kernel launch");
        }
    }
    return GARAGE_EC_OK;
}

// Device-resident reconstruct.  plan/counter scratch supplied by the caller (device).
int run_reconstruct(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present, const uint8_t *want,
                    int32_t *status, const uint32_t *shard_len, size_t stride, size_t n,
                    StripePlan *plan, uint32_t *counter, cudaStream_t st, bool present_is_bad = false)
{
    PlanParams q;
    memset(&q, 0, sizeof(q));
    q.present = present;
    q.want = want;
    q.status = status;
    q.plan = plan;
    q.counter = counter;
    q.n = (uint32_t)n;
    q.k = (uint32_t)ctx->k;
    q.m = (uint32_t)ctx->m;
    q.present_is_bad = present_is_bad ? 1u : 0u;
    memcpy(q.P, ctx->P, (size_t)ctx->k * ctx->m);
    const unsigned blocks = (unsigned)((n + kPlanWarps - 1) / kPlanWarps);
    rs_plan_kernel<<<blocks, kPlanWarps * 32, 0, st>>>(q);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "rs_plan_kernel launch");

    TimedLaunch tl(ctx, st);
    const size_t pitch = (size_t)(ctx->k + ctx->m) * stride;
    for (int r0 = 0; r0 < ctx->m; r0 += kRowsPerPass) {
        if (r0 > 0) {
            e = cudaMemsetAsync(counter, 0, sizeof(uint32_t), st);
            if (e != cudaSuccess) return set_cuda_error(ctx, e, "cudaMemsetAsync(counter)");
        }
        ApplyParams p;
        memset(&p, 0, sizeof(p));
        p.src = shards;
        p.dst = shards;
        p.src_pitch = p.dst_pitch = pitch;
        p.shard_len = shard_len;
        p.plan = plan;
        p.counter = counter;
        p.stride = (uint32_t)stride;
        p.n = (uint32_t)n;
        p.k = (uint32_t)ctx->k;
        p.row_off = (uint32_t)r0;
        p.row_bytes = 128;
        e = launch_apply<kModePlan>(ctx, p, st);
        if (e != cudaSuccess) return set_cuda_error(ctx, e, "rs_apply_kernel<plan> launch");
    }
    return GARAGE_EC_OK;
}

size_t plan_scratch_bytes(size_t n) { return n * sizeof(StripePlan) + 16; }

// ---- error-locating decode (garage_ec_correct) --------------------------------------------
// scratch: mismatch[n] | list[n] | bad[n] | count | err_mask[n]
inline size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }
size_t correct_scratch_bytes(size_t n) { return 3 * align16(n * 4) + 16 + n * 8; }

template <int M>
cudaError_t launch_correct_t(garage_ec_ctx *ctx, const CorrectParams &cp, cudaStream_t st)
{
    const unsigned grid = (unsigned)ctx->sm_count * 8;  // persistent: the number of listed stripes is only known on the device
    rs_correct_scan_kernel<M><<<grid, kCorrectThreads, 0, st>>>(cp);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    rs_correct_apply_kernel<M><<<grid, kCorrectThreads, 0, st>>>(cp);
    ctx->launches.fetch_add(2, std::memory_order_relaxed);
    return cudaGetLastError();
}

// Device-resident correct of n stripes: check (verify kernel), list, scan, apply -- all stream ordered.
int run_correct(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present, int32_t *status, uint8_t *fixed,
                const uint32_t *shard_len, size_t stride, size_t n, uint8_t *scratch, cudaStream_t st)
{
    const size_t tot = ctx->k + ctx->m;
    uint32_t *mismatch = reinterpret_cast<uint32_t *>(scratch);
    uint32_t *list = reinterpret_cast<uint32_t *>(scratch + align16(n * 4));
    uint32_t *bad = reinterpret_cast<uint32_t *>(scratch + 2 * align16(n * 4));
    uint32_t *count = reinterpret_cast<uint32_t *>(scratch + 3 * align16(n * 4));
    auto *err_mask = reinterpret_cast<unsigned long long *>(scratch + 3 * align16(n * 4) + 16);
    cudaError_t e = cudaMemsetAsync(mismatch, 0, n * 4, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(count, 0, 4, st);
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "cudaMemsetAsync(correct scratch)");
    int rc = run_uniform(ctx, kModeVerify, shards, tot * stride, nullptr, 0, mismatch, shard_len, stride, n, st);
    if (rc) return rc;
    CorrectParams cp;
    memset(&cp, 0, sizeof(cp));
    cp.shards = shards;
    cp.present = present;
    cp.shard_len = shard_len;
    cp.mismatch = mismatch;
    cp.status = status;
    cp.fixed = fixed;
    cp.list = list;
    cp.count = count;
    cp.err_mask = err_mask;
    cp.bad = bad;
    cp.stride = (uint32_t)stride;
    cp.n = (uint32_t)n;
    cp.k = (uint32_t)ctx->k;
    cp.m = (uint32_t)ctx->m;
    cp.items_per_stripe = (uint32_t)((stride + kCorrectThreads - 1) / kCorrectThreads);
    memcpy(cp.logx, ctx->grs_logx, tot);
    memcpy(cp.logv, ctx->grs_logv, tot);
    rs_correct_list_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(cp);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "rs_correct_list_kernel launch");
    switch (ctx->m) {
    case 1: e = launch_correct_t<1>(ctx, cp, st); break;
    case 2: e = launch_correct_t<2>(ctx, cp, st); break;
    case 3: e = launch_correct_t<3>(ctx, cp, st); break;
    case 4: e = launch_correct_t<4>(ctx, cp, st); break;
    case 5: e = launch_correct_t<5>(ctx, cp, st); break;
    case 6: e = launch_correct_t<6>(ctx, cp, st); break;
    case 7: e = launch_correct_t<7>(ctx, cp, st); break;
    case 8: e = launch_correct_t<8>(ctx, cp, st); break;
    default: e = cudaErrorInvalidConfiguration;
    }
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "rs_correct kernels launch");
    return GARAGE_EC_OK;
}

// ---- batched async copies ---------------------------------------------------------------
// Reconstruct moves many shard-sized pieces per stripe (only the k survivors go up, only the
// rebuilt shards come back).  One cudaMemcpyBatchAsync per chunk instead of thousands of
// cudaMemcpyAsync calls keeps the CPU off the critical path; adjacent pieces are merged.
struct CopyBatch {
    std::vector<void *> dst, src;
    std::vector<size_t> sz;
    void add(void *d, const void *s, size_t n)
    {
        if (!n) return;
        if (!dst.empty() && static_cast<uint8_t *>(dst.back()) + sz.back() == d &&
            static_cast<const uint8_t *>(src.back()) + sz.back() == s) {
            sz.back() += n;
            return;
        }
        dst.push_back(d);
        src.push_back(const_cast<void *>(s));
        sz.push_back(n);
    }
    int flush(garage_ec_ctx *ctx, cudaMemcpyKind kind, cudaStream_t st)
    {
        const size_t cnt = dst.size();
        if (!cnt) return GARAGE_EC_OK;
        if (fault_hit(ctx)) {
            dst.clear();
            src.clear();
            sz.clear();
            return set_cuda_error(ctx, cudaErrorUnknown, "injected fault at batched copy");
        }
        bool done = false;
        if (cnt > 1 && ctx->batch_copy_ok.load(std::memory_order_relaxed)) {
            cudaMemcpyAttributes attr;
            memset(&attr, 0, sizeof(attr));
            attr.srcAccessOrder = cudaMemcpySrcAccessOrderStream;
            size_t attr_idx = 0, fail = 0;
            cudaError_t e = cudaMemcpyBatchAsync(dst.data(), src.data(), sz.data(), cnt, &attr, &attr_idx, 1,
                                                 &fail, st);
            if (e == cudaSuccess) {
                done = true;
            } else {
                (void)cudaGetLastError();
                ctx->batch_copy_ok.store(0, std::memory_order_relaxed);
            }
        }
        if (!done)
            for (size_t i = 0; i < cnt; i++) CU_TRY(ctx, cudaMemcpyAsync(dst[i], src[i], sz[i], kind, st));
        dst.clear();
        src.clear();
        sz.clear();
        return GARAGE_EC_OK;
    }
};

// ---- host lanes -----------------------------------------------------------------------
// A lane's buffers are sized for a full pipeline chunk the first time they are needed (not for the
// batch at hand): a batching front-end calls with a different number of blocks every time, and every
// cudaFree + cudaMalloc to grow a lane synchronises the whole device -- with growth-on-demand the first few
// hundred calls of a fresh context paid milliseconds each (profiles/r02_summary.md, block-manager bench)
constexpr size_t kLaneFloorBytes = 128ull << 20, kLaneSmallFloorBytes = 2ull << 20;
int lane_reserve(garage_ec_ctx *ctx, HostLane &L, size_t buf_bytes, size_t small_bytes)
{
    if (buf_bytes < kLaneFloorBytes) buf_bytes = kLaneFloorBytes;
    if (small_bytes < kLaneSmallFloorBytes) small_bytes = kLaneSmallFloorBytes;
    if (!L.stream) CU_TRY(ctx, cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
    if (L.d_cap < buf_bytes) {
        if (L.d_buf) cudaFree(L.d_buf);
        L.d_buf = nullptr;
        L.d_cap = 0;
        CU_TRY(ctx, cudaMalloc(&L.d_buf, buf_bytes));
        L.d_cap = buf_bytes;
    }
    if (L.small_cap < small_bytes) {
        if (L.d_small) cudaFree(L.d_small);
        L.d_small = nullptr;
        L.small_cap = 0;
        CU_TRY(ctx, cudaMalloc(&L.d_small, small_bytes));
        L.small_cap = small_bytes;
    }
    return GARAGE_EC_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int create_common(garage_ec_ctx **out, int device, int k, int m, const uint8_t *P, int kind)
{
    if (!out) return GARAGE_EC_E_INVALID;
    *out = nullptr;
    if (k < 1 || k > kMaxK || m < 1 || m > kMaxM) return GARAGE_EC_E_INVALID;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        (void)cudaGetLastError();
        return GARAGE_EC_E_NODEVICE;
    }
    if (device < 0 || device >= ndev) return GARAGE_EC_E_NODEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return GARAGE_EC_E_NODEVICE;
    if (prop.major != 10) return GARAGE_EC_E_NODEVICE;  // built for sm_100a only
    garage_ec_ctx *ctx = new (std::nothrow) garage_ec_ctx();
    if (!ctx) return GARAGE_EC_E_NOMEM;
    ctx->device = device;
    ctx->k = k;
    ctx->m = m;
    if (P) {
        memcpy(ctx->P, P, (size_t)k * m);
    } else if (!h_build_matrix(k, m, kind, ctx->P)) {
        delete ctx;
        return GARAGE_EC_E_INVALID;
    }
    {
        uint8_t v[kMaxK + kMaxM];
        ctx->grs_ok = h_grs_multipliers(k, m, ctx->P, v);
        for (int r = 0; ctx->grs_ok && r < k + m; r++) {
            ctx->grs_logx[r] = h_gf_log[(uint8_t)(r ^ kLocShift)];
            ctx->grs_logv[r] = h_gf_log[v[r]];
        }
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaSetDevice(device) != cudaSuccess) {
        delete ctx;
        return GARAGE_EC_E_NODEVICE;
    }
    {
        cudaMemPoolProps props;
        memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&ctx->pool, &props) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            (void)cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep);
        } else {
            ctx->pool = nullptr;  // fall back to the default pool
        }
        (void)cudaGetLastError();
    }
    probe_numa(ctx);
    ctx->trace = getenv("GARAGE_EC_TRACE") != nullptr;
    if (const char *b = getenv("GARAGE_EC_BATCHCOPY")) ctx->batch_copy_ok.store(b[0] != '0');
    if (const char *z = getenv("GARAGE_EC_ZEROCOPY")) ctx->zero_copy_rec = ctx->zero_copy_enc = z[0] == '1';
    *out = ctx;
    return GARAGE_EC_OK;
}

}  // namespace

// ======================================================================= C ABI
extern "C" {

int garage_ec_abi_version(void) { return GARAGE_EC_ABI_VERSION; }

const char *garage_ec_strerror(int code)
{
    switch (code) {
    case GARAGE_EC_OK: return "ok";
    case GARAGE_EC_E_INVALID: return "invalid argument or geometry";
    case GARAGE_EC_E_CUDA: return "CUDA runtime error";
    case GARAGE_EC_E_NOMEM: return "out of memory";
    case GARAGE_EC_E_UNRECOVERABLE: return "stripe unrecoverable: fewer than k shards present";
    case GARAGE_EC_E_NODEVICE: return "no usable sm_100 CUDA device (no CPU fallback)";
    case GARAGE_EC_E_ALIGN: return "pointer or stride not 16-byte aligned";
    case GARAGE_EC_E_UNCORRECTABLE: return "stripe uncorrectable: a column has more wrong shards than the parity can locate";
    default: return "unknown error";
    }
}

int garage_ec_create(garage_ec_ctx **out, int cuda_device, int k, int m, int matrix_kind)
{
    if (matrix_kind != GARAGE_EC_VANDERMONDE && matrix_kind != GARAGE_EC_CAUCHY) {
        if (out) *out = nullptr;
        return GARAGE_EC_E_INVALID;
    }
    if (matrix_kind == GARAGE_EC_CAUCHY && k + m > 256) return GARAGE_EC_E_INVALID;
    return create_common(out, cuda_device, k, m, nullptr, matrix_kind);
}

int garage_ec_create_with_matrix(garage_ec_ctx **out, int cuda_device, int k, int m,
                                 const uint8_t *parity_rows)
{
    if (!parity_rows) {
        if (out) *out = nullptr;
        return GARAGE_EC_E_INVALID;
    }
    return create_common(out, cuda_device, k, m, parity_rows, 0);
}

void garage_ec_destroy(garage_ec_ctx *ctx)
{
    if (!ctx) return;
    if (ctx->trace && ctx->tr_calls.load())
        fprintf(stderr, "garage_ec trace ctx %p: encode_blocks calls=%llu blocks=%llu  per call: prep %.1f us, issue %.1f us, sync %.1f us\n",
                (void *)ctx, (unsigned long long)ctx->tr_calls.load(), (unsigned long long)ctx->tr_blocks.load(),
                (double)ctx->tr_prep_us.load() / ctx->tr_calls.load(), (double)ctx->tr_issue_us.load() / ctx->tr_calls.load(),
                (double)ctx->tr_sync_us.load() / ctx->tr_calls.load());
    if (ctx->trace && ctx->tr_calls.load())
        fprintf(stderr, "    device time of the first chunk per call: H2D %.1f us, split+encode %.1f us, parity D2H %.1f us, tags+D2H %.1f us\n",
                ctx->tr_gpu_ns[0].load() / 1e3 / ctx->tr_calls.load(), ctx->tr_gpu_ns[1].load() / 1e3 / ctx->tr_calls.load(),
                ctx->tr_gpu_ns[2].load() / 1e3 / ctx->tr_calls.load(), ctx->tr_gpu_ns[3].load() / 1e3 / ctx->tr_calls.load());
    cudaSetDevice(ctx->device);
    for (LaneSet *set : ctx->free_sets) {
        for (HostLane &L : set->lanes) {
            if (L.stream) {
                cudaStreamSynchronize(L.stream);
                cudaStreamDestroy(L.stream);
            }
            if (L.d_buf) cudaFree(L.d_buf);
            if (L.d_small) cudaFree(L.d_small);
            if (L.done) cudaEventDestroy(L.done);
        }
        delete set;
    }
    for (auto &pr : ctx->pending) {
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    for (cudaEvent_t e : ctx->free_events) cudaEventDestroy(e);
    if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
    delete ctx;
}

int garage_ec_matrix(const garage_ec_ctx *ctx, uint8_t *out_m_by_k)
{
    if (!ctx || !out_m_by_k) return GARAGE_EC_E_INVALID;
    memcpy(out_m_by_k, ctx->P, (size_t)ctx->k * ctx->m);
    return GARAGE_EC_OK;
}

int garage_ec_params(const garage_ec_ctx *ctx, int *k, int *m, int *cuda_device)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    if (k) *k = ctx->k;
    if (m) *m = ctx->m;
    if (cuda_device) *cuda_device = ctx->device;
    return GARAGE_EC_OK;
}

const char *garage_ec_last_error(const garage_ec_ctx *ctx) { return ctx ? ctx->last_error : ""; }

uint32_t garage_ec_shard_len(uint32_t block_len, int k)
{
    if (k < 1) return 0;
    return (uint32_t)(((unsigned long long)block_len + (unsigned)k - 1) / (unsigned)k);
}

size_t garage_ec_stride_for(uint32_t shard_len) { return align_up(shard_len ? shard_len : 1, 128); }

uint64_t garage_ec_launch_count(const garage_ec_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

int garage_ec_set_timing(garage_ec_ctx *ctx, int enabled)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    std::lock_guard<std::mutex> g(ctx->misc_mu);
    ctx->timing = enabled != 0;
    return GARAGE_EC_OK;
}

int garage_ec_timing_read(garage_ec_ctx *ctx, double *total_ms, uint64_t *launches)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    cudaSetDevice(ctx->device);
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> todo;
    {
        std::lock_guard<std::mutex> g(ctx->misc_mu);
        todo.swap(ctx->pending);
    }
    double sum = 0;
    uint64_t cnt = 0;
    int rc = GARAGE_EC_OK;
    for (auto &pr : todo) {
        float ms = 0;
        cudaError_t e = cudaEventSynchronize(pr.second);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, pr.first, pr.second);
        if (e == cudaSuccess) {
            sum += ms;
            cnt++;
        } else {
            rc = set_cuda_error(ctx, e, "timing event");
        }
    }
    {
        std::lock_guard<std::mutex> g(ctx->misc_mu);
        for (auto &pr : todo) {
            ctx->free_events.push_back(pr.first);
            ctx->free_events.push_back(pr.second);
        }
    }
    if (total_ms) *total_ms = sum;
    if (launches) *launches = cnt;
    return rc;
}

static int host_alloc_impl(garage_ec_ctx *ctx, void **out, size_t bytes, unsigned extra_flags);

int garage_ec_host_alloc(garage_ec_ctx *ctx, void **out, size_t bytes) { return host_alloc_impl(ctx, out, bytes, 0); }

int garage_ec_host_alloc_wc(garage_ec_ctx *ctx, void **out, size_t bytes)
{
    return host_alloc_impl(ctx, out, bytes, cudaHostAllocWriteCombined);
}

static int host_alloc_impl(garage_ec_ctx *ctx, void **out, size_t bytes, unsigned extra_flags)
{
    if (!ctx || !out || !bytes) return GARAGE_EC_E_INVALID;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    // Place the pages on the GPU's NUMA node: the driver allocates and pins them inside this call,
    // under the calling thread's memory policy and CPU.  Both are set for the duration of the call
    // (preferred-node policy; where the sandbox forbids set_mempolicy, running on a CPU of the node
    // gives the same result through the default local-allocation policy) and restored afterwards.
    cpu_set_t saved_cpus;
    bool moved = false, policy_set = false;
    if (ctx->numa_node >= 0) {
        unsigned long mask[16] = {0};
        if (ctx->numa_node < (int)(sizeof(mask) * 8)) {
            mask[ctx->numa_node / (8 * sizeof(unsigned long))] |= 1ul << (ctx->numa_node % (8 * sizeof(unsigned long)));
            policy_set = syscall(SYS_set_mempolicy, MPOL_PREFERRED, mask, sizeof(mask) * 8) == 0;
        }
        if (ctx->have_node_cpus && sched_getaffinity(0, sizeof(saved_cpus), &saved_cpus) == 0) {
            cpu_set_t want;
            CPU_AND(&want, &saved_cpus, &ctx->node_cpus);
            if (CPU_COUNT(&want) > 0 && sched_setaffinity(0, sizeof(want), &want) == 0) moved = true;
        }
    }
    cudaError_t e = fault_hit(ctx) ? cudaErrorMemoryAllocation : cudaHostAlloc(out, bytes, cudaHostAllocPortable | extra_flags);
    if (moved) sched_setaffinity(0, sizeof(saved_cpus), &saved_cpus);
    if (policy_set) syscall(SYS_set_mempolicy, MPOL_DEFAULT, nullptr, 0ul);
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "cudaHostAlloc");
    ctx->last_alloc_node = node_of_page(*out);
    return GARAGE_EC_OK;
}

int garage_ec_numa_info(const garage_ec_ctx *ctx, int *gpu_node, int *last_alloc_node)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    if (gpu_node) *gpu_node = ctx->numa_node;
    if (last_alloc_node) *last_alloc_node = ctx->last_alloc_node;
    return GARAGE_EC_OK;
}

int garage_ec_bind_thread(const garage_ec_ctx *ctx)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    if (ctx->numa_node < 0 || !ctx->have_node_cpus) return 1;  // nothing known: leave the thread alone
    cpu_set_t cur, want;
    if (sched_getaffinity(0, sizeof(cur), &cur) != 0) return 1;
    CPU_AND(&want, &cur, &ctx->node_cpus);
    if (CPU_COUNT(&want) == 0) return 1;  // the cgroup does not allow any CPU of that node
    return sched_setaffinity(0, sizeof(want), &want) == 0 ? GARAGE_EC_OK : 1;
}

void garage_ec_host_free(garage_ec_ctx *ctx, void *ptr)
{
    if (!ctx || !ptr) return;
    cudaSetDevice(ctx->device);
    cudaFreeHost(ptr);
}

int garage_ec_fill_random(garage_ec_ctx *ctx, uint8_t *dst_device, size_t len, uint64_t seed,
                          uint64_t offset, void *cuda_stream)
{
    if (!ctx || !dst_device || (len & 7) || (offset & 7) ||
        (reinterpret_cast<uintptr_t>(dst_device) & 7))
        return GARAGE_EC_E_INVALID;
    if (!len) return GARAGE_EC_OK;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    fill_random_kernel<<<ctx->sm_count * 8, 256, 0, (cudaStream_t)cuda_stream>>>(
        reinterpret_cast<unsigned long long *>(dst_device), len / 8, seed, offset / 8);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    CU_TRY(ctx, cudaGetLastError());
    return GARAGE_EC_OK;
}

// --------------------------------------------------------------------------- ENCODE
// pinned host memory the device addresses through the same pointer (cudaHostAlloc / cudaHostRegister under UVA)
static bool device_addressable_host(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost && a.devicePointer == p;
}

static int encode_host(garage_ec_ctx *ctx, const uint8_t *data, uint8_t *parity,
                       const uint32_t *shard_len, size_t stride, size_t n)
{
    LEASE_LANES(ctx, lanes);
    if (ctx->zero_copy_enc && device_addressable_host(data) && device_addressable_host(parity)) {
        // one launch over the whole batch: the TMA / vector loads pull the data shards across PCIe, the parity stores
        // go straight to the caller's buffer -- no staging copies, no chunk boundaries
        HostLane &L = lanes[0];
        int rc = lane_reserve(ctx, L, 0, align_up(n * 4, 16));
        if (rc) return rc;
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small, shard_len, n * 4, cudaMemcpyHostToDevice, L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small);
        }
        rc = run_uniform(ctx, kModeEncode, data, ctx->k * stride, parity, ctx->m * stride, nullptr, d_len, stride, n, L.stream,
                         /*allow_tmap=*/false);
        if (rc) return rc;
        CU_TRY(ctx, lane_wait(ctx, L));
        return GARAGE_EC_OK;
    }
    const size_t k = ctx->k, m = ctx->m;
    size_t cs = kHostChunkBytes / (k * stride);
    if (cs < 1) cs = 1;
    if (cs > n) cs = n;
    const size_t in_b = cs * k * stride, out_b = cs * m * stride;
    for (HostLane &L : lanes.set->lanes) {
        int rc = lane_reserve(ctx, L, in_b + out_b, align_up(cs * 4, 16));
        if (rc) return rc;
    }
    size_t c = 0;
    for (size_t s0 = 0; s0 < n; s0 += cs, c++) {
        HostLane &L = lanes[c % kHostLanes];
        const size_t cnt = n - s0 < cs ? n - s0 : cs;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_buf, data + s0 * k * stride, cnt * k * stride,
                                    cudaMemcpyHostToDevice, L.stream));
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small, shard_len + s0, cnt * 4, cudaMemcpyHostToDevice,
                                        L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small);
        }
        int rc = run_uniform(ctx, kModeEncode, L.d_buf, k * stride, L.d_buf + in_b, m * stride,
                             nullptr, d_len, stride, cnt, L.stream);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(parity + s0 * m * stride, L.d_buf + in_b, cnt * m * stride,
                                    cudaMemcpyDeviceToHost, L.stream));
    }
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    return GARAGE_EC_OK;
}

int garage_ec_encode(garage_ec_ctx *ctx, const uint8_t *data, uint8_t *parity,
                     const uint32_t *shard_len, size_t stride, size_t n_stripes, int mem_kind,
                     void *cuda_stream)
{
    if (!ctx || (mem_kind != GARAGE_EC_MEM_HOST && mem_kind != GARAGE_EC_MEM_DEVICE))
        return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_stripes, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_stripes == 0) return GARAGE_EC_OK;
    if (!data || !parity) return GARAGE_EC_E_INVALID;
    if (!aligned16(data) || !aligned16(parity)) return GARAGE_EC_E_ALIGN;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (mem_kind == GARAGE_EC_MEM_HOST) return encode_host(ctx, data, parity, shard_len, stride, n_stripes);
    return run_uniform(ctx, kModeEncode, data, (size_t)ctx->k * stride, parity, (size_t)ctx->m * stride,
                       nullptr, shard_len, stride, n_stripes, (cudaStream_t)cuda_stream);
}

// --------------------------------------------------------------------------- VERIFY
static int verify_host(garage_ec_ctx *ctx, const uint8_t *shards, uint32_t *mismatch,
                       const uint32_t *shard_len, size_t stride, size_t n)
{
    LEASE_LANES(ctx, lanes);
    const size_t tot = ctx->k + ctx->m;
    size_t cs = kHostChunkBytes / (tot * stride);
    if (cs < 1) cs = 1;
    if (cs > n) cs = n;
    const size_t small = align_up(cs * 4, 16);
    for (HostLane &L : lanes.set->lanes) {
        int rc = lane_reserve(ctx, L, cs * tot * stride, 2 * small);
        if (rc) return rc;
    }
    size_t c = 0;
    for (size_t s0 = 0; s0 < n; s0 += cs, c++) {
        HostLane &L = lanes[c % kHostLanes];
        const size_t cnt = n - s0 < cs ? n - s0 : cs;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_buf, shards + s0 * tot * stride, cnt * tot * stride,
                                    cudaMemcpyHostToDevice, L.stream));
        uint32_t *d_mm = reinterpret_cast<uint32_t *>(L.d_small);
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + small, shard_len + s0, cnt * 4,
                                        cudaMemcpyHostToDevice, L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small + small);
        }
        CU_TRY(ctx, cudaMemsetAsync(d_mm, 0, cnt * 4, L.stream));
        int rc = run_uniform(ctx, kModeVerify, L.d_buf, tot * stride, nullptr, 0, d_mm, d_len, stride,
                             cnt, L.stream);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(mismatch + s0, d_mm, cnt * 4, cudaMemcpyDeviceToHost, L.stream));
    }
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    return GARAGE_EC_OK;
}

int garage_ec_verify(garage_ec_ctx *ctx, const uint8_t *shards, uint32_t *mismatch,
                     const uint32_t *shard_len, size_t stride, size_t n_stripes, int mem_kind,
                     void *cuda_stream)
{
    if (!ctx || (mem_kind != GARAGE_EC_MEM_HOST && mem_kind != GARAGE_EC_MEM_DEVICE))
        return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_stripes, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_stripes == 0) return GARAGE_EC_OK;
    if (!shards || !mismatch) return GARAGE_EC_E_INVALID;
    if (!aligned16(shards)) return GARAGE_EC_E_ALIGN;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (mem_kind == GARAGE_EC_MEM_HOST) return verify_host(ctx, shards, mismatch, shard_len, stride, n_stripes);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    CU_TRY(ctx, cudaMemsetAsync(mismatch, 0, n_stripes * 4, st));
    return run_uniform(ctx, kModeVerify, shards, (size_t)(ctx->k + ctx->m) * stride, nullptr, 0, mismatch,
                       shard_len, stride, n_stripes, st);
}

// --------------------------------------------------------------------------- RECONSTRUCT
// `stripes` != NULL: stripe s lives at stripes[s] (its k+m shards `stride` apart) instead of
// shards + s*(k+m)*stride -- the gather form used by batching front-ends whose callers each own
// a pinned slot (garage_ec_reconstruct_stripes)
static int reconstruct_host(garage_ec_ctx *ctx, uint8_t *shards, uint8_t *const *stripes, const uint8_t *present,
                            const uint8_t *want, int32_t *status, const uint32_t *shard_len,
                            size_t stride, size_t n)
{
    auto shard_at = [&](size_t s, size_t i) -> uint8_t * {
        return stripes ? stripes[s] + i * stride : shards + (s * (size_t)(ctx->k + ctx->m) + i) * stride;
    };
    // declared before the lane lease: they must outlive the stream work the lease waits for
    std::vector<int32_t> st_host(status ? 0 : n);
    CopyBatch up, down;
    LEASE_LANES(ctx, lanes);
    if (ctx->zero_copy_rec && !stripes && device_addressable_host(shards)) {
        // the kernel reads the k survivors of every stripe and writes the rebuilt shards in the caller's pinned buffer
        const size_t tot_ = ctx->k + ctx->m;
        const size_t zo_present = 0, zo_want = align_up(n * tot_, 16), zo_status = zo_want + align_up(n * tot_, 16);
        const size_t zo_len = zo_status + align_up(n * 4, 16), zo_plan = zo_len + align_up(n * 4, 16);
        HostLane &L = lanes[0];
        int rcz = lane_reserve(ctx, L, 0, zo_plan + plan_scratch_bytes(n));
        if (rcz) return rcz;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_small + zo_present, present, n * tot_, cudaMemcpyHostToDevice, L.stream));
        const uint8_t *d_want = nullptr;
        if (want) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + zo_want, want, n * tot_, cudaMemcpyHostToDevice, L.stream));
            d_want = L.d_small + zo_want;
        }
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + zo_len, shard_len, n * 4, cudaMemcpyHostToDevice, L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small + zo_len);
        }
        StripePlan *d_plan = reinterpret_cast<StripePlan *>(L.d_small + zo_plan);
        uint32_t *d_counter = reinterpret_cast<uint32_t *>(L.d_small + zo_plan + n * sizeof(StripePlan));
        rcz = run_reconstruct(ctx, shards, L.d_small + zo_present, d_want, reinterpret_cast<int32_t *>(L.d_small + zo_status), d_len,
                              stride, n, d_plan, d_counter, L.stream);
        if (rcz) return rcz;
        int32_t *st_o = status ? status : st_host.data();
        CU_TRY(ctx, cudaMemcpyAsync(st_o, L.d_small + zo_status, n * 4, cudaMemcpyDeviceToHost, L.stream));
        CU_TRY(ctx, lane_wait(ctx, L));
        for (size_t s = 0; s < n; s++)
            if (st_o[s] != 0) return GARAGE_EC_E_UNRECOVERABLE;
        return GARAGE_EC_OK;
    }
    const size_t k = ctx->k, tot = ctx->k + ctx->m;
    size_t cs = kHostChunkBytes / (tot * stride);
    if (cs < 1) cs = 1;
    if (cs > n) cs = n;
    // small buffer layout per lane: present | want | status | shard_len | plan+counter
    const size_t o_present = 0, o_want = align_up(cs * tot, 16), o_status = o_want + align_up(cs * tot, 16);
    const size_t o_len = o_status + align_up(cs * 4, 16), o_plan = o_len + align_up(cs * 4, 16);
    const size_t small = o_plan + plan_scratch_bytes(cs);
    for (HostLane &L : lanes.set->lanes) {
        int rc = lane_reserve(ctx, L, cs * tot * stride, small);
        if (rc) return rc;
    }
    int32_t *st_out = status ? status : st_host.data();
    int rc = GARAGE_EC_OK;
    size_t c = 0;
    for (size_t s0 = 0; s0 < n; s0 += cs, c++) {
        HostLane &L = lanes[c % kHostLanes];
        const size_t cnt = n - s0 < cs ? n - s0 : cs;
        uint8_t *d_sh = L.d_buf;
        // H2D: only the k survivors (first k present shards) of stripes that have work to do
        for (size_t s = s0; s < s0 + cnt; s++) {
            const uint8_t *pr = present + s * tot;
            size_t np = 0;
            bool work = false;
            for (size_t i = 0; i < tot; i++) {
                np += pr[i] ? 1 : 0;
                work |= !pr[i] && (!want || want[s * tot + i]);
            }
            if (np < k || !work) continue;
            size_t used = 0;
            for (size_t i = 0; i < tot && used < k; i++) {
                if (!pr[i]) continue;
                up.add(d_sh + ((s - s0) * tot + i) * stride, shard_at(s, i), stride);
                used++;
            }
        }
        rc = up.flush(ctx, cudaMemcpyHostToDevice, L.stream);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_present, present + s0 * tot, cnt * tot,
                                    cudaMemcpyHostToDevice, L.stream));
        const uint8_t *d_want = nullptr;
        if (want) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_want, want + s0 * tot, cnt * tot,
                                        cudaMemcpyHostToDevice, L.stream));
            d_want = L.d_small + o_want;
        }
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_len, shard_len + s0, cnt * 4, cudaMemcpyHostToDevice,
                                        L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small + o_len);
        }
        StripePlan *d_plan = reinterpret_cast<StripePlan *>(L.d_small + o_plan);
        uint32_t *d_counter = reinterpret_cast<uint32_t *>(L.d_small + o_plan + cnt * sizeof(StripePlan));
        rc = run_reconstruct(ctx, d_sh, L.d_small + o_present, d_want,
                             reinterpret_cast<int32_t *>(L.d_small + o_status), d_len, stride, cnt,
                             d_plan, d_counter, L.stream);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(st_out + s0, L.d_small + o_status, cnt * 4, cudaMemcpyDeviceToHost,
                                    L.stream));
        // D2H: exactly the shards that were rebuilt
        for (size_t s = s0; s < s0 + cnt; s++) {
            const uint8_t *pr = present + s * tot;
            size_t np = 0;
            for (size_t i = 0; i < tot; i++) np += pr[i] ? 1 : 0;
            if (np < k) continue;
            const size_t len = shard_len ? shard_len[s] : stride;
            const size_t bytes = align_up(len, 16);
            for (size_t i = 0; i < tot; i++) {
                if (pr[i] || (want && !want[s * tot + i])) continue;
                down.add(shard_at(s, i), d_sh + ((s - s0) * tot + i) * stride, bytes);
            }
        }
        rc = down.flush(ctx, cudaMemcpyDeviceToHost, L.stream);
        if (rc) return rc;
    }
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    for (size_t s = 0; s < n; s++)
        if (st_out[s] != 0) return GARAGE_EC_E_UNRECOVERABLE;
    return GARAGE_EC_OK;
}

int garage_ec_reconstruct(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present,
                          const uint8_t *want, int32_t *status, const uint32_t *shard_len,
                          size_t stride, size_t n_stripes, int mem_kind, void *cuda_stream)
{
    if (!ctx || (mem_kind != GARAGE_EC_MEM_HOST && mem_kind != GARAGE_EC_MEM_DEVICE))
        return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_stripes, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_stripes == 0) return GARAGE_EC_OK;
    if (!shards || !present) return GARAGE_EC_E_INVALID;
    if (!aligned16(shards)) return GARAGE_EC_E_ALIGN;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (mem_kind == GARAGE_EC_MEM_HOST)
        return reconstruct_host(ctx, shards, nullptr, present, want, status, shard_len, stride, n_stripes);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    void *scratch = nullptr;
    CU_TRY(ctx, ctx->pool ? cudaMallocFromPoolAsync(&scratch, plan_scratch_bytes(n_stripes), ctx->pool, st)
                          : cudaMallocAsync(&scratch, plan_scratch_bytes(n_stripes), st));
    StripePlan *plan = reinterpret_cast<StripePlan *>(scratch);
    uint32_t *counter =
        reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(scratch) + n_stripes * sizeof(StripePlan));
    rc = run_reconstruct(ctx, shards, present, want, status, shard_len, stride, n_stripes, plan, counter, st);
    cudaError_t e = cudaFreeAsync(scratch, st);
    if (rc) return rc;
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "cudaFreeAsync");
    return GARAGE_EC_OK;
}

int garage_ec_reconstruct_stripes(garage_ec_ctx *ctx, uint8_t *const *stripes, const uint8_t *present,
                                  const uint8_t *want, int32_t *status, const uint32_t *shard_len, size_t stride,
                                  size_t n_stripes)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_stripes, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_stripes == 0) return GARAGE_EC_OK;
    if (!stripes || !present) return GARAGE_EC_E_INVALID;
    for (size_t s = 0; s < n_stripes; s++) {
        if (!stripes[s]) return GARAGE_EC_E_INVALID;
        if (!aligned16(stripes[s])) return GARAGE_EC_E_ALIGN;
    }
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    return reconstruct_host(ctx, nullptr, stripes, present, want, status, shard_len, stride, n_stripes);
}

// --------------------------------------------------------------------------- CORRECT
// HOST: the present shards go up; once a chunk's status and fixed flags are on the host, exactly the
// rebuilt (absent) and fixed shards of its corrected stripes come back -- a clean chunk downloads only
// those two arrays.  Same per-lane Pending / finish pattern as the scrub sweep.
static int correct_host(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present, int32_t *status, uint8_t *fixed,
                        const uint32_t *shard_len, size_t stride, size_t n)
{
    const size_t tot = ctx->k + ctx->m;
    // declared before the lane lease: they must outlive the stream work the lease waits for
    std::vector<int32_t> st_host(status ? 0 : n);
    std::vector<uint8_t> fx_host(fixed ? 0 : n * tot);
    CopyBatch up, down;
    LEASE_LANES(ctx, lanes);
    size_t cs = kHostChunkBytes / (tot * stride);
    if (cs < 1) cs = 1;
    if (cs > n) cs = n;
    const size_t o_present = 0, o_fixed = align_up(cs * tot, 16), o_status = o_fixed + align_up(cs * tot, 16);
    const size_t o_len = o_status + align_up(cs * 4, 16), o_scr = o_len + align_up(cs * 4, 16);
    const size_t small = o_scr + correct_scratch_bytes(cs);
    for (HostLane &L : lanes.set->lanes) {
        int rc = lane_reserve(ctx, L, cs * tot * stride, small);
        if (rc) return rc;
    }
    int32_t *st_out = status ? status : st_host.data();
    uint8_t *fx_out = fixed ? fixed : fx_host.data();
    struct Pending {
        bool active = false;
        size_t s0 = 0, cnt = 0;
    } pend[kHostLanes];
    auto finish = [&](size_t lane_i) -> int {
        Pending &P = pend[lane_i];
        if (!P.active) return GARAGE_EC_OK;
        HostLane &L = lanes[lane_i];
        CU_TRY(ctx, lane_wait(ctx, L));  // status + fixed of this chunk are on the host
        for (size_t s = P.s0; s < P.s0 + P.cnt; s++) {
            if (st_out[s] != 0) continue;
            const size_t len = shard_len ? shard_len[s] : stride;
            for (size_t i = 0; i < tot; i++)
                if ((present && !present[s * tot + i]) || fx_out[s * tot + i])
                    down.add(shards + (s * tot + i) * stride, L.d_buf + ((s - P.s0) * tot + i) * stride, align_up(len, 16));
        }
        int r = down.flush(ctx, cudaMemcpyDeviceToHost, L.stream);
        P.active = false;
        return r;
    };
    size_t c = 0;
    for (size_t s0 = 0; s0 < n; s0 += cs, c++) {
        const size_t lane_i = c % kHostLanes;
        HostLane &L = lanes[lane_i];
        int rc = finish(lane_i);
        if (rc) return rc;
        const size_t cnt = n - s0 < cs ? n - s0 : cs;
        if (present) {
            for (size_t s = s0; s < s0 + cnt; s++)
                for (size_t i = 0; i < tot; i++)
                    if (present[s * tot + i])
                        up.add(L.d_buf + ((s - s0) * tot + i) * stride, shards + (s * tot + i) * stride, stride);
            rc = up.flush(ctx, cudaMemcpyHostToDevice, L.stream);
            if (rc) return rc;
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_present, present + s0 * tot, cnt * tot, cudaMemcpyHostToDevice,
                                        L.stream));
        } else {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_buf, shards + s0 * tot * stride, cnt * tot * stride, cudaMemcpyHostToDevice,
                                        L.stream));
        }
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_len, shard_len + s0, cnt * 4, cudaMemcpyHostToDevice, L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small + o_len);
        }
        rc = run_correct(ctx, L.d_buf, present ? L.d_small + o_present : nullptr,
                         reinterpret_cast<int32_t *>(L.d_small + o_status), L.d_small + o_fixed, d_len, stride, cnt,
                         L.d_small + o_scr, L.stream);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(st_out + s0, L.d_small + o_status, cnt * 4, cudaMemcpyDeviceToHost, L.stream));
        CU_TRY(ctx, cudaMemcpyAsync(fx_out + s0 * tot, L.d_small + o_fixed, cnt * tot, cudaMemcpyDeviceToHost, L.stream));
        pend[lane_i].active = true;
        pend[lane_i].s0 = s0;
        pend[lane_i].cnt = cnt;
    }
    for (size_t l = 0; l < (size_t)kHostLanes; l++) {
        int rc = finish(l);
        if (rc) return rc;
    }
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    bool unrec = false, uncorr = false;
    for (size_t s = 0; s < n; s++) {
        unrec |= st_out[s] == GARAGE_EC_E_UNRECOVERABLE;
        uncorr |= st_out[s] == GARAGE_EC_E_UNCORRECTABLE;
    }
    return unrec ? GARAGE_EC_E_UNRECOVERABLE : (uncorr ? GARAGE_EC_E_UNCORRECTABLE : GARAGE_EC_OK);
}

int garage_ec_correct(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *present, int32_t *status, uint8_t *fixed,
                      const uint32_t *shard_len, size_t stride, size_t n_stripes, int mem_kind, void *cuda_stream)
{
    if (!ctx || (mem_kind != GARAGE_EC_MEM_HOST && mem_kind != GARAGE_EC_MEM_DEVICE)) return GARAGE_EC_E_INVALID;
    if (!ctx->grs_ok) return GARAGE_EC_E_INVALID;  // custom matrix without GRS structure: errors cannot be located
    int rc = check_geometry(ctx, stride, n_stripes, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_stripes == 0) return GARAGE_EC_OK;
    if (!shards) return GARAGE_EC_E_INVALID;
    if (!aligned16(shards)) return GARAGE_EC_E_ALIGN;
    if (n_stripes * (size_t)(ctx->k + ctx->m) > 0xffffffffull) return GARAGE_EC_E_INVALID;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (mem_kind == GARAGE_EC_MEM_HOST)
        return correct_host(ctx, shards, present, status, fixed, shard_len, stride, n_stripes);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    void *scratch = nullptr;
    CU_TRY(ctx, ctx->pool ? cudaMallocFromPoolAsync(&scratch, correct_scratch_bytes(n_stripes), ctx->pool, st)
                          : cudaMallocAsync(&scratch, correct_scratch_bytes(n_stripes), st));
    rc = run_correct(ctx, shards, present, status, fixed, shard_len, stride, n_stripes, static_cast<uint8_t *>(scratch), st);
    cudaError_t e = cudaFreeAsync(scratch, st);
    if (rc) return rc;
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "cudaFreeAsync");
    return GARAGE_EC_OK;
}

// --------------------------------------------------------------------------- SHARD SUMS
static int run_sums(garage_ec_ctx *ctx, const uint8_t *shards, const uint8_t *expect, const uint32_t *shard_len,
                    size_t stride, size_t n_shards, int per_stripe, uint8_t *sums, uint8_t *bad, cudaStream_t st,
                    int out_per_stripe = 0, int out_off = 0, const uint8_t *shards2 = nullptr, size_t n_shards2 = 0,
                    int per_stripe2 = 1, int out_off2 = 0)
{
    SumParams q;
    memset(&q, 0, sizeof(q));
    q.base = shards;
    q.shard_len = shard_len;
    q.expect = expect;
    q.sums = sums;
    q.bad = bad;
    q.stride = (uint32_t)stride;
    q.per_stripe = (uint32_t)per_stripe;
    q.n_shards = (uint32_t)(n_shards + n_shards2);
    q.out_per_stripe = (uint32_t)(out_per_stripe ? out_per_stripe : per_stripe);
    q.out_off = (uint32_t)out_off;
    q.base2 = shards2;
    q.n_first = (uint32_t)n_shards;
    q.per_stripe2 = (uint32_t)per_stripe2;
    q.out_off2 = (uint32_t)out_off2;
    n_shards += n_shards2;
    // few shards: four lanes per shard (4x the parallelism, but the quad shuffles make it
    // LSU-bound: measured 5.4 ms vs 7.6 ms at 18 432 shards and 6.0 vs 5.7 ms at 28 672);
    // from ~24 000 shards on one thread per shard keeps the schedulers busy enough
    if (ctx->sum_kind.load(std::memory_order_relaxed) == GARAGE_EC_SUM_ADLER8) {
        // one warp per (shard, segment), 8 warps per block, persistent grid
        if (n_shards >= (1u << 29)) return GARAGE_EC_E_INVALID;
        if (expect && bad) {
            // segments OR their verdict into the shard's flag: clear the flags of this launch first.  Flags of
            // one launch are contiguous when out_per_stripe == per_stripe (check_sums / scrub_repair)
            const size_t nflags = (n_shards / (size_t)q.per_stripe) * q.out_per_stripe;
            cudaError_t e0 = cudaMemsetAsync(bad, 0, nflags, st);
            if (e0 != cudaSuccess) return set_cuda_error(ctx, e0, "cudaMemsetAsync(bad)");
        }
        const unsigned blocks = (unsigned)std::min<size_t>(n_shards, (size_t)ctx->sm_count * 8);
        adler8_shards_kernel<<<blocks, 256, 0, st>>>(q);
    } else if (n_shards < 24000)
        blake2sum_shards_quad_kernel<<<(unsigned)((n_shards + kQuadThreads / 4 - 1) / (kQuadThreads / 4)), kQuadThreads, 0,
                                       st>>>(q);
    else
        blake2sum_shards_kernel<<<(unsigned)((n_shards + 127) / 128), 128, 0, st>>>(q);
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_cuda_error(ctx, e, "blake2sum_shards_kernel launch");
    return GARAGE_EC_OK;
}

static int sums_common(garage_ec_ctx *ctx, const uint8_t *shards, const uint8_t *expect, const uint32_t *shard_len,
                       size_t stride, size_t n, int per, uint8_t *sums_out, uint8_t *bad_out, int mem_kind,
                       void *cuda_stream)
{
    if (!ctx || (mem_kind != GARAGE_EC_MEM_HOST && mem_kind != GARAGE_EC_MEM_DEVICE)) return GARAGE_EC_E_INVALID;
    if (per < 1 || per > kMaxK + kMaxM) return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n, per);
    if (rc) return rc;
    if (n == 0) return GARAGE_EC_OK;
    if (!shards || (!sums_out && !bad_out)) return GARAGE_EC_E_INVALID;
    if (!aligned16(shards)) return GARAGE_EC_E_ALIGN;
    if (n * (size_t)per > 0xffffffffull) return GARAGE_EC_E_INVALID;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (mem_kind == GARAGE_EC_MEM_DEVICE)
        return run_sums(ctx, shards, expect, shard_len, stride, n * per, per, sums_out, bad_out,
                        (cudaStream_t)cuda_stream);
    // HOST: chunked through the lanes (H2D shards [+ expect], kernel, D2H sums / bad flags)
    LEASE_LANES(ctx, lanes);
    size_t cs = kHostChunkBytes / ((size_t)per * stride);
    if (cs < 1) cs = 1;
    if (cs > n) cs = n;
    const size_t o_len = 0, o_exp = align_up(cs * 4, 16), o_sum = o_exp + cs * per * 32, o_bad = o_sum + cs * per * 32;
    const size_t small = o_bad + align_up(cs * per, 16);
    for (HostLane &L : lanes.set->lanes) {
        rc = lane_reserve(ctx, L, cs * per * stride, small);
        if (rc) return rc;
    }
    size_t c = 0;
    for (size_t s0 = 0; s0 < n; s0 += cs, c++) {
        HostLane &L = lanes[c % kHostLanes];
        const size_t cnt = n - s0 < cs ? n - s0 : cs;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_buf, shards + s0 * per * stride, cnt * per * stride, cudaMemcpyHostToDevice,
                                    L.stream));
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_len, shard_len + s0, cnt * 4, cudaMemcpyHostToDevice, L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small + o_len);
        }
        const uint8_t *d_exp = nullptr;
        if (expect) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_exp, expect + s0 * per * 32, cnt * per * 32,
                                        cudaMemcpyHostToDevice, L.stream));
            d_exp = L.d_small + o_exp;
        }
        rc = run_sums(ctx, L.d_buf, d_exp, d_len, stride, cnt * per, per, sums_out ? L.d_small + o_sum : nullptr,
                      bad_out ? L.d_small + o_bad : nullptr, L.stream);
        if (rc) return rc;
        if (sums_out)
            CU_TRY(ctx, cudaMemcpyAsync(sums_out + s0 * per * 32, L.d_small + o_sum, cnt * per * 32,
                                        cudaMemcpyDeviceToHost, L.stream));
        if (bad_out)
            CU_TRY(ctx, cudaMemcpyAsync(bad_out + s0 * per, L.d_small + o_bad, cnt * per, cudaMemcpyDeviceToHost,
                                        L.stream));
    }
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    return GARAGE_EC_OK;
}

int garage_ec_shard_sums(garage_ec_ctx *ctx, const uint8_t *shards, const uint32_t *shard_len, size_t stride,
                         size_t n_stripes, int shards_per_stripe, uint8_t *sums_out, int mem_kind, void *cuda_stream)
{
    if (!sums_out) return GARAGE_EC_E_INVALID;
    return sums_common(ctx, shards, nullptr, shard_len, stride, n_stripes, shards_per_stripe, sums_out, nullptr,
                       mem_kind, cuda_stream);
}

int garage_ec_check_sums(garage_ec_ctx *ctx, const uint8_t *shards, const uint8_t *expect, const uint32_t *shard_len,
                         size_t stride, size_t n_stripes, int shards_per_stripe, uint8_t *bad_out, int mem_kind,
                         void *cuda_stream)
{
    if (!expect || !bad_out) return GARAGE_EC_E_INVALID;
    return sums_common(ctx, shards, expect, shard_len, stride, n_stripes, shards_per_stripe, nullptr, bad_out,
                       mem_kind, cuda_stream);
}

void garage_ec_blake2sum(const uint8_t *data, size_t len, uint8_t out32[32]) { blake2sum_host(data, len, out32); }

// A plain memcpy leaves the destination lines modified in the writing core's cache, and the DMA read that follows has
// to pull them out of there snoop by snoop: measured on the B200 hosts, 6.7 GB/s for the upload of a batch of freshly
// landed 1 MiB blocks against 45 GB/s for the same batch at rest in DRAM (profiles/r02_summary.md).  Non-temporal
// stores send the lines to memory instead.  GARAGE_EC_NT_COPY=0 falls back to memcpy (A/B measurements).
void garage_ec_copy_for_dma(void *dst_v, const void *src_v, size_t n)
{
    uint8_t *dst = static_cast<uint8_t *>(dst_v);
    const uint8_t *src = static_cast<const uint8_t *>(src_v);
#if defined(__x86_64__)
    static const bool nt = [] {
        const char *e = getenv("GARAGE_EC_NT_COPY");
        return !(e && e[0] == '0');
    }();
    if (nt && n >= 4096) {
        const size_t head = (size_t)(-(uintptr_t)dst & 63);
        memcpy(dst, src, head);
        dst += head, src += head, n -= head;
        const size_t body = n & ~(size_t)63;
        for (size_t i = 0; i < body; i += 64) {
            const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i));
            const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 16));
            const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 32));
            const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i + 48));
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i), a);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 32), c);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst + i + 48), d);
        }
        _mm_sfence();
        memcpy(dst + body, src + body, n - body);
        return;
    }
#endif
    if (n) memcpy(dst, src, n);
}

int garage_ec_set_wait_mode(garage_ec_ctx *ctx, int blocking)
{
    if (!ctx || (blocking != 0 && blocking != 1)) return GARAGE_EC_E_INVALID;
    ctx->wait_blocking.store(blocking, std::memory_order_relaxed);
    return GARAGE_EC_OK;
}

int garage_ec_set_sum_kind(garage_ec_ctx *ctx, int kind)
{
    if (!ctx || (kind != GARAGE_EC_SUM_BLAKE2 && kind != GARAGE_EC_SUM_ADLER8)) return GARAGE_EC_E_INVALID;
    ctx->sum_kind.store(kind, std::memory_order_relaxed);
    return GARAGE_EC_OK;
}

// Host-side adler8 with AVX2 (the read path checks the tag of every shard it touches: at 2.8 GB/s the scalar loop
// was a third of the CPU time of a GET in the block manager).  Adler-32 over a run of N = 32 * blocks bytes:
//   a' = a + sum d,   b' = b + N a + sum_{j,i} (N - 32 j - i) d[j][i]
// and N - 32 j - i = (32 - i) + 32 (blocks - 1 - j): a weighted sum inside each 32-byte block (pmaddubsw with the
// taps 32..1) plus 32 times, for every block, the byte sum of all blocks before it.  Runs are capped like zlib's
// NMAX so that nothing overflows 32 bits.  Same values as adler8_host (blake2b.h) and zlib.adler32.
#if defined(__x86_64__)
__attribute__((target("avx2"))) static uint32_t adler32_avx2(const uint8_t *p, size_t n)
{
    uint32_t a = 1, b = 0;
    const __m256i tap = _mm256_setr_epi8(32, 31, 30, 29, 28, 27, 26, 25, 24, 23, 22, 21, 20, 19, 18, 17, 16, 15, 14, 13, 12, 11,
                                         10, 9, 8, 7, 6, 5, 4, 3, 2, 1);
    const __m256i ones = _mm256_set1_epi16(1), zero = _mm256_setzero_si256();
    while (n >= 32) {
        size_t blocks = n / 32;
        if (blocks > 5552 / 32) blocks = 5552 / 32;
        n -= blocks * 32;
        uint64_t bb = (uint64_t)b + (uint64_t)a * (uint64_t)(blocks * 32);
        __m256i v_before = zero, v_sum = zero, v_tap = zero;
        for (size_t j = 0; j < blocks; j++, p += 32) {
            const __m256i d = _mm256_loadu_si256(reinterpret_cast<const __m256i *>(p));
            v_before = _mm256_add_epi32(v_before, v_sum);
            v_sum = _mm256_add_epi32(v_sum, _mm256_sad_epu8(d, zero));
            v_tap = _mm256_add_epi32(v_tap, _mm256_madd_epi16(_mm256_maddubs_epi16(d, tap), ones));
        }
        alignas(32) uint32_t s[8], t[8], w[8];
        _mm256_store_si256(reinterpret_cast<__m256i *>(s), v_sum);
        _mm256_store_si256(reinterpret_cast<__m256i *>(t), v_tap);
        _mm256_store_si256(reinterpret_cast<__m256i *>(w), v_before);
        uint64_t aa = a;
        for (int i = 0; i < 8; i++) {
            aa += s[i];
            bb += (uint64_t)t[i] + 32ull * w[i];
        }
        a = (uint32_t)(aa % 65521);
        b = (uint32_t)(bb % 65521);
    }
    for (; n; n--, p++) {
        a += *p;
        b += a;
    }
    a %= 65521;
    b %= 65521;
    return (b << 16) | a;
}

static void adler8_host_fast(const uint8_t *data, size_t len, uint8_t out[32])
{
    static const bool avx2 = __builtin_cpu_supports("avx2");
    if (!avx2 || len > 0xffffffffull) return adler8_host(data, len, out);
    const size_t seg = adler8_seg_bytes((uint32_t)len);
    for (int s = 0; s < 8; s++) {
        const size_t start = (size_t)s * seg;
        uint32_t v = 1;  // Adler-32 of nothing
        if (start < len) v = adler32_avx2(data + start, len < start + seg ? len - start : seg);
        memcpy(out + 4 * s, &v, 4);  // little endian
    }
}
#else
static void adler8_host_fast(const uint8_t *data, size_t len, uint8_t out[32]) { adler8_host(data, len, out); }
#endif

int garage_ec_shard_sum_host(int kind, const uint8_t *data, size_t len, uint8_t out32[32])
{
    if (!out32 || (!data && len)) return GARAGE_EC_E_INVALID;
    if (kind == GARAGE_EC_SUM_BLAKE2) blake2sum_host(data, len, out32);
    else if (kind == GARAGE_EC_SUM_ADLER8) adler8_host_fast(data, len, out32);
    else return GARAGE_EC_E_INVALID;
    return GARAGE_EC_OK;
}

// --------------------------------------------------------------------------- SCRUB + REPAIR
int garage_ec_scrub_repair(garage_ec_ctx *ctx, uint8_t *shards, const uint8_t *expect_sums, uint8_t *bad_out,
                           int32_t *status, const uint32_t *shard_len, size_t stride, size_t n_stripes, int mem_kind,
                           void *cuda_stream)
{
    if (!ctx || (mem_kind != GARAGE_EC_MEM_HOST && mem_kind != GARAGE_EC_MEM_DEVICE)) return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_stripes, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_stripes == 0) return GARAGE_EC_OK;
    if (!shards || !expect_sums || !bad_out) return GARAGE_EC_E_INVALID;
    if (!aligned16(shards)) return GARAGE_EC_E_ALIGN;
    const size_t tot = ctx->k + ctx->m;
    if (n_stripes * tot > 0xffffffffull) return GARAGE_EC_E_INVALID;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (mem_kind == GARAGE_EC_MEM_DEVICE) {
        cudaStream_t st = (cudaStream_t)cuda_stream;
        rc = run_sums(ctx, shards, expect_sums, shard_len, stride, n_stripes * tot, (int)tot, nullptr, bad_out, st);
        if (rc) return rc;
        void *scratch = nullptr;
        CU_TRY(ctx, ctx->pool ? cudaMallocFromPoolAsync(&scratch, plan_scratch_bytes(n_stripes), ctx->pool, st)
                          : cudaMallocAsync(&scratch, plan_scratch_bytes(n_stripes), st));
        StripePlan *plan = reinterpret_cast<StripePlan *>(scratch);
        uint32_t *counter =
            reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(scratch) + n_stripes * sizeof(StripePlan));
        rc = run_reconstruct(ctx, shards, bad_out, nullptr, status, shard_len, stride, n_stripes, plan, counter, st,
                             /*present_is_bad=*/true);
        cudaError_t e = cudaFreeAsync(scratch, st);
        if (rc) return rc;
        if (e != cudaSuccess) return set_cuda_error(ctx, e, "cudaFreeAsync");
        return GARAGE_EC_OK;
    }
    // HOST: every shard goes up (it has to be hashed); only the rebuilt shards come back.  The
    // rebuilt set is known once the bad flags are on the host, so each lane's chunk is finished
    // (flags read, copies issued) when the lane comes round again.
    std::vector<int32_t> st_host(status ? 0 : n_stripes);  // outlives the lane lease below
    CopyBatch down;
    LEASE_LANES(ctx, lanes);
    size_t cs = kHostChunkBytes / (tot * stride);
    if (cs < 1) cs = 1;
    if (cs > n_stripes) cs = n_stripes;
    const size_t o_exp = 0, o_bad = o_exp + cs * tot * 32, o_status = o_bad + align_up(cs * tot, 16);
    const size_t o_len = o_status + align_up(cs * 4, 16), o_plan = o_len + align_up(cs * 4, 16);
    const size_t small = o_plan + plan_scratch_bytes(cs);
    for (HostLane &L : lanes.set->lanes) {
        rc = lane_reserve(ctx, L, cs * tot * stride, small);
        if (rc) return rc;
    }
    int32_t *st_out = status ? status : st_host.data();
    struct Pending {
        bool active = false;
        size_t s0 = 0, cnt = 0;
    } pend[kHostLanes];
    auto finish = [&](size_t lane_i) -> int {
        Pending &P = pend[lane_i];
        if (!P.active) return GARAGE_EC_OK;
        HostLane &L = lanes[lane_i];
        CU_TRY(ctx, lane_wait(ctx, L));  // bad flags + status of this chunk are on the host
        for (size_t s = P.s0; s < P.s0 + P.cnt; s++) {
            if (st_out[s] != 0) continue;
            const size_t len = shard_len ? shard_len[s] : stride;
            for (size_t i = 0; i < tot; i++)
                if (bad_out[s * tot + i])
                    down.add(shards + (s * tot + i) * stride, L.d_buf + ((s - P.s0) * tot + i) * stride,
                             align_up(len, 16));
        }
        int r = down.flush(ctx, cudaMemcpyDeviceToHost, L.stream);
        P.active = false;
        return r;
    };
    size_t c = 0;
    for (size_t s0 = 0; s0 < n_stripes; s0 += cs, c++) {
        const size_t lane_i = c % kHostLanes;
        HostLane &L = lanes[lane_i];
        rc = finish(lane_i);
        if (rc) return rc;
        const size_t cnt = n_stripes - s0 < cs ? n_stripes - s0 : cs;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_buf, shards + s0 * tot * stride, cnt * tot * stride, cudaMemcpyHostToDevice,
                                    L.stream));
        CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_exp, expect_sums + s0 * tot * 32, cnt * tot * 32,
                                    cudaMemcpyHostToDevice, L.stream));
        const uint32_t *d_len = nullptr;
        if (shard_len) {
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_len, shard_len + s0, cnt * 4, cudaMemcpyHostToDevice, L.stream));
            d_len = reinterpret_cast<const uint32_t *>(L.d_small + o_len);
        }
        rc = run_sums(ctx, L.d_buf, L.d_small + o_exp, d_len, stride, cnt * tot, (int)tot, nullptr, L.d_small + o_bad,
                      L.stream);
        if (rc) return rc;
        StripePlan *d_plan = reinterpret_cast<StripePlan *>(L.d_small + o_plan);
        uint32_t *d_counter = reinterpret_cast<uint32_t *>(L.d_small + o_plan + cnt * sizeof(StripePlan));
        rc = run_reconstruct(ctx, L.d_buf, L.d_small + o_bad, nullptr, reinterpret_cast<int32_t *>(L.d_small + o_status),
                             d_len, stride, cnt, d_plan, d_counter, L.stream, true);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(bad_out + s0 * tot, L.d_small + o_bad, cnt * tot, cudaMemcpyDeviceToHost, L.stream));
        CU_TRY(ctx, cudaMemcpyAsync(st_out + s0, L.d_small + o_status, cnt * 4, cudaMemcpyDeviceToHost, L.stream));
        pend[lane_i].active = true;
        pend[lane_i].s0 = s0;
        pend[lane_i].cnt = cnt;
    }
    for (size_t l = 0; l < (size_t)kHostLanes; l++) {
        rc = finish(l);
        if (rc) return rc;
    }
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    for (size_t s = 0; s < n_stripes; s++)
        if (st_out[s] != 0) return GARAGE_EC_E_UNRECOVERABLE;
    return GARAGE_EC_OK;
}

// --------------------------------------------------------------------------- BLOCK-LEVEL
int garage_ec_encode_blocks(garage_ec_ctx *ctx, const uint8_t *const *blocks, const uint32_t *block_len,
                            size_t n_blocks, uint8_t *parity_out, size_t stride)
{
    return garage_ec_encode_blocks_with_sums(ctx, blocks, block_len, n_blocks, parity_out, nullptr, stride);
}

int garage_ec_encode_blocks_with_sums(garage_ec_ctx *ctx, const uint8_t *const *blocks, const uint32_t *block_len,
                                      size_t n_blocks, uint8_t *parity_out, uint8_t *sums_out, size_t stride)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_blocks, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_blocks == 0) return GARAGE_EC_OK;
    if (!blocks || !block_len || !parity_out) return GARAGE_EC_E_INVALID;
    const size_t k = ctx->k, m = ctx->m;
    uint32_t max_len = 0;
    for (size_t s = 0; s < n_blocks; s++) {
        if (!blocks[s] && block_len[s]) return GARAGE_EC_E_INVALID;
        if (garage_ec_shard_len(block_len[s], (int)k) > stride) return GARAGE_EC_E_INVALID;
        max_len = block_len[s] > max_len ? block_len[s] : max_len;
    }
    const auto tr0 = std::chrono::steady_clock::now();
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    size_t cs = kHostChunkBytes / (k * stride);
    if (cs < 1) cs = 1;
    if (cs > n_blocks) cs = n_blocks;
    // per lane: [blocks as they arrive, contiguous, `pitch` apart][k data shards][m parity shards]
    const size_t pitch = align_up((size_t)max_len + 16, 16);  // + one aligned word of slack for the split kernel
    const size_t blk_b = align_up(cs * pitch, 256), in_b = cs * k * stride, out_b = cs * m * stride;
    std::vector<uint32_t> lens(2 * cs * kHostLanes);  // [shard_len | block_len] per lane; outlives the lane lease below
    CopyBatch up;
    LEASE_LANES(ctx, lanes);
    for (HostLane &L : lanes.set->lanes) {
        rc = lane_reserve(ctx, L, blk_b + in_b + out_b, align_up(cs * 8, 16) + cs * (k + m) * 32);
        if (rc) return rc;
    }
    const size_t o_blen = cs * 4, o_sums = align_up(cs * 8, 16);
    const auto tr1 = std::chrono::steady_clock::now();
    cudaEvent_t tev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if (ctx->trace)
        for (auto &e : tev) cudaEventCreate(&e);
    auto mark = [&](int i, size_t chunk, cudaStream_t st) {
        if (ctx->trace && chunk == 0 && tev[i]) cudaEventRecord(tev[i], st);
    };
    size_t c = 0;
    for (size_t s0 = 0; s0 < n_blocks; s0 += cs, c++) {
        const size_t lane_i = c % kHostLanes;
        HostLane &L = lanes[lane_i];
        const size_t cnt = n_blocks - s0 < cs ? n_blocks - s0 : cs;
        // the pageable `lens` slot of this lane is reused: wait for the lane's previous chunk
        if (c >= (size_t)kHostLanes) CU_TRY(ctx, lane_wait(ctx, L));
        mark(0, c, L.stream);
        uint32_t *hl = lens.data() + lane_i * 2 * cs, *hb = hl + cs;
        uint8_t *d_blk = L.d_buf, *d_data = L.d_buf + blk_b, *d_par = d_data + in_b;
        for (size_t s = 0; s < cnt; s++) {
            hl[s] = garage_ec_shard_len(block_len[s0 + s], (int)k);
            hb[s] = block_len[s0 + s];
            // H2D: the block as ONE contiguous copy; the framing happens on the device
            up.add(d_blk + s * pitch, blocks[s0 + s], block_len[s0 + s]);
        }
        rc = up.flush(ctx, cudaMemcpyHostToDevice, L.stream);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(L.d_small, hl, cnt * 4, cudaMemcpyHostToDevice, L.stream));
        CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_blen, hb, cnt * 4, cudaMemcpyHostToDevice, L.stream));
        mark(1, c, L.stream);
        SplitParams sp;
        sp.blocks = d_blk;
        sp.block_len = reinterpret_cast<const uint32_t *>(L.d_small + o_blen);
        sp.shards = d_data;
        sp.block_pitch = pitch;
        sp.stride = (uint32_t)stride;
        sp.k = (uint32_t)k;
        sp.n = (uint32_t)cnt;
        // ~4 CTAs per SM whatever the batch size (one CTA per block left 13 SMs copying 1 MiB each: 150 us)
        sp.parts = (uint32_t)std::max<size_t>(1, std::min<size_t>(64, ((size_t)ctx->sm_count * 4 + cnt - 1) / cnt));
        split_blocks_kernel<<<(unsigned)std::min<size_t>(cnt * sp.parts, (size_t)ctx->sm_count * 8), 256, 0, L.stream>>>(sp);
        ctx->launches.fetch_add(1, std::memory_order_relaxed);
        CU_TRY(ctx, cudaGetLastError());
        rc = run_uniform(ctx, kModeEncode, d_data, k * stride, d_par, m * stride, nullptr,
                         reinterpret_cast<const uint32_t *>(L.d_small), stride, cnt, L.stream);
        if (rc) return rc;
        mark(2, c, L.stream);
        CU_TRY(ctx, cudaMemcpyAsync(parity_out + s0 * m * stride, d_par, cnt * m * stride, cudaMemcpyDeviceToHost, L.stream));
        mark(3, c, L.stream);
        if (sums_out) {
            // per-shard tags of all k+m shards while they are on the device (row f2): [s][k+m][32]
            const uint32_t *d_len = reinterpret_cast<const uint32_t *>(L.d_small);
            rc = run_sums(ctx, d_data, nullptr, d_len, stride, cnt * k, (int)k, L.d_small + o_sums, nullptr, L.stream,
                          (int)(k + m), 0, d_par, cnt * m, (int)m, (int)k);
            if (rc) return rc;
            CU_TRY(ctx, cudaMemcpyAsync(sums_out + s0 * (k + m) * 32, L.d_small + o_sums, cnt * (k + m) * 32,
                                        cudaMemcpyDeviceToHost, L.stream));
        }
        mark(4, c, L.stream);
    }
    const auto tr2 = std::chrono::steady_clock::now();
    for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
    if (ctx->trace) {
        const auto tr3 = std::chrono::steady_clock::now();
        auto us = [](auto a, auto b) { return (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(b - a).count(); };
        ctx->tr_calls++;
        ctx->tr_blocks += n_blocks;
        ctx->tr_prep_us += us(tr0, tr1);
        ctx->tr_issue_us += us(tr1, tr2);
        ctx->tr_sync_us += us(tr2, tr3);
        for (int i = 0; i < 4; i++) {
            float ms = 0;
            if (tev[i] && tev[i + 1] && cudaEventElapsedTime(&ms, tev[i], tev[i + 1]) == cudaSuccess)
                ctx->tr_gpu_ns[i] += (uint64_t)(ms * 1e6);
        }
        (void)cudaGetLastError();
        for (auto e : tev)
            if (e) cudaEventDestroy(e);  // (an error return above leaks them: trace mode is a tuning aid only)
    }
    return GARAGE_EC_OK;
}

int garage_ec_decode_blocks(garage_ec_ctx *ctx, const uint8_t *shards, const uint8_t *present,
                            const uint32_t *block_len, size_t n_blocks, size_t stride,
                            uint8_t *const *blocks_out, int32_t *status)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    int rc = check_geometry(ctx, stride, n_blocks, ctx->k + ctx->m);
    if (rc) return rc;
    if (n_blocks == 0) return GARAGE_EC_OK;
    if (!shards || !present || !block_len || !blocks_out) return GARAGE_EC_E_INVALID;
    if (!aligned16(shards)) return GARAGE_EC_E_ALIGN;
    const size_t k = ctx->k, tot = ctx->k + ctx->m;
    CU_TRY(ctx, cudaSetDevice(ctx->device));

    // stripes with an absent data shard go to the GPU; the rest is a host-side join
    std::vector<size_t> need;
    bool any_bad = false;
    for (size_t s = 0; s < n_blocks; s++) {
        const uint8_t *pr = present + s * tot;
        size_t np = 0;
        bool data_missing = false;
        for (size_t i = 0; i < tot; i++) np += pr[i] ? 1 : 0;
        for (size_t j = 0; j < k; j++) data_missing |= !pr[j];
        if (garage_ec_shard_len(block_len[s], (int)k) > stride) return GARAGE_EC_E_INVALID;
        if (np < k) {
            if (status) status[s] = GARAGE_EC_E_UNRECOVERABLE;
            any_bad = true;
            continue;
        }
        if (status) status[s] = 0;
        if (data_missing) need.push_back(s);
    }
    size_t cs = kHostChunkBytes / (tot * stride);
    if (cs < 1) cs = 1;
    if (!need.empty()) {
        if (cs > need.size()) cs = need.size();
        const size_t o_present = 0, o_want = align_up(cs * tot, 16), o_status = o_want + align_up(cs * tot, 16);
        const size_t o_len = o_status + align_up(cs * 4, 16), o_plan = o_len + align_up(cs * 4, 16);
        const size_t small = o_plan + plan_scratch_bytes(cs);
        // host staging and copy lists are declared before the lane lease: they outlive its stream work
        std::vector<uint8_t> h_small((2 * cs * tot + cs * 4) * kHostLanes);
        CopyBatch up, down;
        LEASE_LANES(ctx, lanes);
        for (HostLane &L : lanes.set->lanes) {
            rc = lane_reserve(ctx, L, cs * tot * stride, small);
            if (rc) return rc;
        }
        size_t c = 0;
        for (size_t q0 = 0; q0 < need.size(); q0 += cs, c++) {
            const size_t lane_i = c % kHostLanes;
            HostLane &L = lanes[lane_i];
            const size_t cnt = need.size() - q0 < cs ? need.size() - q0 : cs;
            if (c >= (size_t)kHostLanes) CU_TRY(ctx, lane_wait(ctx, L));
            uint8_t *hp = h_small.data() + lane_i * (2 * cs * tot + cs * 4);
            uint8_t *hw = hp + cs * tot;
            uint32_t *hl = reinterpret_cast<uint32_t *>(hw + cs * tot);
            for (size_t q = 0; q < cnt; q++) {
                const size_t s = need[q0 + q];
                memcpy(hp + q * tot, present + s * tot, tot);
                for (size_t i = 0; i < tot; i++) hw[q * tot + i] = i < k ? 1 : 0;  // data shards only
                hl[q] = garage_ec_shard_len(block_len[s], (int)k);
                // H2D: only the k survivors the kernel reads (the first k present shards) -- the
                // GET path is PCIe-bound, absent and surplus shards stay on the host
                size_t used = 0;
                for (size_t i = 0; i < tot && used < k; i++) {
                    if (!present[s * tot + i]) continue;
                    up.add(L.d_buf + (q * tot + i) * stride, shards + (s * tot + i) * stride, align_up(hl[q], 16));
                    used++;
                }
            }
            rc = up.flush(ctx, cudaMemcpyHostToDevice, L.stream);
            if (rc) return rc;
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_present, hp, cnt * tot, cudaMemcpyHostToDevice, L.stream));
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_want, hw, cnt * tot, cudaMemcpyHostToDevice, L.stream));
            CU_TRY(ctx, cudaMemcpyAsync(L.d_small + o_len, hl, cnt * 4, cudaMemcpyHostToDevice, L.stream));
            StripePlan *d_plan = reinterpret_cast<StripePlan *>(L.d_small + o_plan);
            uint32_t *d_counter = reinterpret_cast<uint32_t *>(L.d_small + o_plan + cnt * sizeof(StripePlan));
            rc = run_reconstruct(ctx, L.d_buf, L.d_small + o_present, L.d_small + o_want,
                                 reinterpret_cast<int32_t *>(L.d_small + o_status),
                                 reinterpret_cast<const uint32_t *>(L.d_small + o_len), stride, cnt, d_plan,
                                 d_counter, L.stream);
            if (rc) return rc;
            // rebuilt data shards land directly in the output blocks
            for (size_t q = 0; q < cnt; q++) {
                const size_t s = need[q0 + q];
                const size_t Ls = hl[q];
                for (size_t j = 0; j < k; j++) {
                    if (present[s * tot + j]) continue;
                    const size_t off = j * Ls;
                    if (off >= block_len[s]) continue;
                    const size_t have = block_len[s] - off < Ls ? block_len[s] - off : Ls;
                    down.add(blocks_out[s] + off, L.d_buf + (q * tot + j) * stride, have);
                }
            }
            rc = down.flush(ctx, cudaMemcpyDeviceToHost, L.stream);
            if (rc) return rc;
        }
        // host-side join of the data shards that did arrive, while the GPU works
        // (framing: block = shard0|shard1|...)
        for (size_t s = 0; s < n_blocks; s++) {
            const uint8_t *pr = present + s * tot;
            size_t np = 0;
            for (size_t i = 0; i < tot; i++) np += pr[i] ? 1 : 0;
            if (np < k) continue;
            const size_t Ls = garage_ec_shard_len(block_len[s], (int)k);
            for (size_t j = 0; j < k; j++) {
                if (!pr[j]) continue;
                const size_t off = j * Ls;
                if (off >= block_len[s]) continue;
                const size_t have = block_len[s] - off < Ls ? block_len[s] - off : Ls;
                memcpy(blocks_out[s] + off, shards + (s * tot + j) * stride, have);
            }
        }
        for (HostLane &L : lanes.set->lanes) CU_TRY(ctx, lane_wait(ctx, L));
        return any_bad ? GARAGE_EC_E_UNRECOVERABLE : GARAGE_EC_OK;
    }
    for (size_t s = 0; s < n_blocks; s++) {
        const uint8_t *pr = present + s * tot;
        size_t np = 0;
        for (size_t i = 0; i < tot; i++) np += pr[i] ? 1 : 0;
        if (np < k) continue;
        const size_t Ls = garage_ec_shard_len(block_len[s], (int)k);
        for (size_t j = 0; j < k; j++) {
            const size_t off = j * Ls;
            if (off >= block_len[s]) continue;
            const size_t have = block_len[s] - off < Ls ? block_len[s] - off : Ls;
            memcpy(blocks_out[s] + off, shards + (s * tot + j) * stride, have);
        }
    }
    return any_bad ? GARAGE_EC_E_UNRECOVERABLE : GARAGE_EC_OK;
}

// ---- test hook -------------------------------------------------------------------------------
int garage_ec_debug_fail_after(garage_ec_ctx *ctx, long n_calls)
{
    if (!ctx) return GARAGE_EC_E_INVALID;
    ctx->fault_countdown.store(n_calls, std::memory_order_relaxed);
    return GARAGE_EC_OK;
}

}  // extern "C"
