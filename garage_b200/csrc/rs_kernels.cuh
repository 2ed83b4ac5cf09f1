// rs_kernels.cuh -- sm_100a kernels of the Garage erasure-coding block path.
//
// What they compute (normative definition: DESIGN.md "Arithmetic"):
//     out[i][t] = XOR_j C[i][j] * src[j][t]         over GF(2^8)/0x11D, byte-wise
// for rows i of a small coefficient matrix C (the parity rows P for encode/verify, a
// per-stripe composed decode matrix for reconstruct) and the k source shards of a stripe.
// Reference call sites this replaces work at: BlockManager::rpc_put_block
// (src/block/manager.rs:366-408), rpc_get_raw_block_internal (manager.rs:276-339),
// BlockResyncManager::resync_block (src/block/resync.rs:460-500), DataBlock::verify /
// ScrubWorker::work (src/block/block.rs:69-83, src/block/repair.rs:438-490).
//
// Design (DESIGN.md "Kernels"):
//  * HBM-bound byte work, no tensor cores.  The per-byte GF multiply-accumulate for up to 4
//    output rows is ONE shared-memory lookup: T_j[x] = {C0j*x, C1j*x, C2j*x, C3j*x} packed in
//    a 32-bit word, so a data byte costs one LDS + one XOR for all four rows.
//  * Conflict-free lookups with small tables ("sub-warp interleaving", mixed group sizes).
//    G tables share one 32 KB group: table `sub` of the group is replicated R = 32/G times in
//    banks [sub*R, sub*R + R) of every 128-byte row x.  The warp is cut in G sub-warps of R
//    lanes; at phase p of the group sub-warp q works on source base + (p xor q), so every
//    sub-warp is in a different table and every lane owns its bank:
//    word = group*8192 + x*32 + (lane xor p*R).  XOR accumulation commutes, so the per-lane
//    source order costs nothing.  k sources are decomposed greedily into groups of 32/16/8/4/2/1
//    tables (no padding lookups): RS(10,4) = one group of 8 + one group of 2 = 64 KB (round 1
//    used uniform G = 2: 160 KB), k = 16 -> 32 KB, k = 32 -> 32 KB.
//  * Two ways to bring a 16-byte column of every source to the lanes (StreamCfg::kTma):
//      LDG  : k x ld.global.nc.v4 per lane straight into registers, the next column's vectors
//             prefetched into a second register set (group size capped at 8 so that a warp
//             instruction still reads >= 64 contiguous bytes per shard);
//      TMA  : one elected lane issues k cp.async.bulk (1-D TMA) copies of 512 bytes -- the
//             warp's 32 columns of each shard -- into the warp's private shared-memory stage
//             and arms the stage's mbarrier with the byte count; the warp waits on the
//             mbarrier, pulls its vectors with conflict-free LDS.128, and immediately re-arms
//             the stage for its next work item, so the copy flies while the lookups run.  No
//             prefetch registers, any lane may read any source row, which is what allows the
//             16- and 32-table groups and k up to 32 at full speed.
//  * Reconstruct (per-stripe matrices) runs WITHOUT block-wide barriers: two table buffers, a
//    builder warp that stages the next stripe's plan and builds its tables while the consumer
//    warps stream the current stripe, mbarriers `full[b]` (tables of buffer b ready) and
//    `empty[b]` (every consumer warp has left the stripe that used buffer b).  Consumer warps
//    claim 32-column chunks from a per-stripe shared counter and flow from stripe to stripe on
//    their own.
//  * log/antilog tables sit in __constant__ memory and are staged to shared memory by the
//    decode-planning kernel; the product tables are built from xtime chains (no log lookups).
//  * Persistent grid: one CTA per SM.
#pragma once
#include <cuda.h>  // CUtensorMap (type only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "blake2b.h"
#include "gf256.h"

namespace garage_ec {

// ---- tuning overrides (tools/build_variants.py); -1 = per-shape default -------------------
#ifndef GEC_TMA_ENC
#define GEC_TMA_ENC -1
#endif
#ifndef GEC_TMA_PLAN
#define GEC_TMA_PLAN -1
#endif
#ifndef GEC_TMA_VER
#define GEC_TMA_VER -1
#endif
#ifndef GEC_NW_ENC
#define GEC_NW_ENC 0  // consumer warps; 0 = default
#endif
#ifndef GEC_NW_PLAN
#define GEC_NW_PLAN 0
#endif
#ifndef GEC_NW_VER
#define GEC_NW_VER 0
#endif
#ifndef GEC_TMAP_FROM_K
// uniform modes, TMA path: ONE 2-D tensor copy (k rows x 512 B) per work item instead of k 1-D copies, from this k
// on.  Measured (profiles/r02_kbench_tmap_and_large_k.log): the single copy saves ~7 issue slots per source row, which
// is what matters for k >= 13 (encode RS(20,4) 0.82 -> 0.94, RS(24,4) 0.77 -> 1.03, verify RS(16,4) 0.93 -> 0.99),
// but k <= 12 encode is faster with k independent 1-D copies in flight (RS(10,4) 1.015 vs 0.92).  0 = never.
#define GEC_TMAP_FROM_K 13
#endif
#define GEC_TMAP (GEC_TMAP_FROM_K > 0)
#ifndef GEC_SPLIT_STAGE
#define GEC_SPLIT_STAGE 1
#endif
#ifndef GEC_LDG_MAXLG
#define GEC_LDG_MAXLG 3  // LDG path: largest table group = 2^3 tables (64 contiguous bytes per shard and instruction)
#endif
#ifndef GEC_TMA_FROM_K
#define GEC_TMA_FROM_K 5  // encode / reconstruct use the TMA staging from this k on (sweep r02_s2: k <= 4 is as fast with LDG)
#endif

constexpr int kMaxK = 32;
constexpr int kMaxM = 8;
constexpr int kRowsPerPass = 4;          // output rows packed in one 32-bit table word
constexpr uint32_t kGroupBytes = 32768;  // one table group: 256 rows x 32 banks x 4 B
constexpr int kMaxGroups = 6;
constexpr uint32_t kStageRowBytes = 512;  // 32 columns x 16 B of one shard
constexpr uint32_t kSmemLimit = 227 * 1024;

enum ApplyMode { kModeEncode = 0, kModePlan = 1, kModeVerify = 2 };

// ---- table layout: k sources -> groups of 2^lg tables ---------------------------------------
struct TabLayout {
    int nslots;   // >= k; slots >= k are zero tables (only when the group budget forces padding)
    int ngroups;  // 32 KB each
    int lg[kMaxGroups];    // log2(tables in the group)
    int base[kMaxGroups];  // first slot of the group
};
// greedy decomposition of the smallest k' >= k that needs <= maxgroups groups of <= 2^maxlg tables
__host__ __device__ constexpr TabLayout make_layout(int k, int maxlg, int maxgroups)
{
    for (int kp = k; kp <= 2 * kMaxK; kp++) {
        TabLayout L{};
        int rem = kp, pos = 0, ng = 0;
        bool ok = true;
        while (rem > 0) {
            int lg = maxlg;
            while ((1 << lg) > rem) lg--;
            if (ng >= kMaxGroups || ng >= maxgroups) {
                ok = false;
                break;
            }
            L.lg[ng] = lg;
            L.base[ng] = pos;
            ng++;
            pos += 1 << lg;
            rem -= 1 << lg;
        }
        if (ok) {
            L.nslots = kp;
            L.ngroups = ng;
            return L;
        }
    }
    return TabLayout{};
}
__host__ __device__ constexpr int slot_group(const TabLayout &L, int u)
{
    int g = 0;
    for (int i = 0; i < L.ngroups; i++)
        if (u >= L.base[i]) g = i;
    return g;
}

// Per-stripe decode plan of one stripe as the streaming kernel needs it (two slots, one per
// table buffer).
struct PlanSlot {
    unsigned long long key_present, key_out;
    uint32_t sid;         // stripe index (>= n: no more work)
    int32_t rows;         // rows to produce in this pass (<= 0: nothing to do)
    uint32_t chunk_next;  // next unclaimed 32-column chunk of this stripe
    uint32_t len;         // shard_len of the stripe
    uint32_t src_off[kMaxK];             // byte offset of source j inside the stripe
    uint32_t dst_off[kRowsPerPass];      // byte offset of output row i inside the stripe
    uint8_t coef[kRowsPerPass * kMaxK];  // coef[i*kMaxK + j]
};
constexpr uint32_t kAuxBytes = 2 * sizeof(PlanSlot) + 8 * (4 + 32) + 64;  // plan slots + mbarriers

// Which way the columns reach the lanes, and how many warps stream, per (k, mode): picked from
// the sweeps on B200 (profiles/r02_sweep_tma_ldg_warps.log: both paths x 8..32 warps for
// k = 4, 6, 8, 10, 12).
__host__ __device__ constexpr bool cfg_default_tma(int k, int mode)
{
    if (mode == kModeVerify) return k == 4 || k > 6;  // verify: LDG with prefetch wins for k = 1..3, 5, 6
    // reconstruct of k = 7 (4+2+1: three table groups, 192 KB for two buffers): LDG 0.95 of peak, TMA with one
    // padded group of 8 and 27 warps 0.79 (profiles/r02_kbench_final.log)
    if (mode == kModePlan && k == 7) return false;
    return k >= GEC_TMA_FROM_K;
}
__host__ __device__ constexpr int cfg_nw_ldg(int k, int mode)
{
    if (mode == kModeVerify) return k <= 4 ? 24 : 16;
    return k <= 4 ? 32 : (k <= 6 ? 24 : (k <= 8 ? 20 : 16));
}
// TMA path, k <= 12: measured optimum (total warps; reconstruct includes the builder warp and is then
// clamped to what the stage memory allows); larger k: by register budget (cfg_nw_tma)
__host__ __device__ constexpr int cfg_nw_tma_small(int k, int mode)
{
    if (mode == kModePlan) return k <= 6 ? 32 : (k <= 8 ? 28 : 24);
    if (mode == kModeVerify) return k <= 4 ? 28 : (k <= 8 ? 20 : 16);
    return k <= 8 ? 20 : 16;
}
// TMA: at most 3 table groups per buffer, fewer (= more zero-table padding) when the table buffers
// would not leave room for the stages of `want_nw` warps (reconstruct doubles the tables: k = 7 as
// 4+2+1 is 192 KB of tables and 8 warps, as one padded group of 8 it is 64 KB and 28 warps)
__host__ __device__ constexpr int cfg_tma_groups(int k, int bufs, int stage_rows, int want_nw)
{
    for (int g = 3; g > 1; g--) {
        const TabLayout L = make_layout(k, 5, g);
        if ((uint32_t)bufs * L.ngroups * kGroupBytes + kAuxBytes + (uint32_t)want_nw * stage_rows * kStageRowBytes <= kSmemLimit) return g;
    }
    return 1;
}
__host__ __device__ constexpr int cfg_nw_tma(int regs_est, uint32_t tab_bytes, int stage_rows)
{
    // the register file is split over the 4 sub-partitions of an SM (16384 registers each), so the
    // per-thread budget only changes with ceil(warps / 4): 8 warps 255, 12: 168, 16: 128, 20: 96, 24: 80
    int nw = 8;
    for (int cand = 24; cand > 8; cand -= 4) {
        const int cap = 16384 / (cand / 4 * 32) / 8 * 8;
        if (cap >= regs_est) {
            nw = cand;
            break;
        }
    }
    while (nw > 4 && tab_bytes + kAuxBytes + (uint32_t)nw * stage_rows * kStageRowBytes > kSmemLimit) nw -= 4;
    return nw;
}

__host__ __device__ constexpr int cfg_fit_nw(int nw, uint32_t tab_bytes, int stage_rows, bool builder)
{
    while (nw > 4 && tab_bytes + kAuxBytes + (uint32_t)(nw - (builder ? 1 : 0)) * stage_rows * kStageRowBytes > kSmemLimit) nw -= 4;
    return nw;
}

// ---- launch shape / shared-memory carve-up per (K, MODE), all compile time ------------------
template <int K, int MODE> struct StreamCfg {
    static constexpr int kTmaOverride = MODE == kModeEncode ? GEC_TMA_ENC : (MODE == kModePlan ? GEC_TMA_PLAN : GEC_TMA_VER);
    static constexpr bool kTma = K > 16 || (kTmaOverride >= 0 ? (kTmaOverride != 0) : cfg_default_tma(K, MODE));
    static constexpr int kBufs = MODE == kModePlan ? 2 : 1;  // table buffers
    // reconstruct of k > 16: the stage holds ONE table group's rows (<= 16) at a time and an item is streamed
    // in one phase per group -- with two table buffers a full k x 512 B stage per warp leaves room for only
    // 7 consumer warps (RS(20,4) reconstruct 0.69 of peak)
    // (the same for encode / verify of k > 16: reading all k vectors of a column into registers at once spills)
    static constexpr bool kSplit = kTma && K > 16 && GEC_SPLIT_STAGE;
    static constexpr int kSrcRows = kSplit ? 16 : K;  // source rows of a stage; stored parity rows (verify) follow
    static constexpr int kStageRows = kTma ? kSrcRows + (MODE == kModeVerify ? kRowsPerPass : 0) : 0;
    static constexpr int kNwOverride = MODE == kModeEncode ? GEC_NW_ENC : (MODE == kModePlan ? GEC_NW_PLAN : GEC_NW_VER);

    // LDG: groups of <= 8 tables (>= 64 contiguous bytes per shard and warp instruction), tables
    // <= 192 KB so that >= 32 KB stay L1 (round 1: 224 KB of tables starved the global loads).
    // TMA: groups of <= 32 tables, <= 3 groups per buffer; the loads bypass L1.
    static constexpr int kMaxLg = kSplit ? 4 : (kTma ? 5 : GEC_LDG_MAXLG);
    static constexpr int kMaxGrp = kTma ? cfg_tma_groups(K, kBufs, kStageRows, K <= 12 ? 16 : 8) : 6 / kBufs;
    static constexpr TabLayout kLay = make_layout(K, kMaxLg, kMaxGrp);
    static constexpr int S = kLay.nslots;
    static constexpr uint32_t kTabBytes = (uint32_t)kBufs * kLay.ngroups * kGroupBytes;

    // consumer warps: LDG shapes from the round-1 sweeps (2 x S x 4 registers of column data);
    // TMA: S x 4 registers of column data, capped by the stage memory
    static constexpr int kWarpsDefault =
        !kTma ? cfg_nw_ldg(K, MODE)
              : (K <= 12 ? cfg_fit_nw(cfg_nw_tma_small(K, MODE), kTabBytes, kStageRows, MODE == kModePlan)
                 : (MODE == kModePlan && (K <= 16 || kSplit))
                     ? cfg_fit_nw(16, kTabBytes, kStageRows, true)  // sweep: RS(14,4) 0.81 -> 0.92, RS(16,4) 0.89 -> 0.95
                     : cfg_nw_tma(4 * (kSplit ? 16 : S) + 76, kTabBytes, kStageRows));
    // an override (tuning builds) is clamped to what the stage memory allows
    static constexpr int kWarpsAll =
        kNwOverride > 0 ? (kTma ? cfg_fit_nw(kNwOverride, kTabBytes, kStageRows, MODE == kModePlan) : kNwOverride) : kWarpsDefault;
    // reconstruct: the last warp is the table builder
    static constexpr int kWarps = MODE == kModePlan ? kWarpsAll - 1 : kWarpsAll;  // consumer warps
    static constexpr int kThreads = 32 * kWarpsAll;
    static constexpr uint32_t kStageBytes = (uint32_t)kWarps * kStageRows * kStageRowBytes;
    static constexpr uint32_t kSmem = kTabBytes + kStageBytes + kAuxBytes;
    static_assert(kLay.nslots >= K && kLay.ngroups >= 1, "no table layout for this k");
    static_assert(kSmem <= kSmemLimit, "shared memory budget exceeded");
    static_assert(kThreads <= 1024 && kWarps >= 1, "bad launch shape");
};

// GF(2^8) antilog / log tables, pinned in constant memory.  Kernels that need general products
// (decode planning) stage them into shared memory with warp-UNIFORM 16-byte constant loads:
// a per-lane byte index into __constant__ memory serialises 32-way in the constant cache (the
// first version of rs_plan_kernel spent 30 of its 40 us there).
struct GfTables {
    uint8_t exp[512];
    uint8_t log[256];
};
__constant__ __align__(16) GfTables c_gf = {GARAGE_EC_GF_EXP_INIT, GARAGE_EC_GF_LOG_INIT};

__device__ __forceinline__ void stage_gf_tables(uint8_t *s_gf /* 768 B, 16-byte aligned */)
{
    const uint4 *src = reinterpret_cast<const uint4 *>(&c_gf);
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (uint32_t i = warp; i < sizeof(GfTables) / 16; i += nwarps) {
        const uint4 v = src[i];  // same address in every lane: one constant-cache broadcast
        if (lane < 4)
            reinterpret_cast<uint32_t *>(s_gf)[i * 4 + lane] = lane == 0 ? v.x : (lane == 1 ? v.y : (lane == 2 ? v.z : v.w));
    }
}

// Per-stripe decode plan, produced by rs_plan_kernel, consumed by rs_apply_kernel<kModePlan>.
struct __align__(16) StripePlan {
    unsigned long long key_present;  // bit i: shard i present
    unsigned long long key_out;      // bit i: shard i is rebuilt
    uint8_t nrows;                   // number of shards rebuilt (0..m)
    uint8_t unrecoverable;           // 1 if < k present
    uint8_t pad[6];
    uint8_t surv[kMaxK];           // source shard indices (first k present)
    uint8_t out_idx[kMaxM];        // rebuilt shard indices
    uint8_t coef[kMaxM][kMaxK];  // out[r] = XOR_j coef[r][j] * shard[surv[j]]
};

struct ApplyParams {
    const uint8_t *src;            // stripe s source base = src + s*src_pitch
    uint8_t *dst;                  // stripe s output base = dst + s*dst_pitch
    unsigned long long src_pitch;  // bytes
    unsigned long long dst_pitch;
    const uint32_t *shard_len;  // device, nullable (=> stride)
    const StripePlan *plan;     // kModePlan
    uint32_t *mismatch;         // kModeVerify
    uint32_t *counter;          // kModePlan dynamic scheduler
    uint32_t stride;            // bytes between shards
    uint32_t n;                 // stripes
    uint32_t k;                 // sources
    uint32_t rows;              // outputs this pass (<= 4), uniform modes
    uint32_t row_off;           // first output row of this pass
    uint32_t items_per_stripe;  // ceil(ceil(stride/16)/32), uniform modes
    uint32_t row_bytes;         // 128: bytes per table row (a register operand keeps x*128 an IMAD)
    uint32_t use_tmap;          // 1: `tmap` is valid (uniform modes, TMA path)
    uint32_t rows_per_stripe;   // shards per stripe in `src` (k for encode, k+m for verify): tensor row of (s, j) = s*rows_per_stripe + j
    uint8_t coef[kRowsPerPass * kMaxK];  // uniform modes: coef[i*k + j]
    // 2-D view of `src` for TMA: dim0 = stride/4 uint32 elements, dim1 = n*rows_per_stripe shards
    // (pitch `stride`), box = 128 elements (512 B = 32 columns) x k rows
    alignas(64) CUtensorMap tmap;
};

// ------------------------------------------------------------------ small device helpers
template <int I, int N, class F> __device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}

__device__ __forceinline__ uint4 ldg_stream(const void *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream(void *p, const uint4 &v)
{
    asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(addr));
    return r;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr)
{
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr) : "memory");
    return r;
}
// zero the bytes at positions >= nbytes (0 < nbytes < 16) of a 16-byte vector
__device__ __forceinline__ uint4 mask_tail(uint4 v, uint32_t nbytes)
{
    uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int lo = 4 * i;
        if ((int)nbytes <= lo) w[i] = 0;
        else if ((int)nbytes < lo + 4) w[i] &= 0xffffffffu >> (8 * (lo + 4 - (int)nbytes));
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// ---- mbarrier + 1-D bulk async copy (TMA) ----------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "GEC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra GEC_DONE;\n"
        "bra GEC_WAIT;\n"
        "GEC_DONE:\n"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// global -> this CTA's shared memory, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// 2-D tiled TMA: box (128 uint32 x K rows) at element column c0, row c1 of the tensor described by
// `tmap` -> dst (row r at dst + r*512); completes 512*K bytes on `bar` (also when the box sticks
// out of the tensor: out-of-bounds elements are filled with zeros and still counted)
__device__ __forceinline__ void tensor_g2s_2d(uint32_t dst, const CUtensorMap *tmap, uint32_t c0, uint32_t c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}

// 4x4 byte transpose: a[p] holds {row0,row1,row2,row3} bytes of byte column p;
// returns r[i] = bytes of row i for columns 0..3.
__device__ __forceinline__ void transpose4x4(const uint32_t a0, const uint32_t a1, const uint32_t a2,
                                             const uint32_t a3, uint32_t &r0, uint32_t &r1,
                                             uint32_t &r2, uint32_t &r3)
{
    const uint32_t t0 = __byte_perm(a0, a1, 0x5140);  // a0.b0 a1.b0 a0.b1 a1.b1
    const uint32_t t1 = __byte_perm(a2, a3, 0x5140);
    const uint32_t t2 = __byte_perm(a0, a1, 0x7362);  // a0.b2 a1.b2 a0.b3 a1.b3
    const uint32_t t3 = __byte_perm(a2, a3, 0x7362);
    r0 = __byte_perm(t0, t1, 0x5410);
    r1 = __byte_perm(t0, t1, 0x7632);
    r2 = __byte_perm(t2, t3, 0x5410);
    r3 = __byte_perm(t2, t3, 0x7632);
}

// multiply four packed GF(2^8) bytes by alpha (= 2): shift left, reduce by 0x11D where bit 7 was set
__device__ __forceinline__ uint32_t xtime4(uint32_t v)
{
    const uint32_t hi = v & 0x80808080u;
    return ((v ^ hi) << 1) ^ ((hi >> 7) * 0x1du);
}

// ------------------------------------------------------------------ product tables
// Build the tables of `rows` (<= 4) coefficient rows coef[i*cstride + j], j < K, into one table
// buffer; slots >= K are zero.  Entry x of table j is XOR_{bit b of x} (packed column j)*alpha^b.
// Every lane owns one 16-byte bank quad (qd = lane & 7) of the rows x = 4*g + (lane >> 3): it
// keeps the eight powers of its quad's table(s) in registers and walks g in Gray-code order, so
// an entry costs ONE xor per table, and one STS.128 instruction of the warp writes 4 full rows
// (512 B over all 32 banks, the minimum 4 wavefronts).  Work unit = (group, 8 Gray steps);
// units are dealt round-robin to the `nw` participating warps (`w` = this warp's index).
template <class LAYC>
__device__ __forceinline__ void build_tables(uint32_t *tab, const uint8_t *coef, uint32_t cstride, uint32_t rows,
                                             uint32_t w, uint32_t nw, int K)
{
    constexpr TabLayout LAY = LAYC::kLay;
    const uint32_t lane = threadIdx.x & 31, qd = lane & 7, xs = lane >> 3;
    auto packed_col = [&](uint32_t j) -> uint32_t {
        uint32_t cur = 0;
        if (j < (uint32_t)K) {
#pragma unroll
            for (uint32_t i = 0; i < kRowsPerPass; i++)
                if (i < rows) cur |= (uint32_t)coef[i * cstride + j] << (8 * i);
        }
        return cur;
    };
    static_for<0, LAY.ngroups>([&](auto gc) {
        constexpr int g = decltype(gc)::value;
        constexpr int lg = LAY.lg[g];
        constexpr int NTQ = lg <= 3 ? 1 : (lg == 4 ? 2 : 4);  // tables inside one bank quad
        // does this warp own a unit of this group at all?
        bool any = false;
#pragma unroll
        for (int sg = 0; sg < 8; sg++) any |= ((uint32_t)(g * 8 + sg) % nw) == w;
        if (!any) return;
        uint32_t pw[NTQ][8];
#pragma unroll
        for (int t = 0; t < NTQ; t++) {
            // banks 4*qd + (4/NTQ)*t ... belong to table (bank >> (5 - lg)) of the group
            const uint32_t bank = 4 * qd + (4 / NTQ) * t;
            uint32_t cur = packed_col(LAY.base[g] + (bank >> (5 - lg)));
#pragma unroll
            for (int b = 0; b < 8; b++) {
                pw[t][b] = cur;
                cur = xtime4(cur);
            }
        }
#pragma unroll 1
        for (uint32_t sg = 0; sg < 8; sg++) {
            if (((uint32_t)(g * 8) + sg) % nw != w) continue;
            const uint32_t n0 = sg * 8;
            uint32_t gx = n0 ^ (n0 >> 1);  // Gray code of the first step of the segment
            uint32_t e[NTQ];
#pragma unroll
            for (int t = 0; t < NTQ; t++) {
                uint32_t v = 0;
                if (xs & 1) v ^= pw[t][0];
                if (xs & 2) v ^= pw[t][1];
#pragma unroll
                for (int b = 0; b < 6; b++)
                    if ((gx >> b) & 1) v ^= pw[t][2 + b];
                e[t] = v;
            }
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const uint32_t x = gx * 4 + xs;
                uint4 v;
                if (NTQ == 1) v = make_uint4(e[0], e[0], e[0], e[0]);
                else if (NTQ == 2) v = make_uint4(e[0], e[0], e[NTQ - 1], e[NTQ - 1]);
                else v = make_uint4(e[0], e[1 % NTQ], e[2 % NTQ], e[3 % NTQ]);
                *reinterpret_cast<uint4 *>(tab + (size_t)g * (kGroupBytes / 4) + x * 32 + qd * 4) = v;
                if (i < 7) {
                    // Gray step n -> n+1 flips bit ctz(n+1); inside an aligned segment of 8 it only
                    // depends on i
                    const int c = (i & 1) == 0 ? 0 : ((i & 3) == 1 ? 1 : 2);
                    gx ^= 1u << c;
#pragma unroll
                    for (int t = 0; t < NTQ; t++) e[t] ^= pw[t][2 + c];
                }
            }
        }
    });
}

// 16 table lookups for one 16-byte vector; acc[4*w + p] ^= T[byte p of word w]
//   base = shared address of (group, this lane's bank for this phase); row_bytes = 128
// The streaming kernels sit at ~75-80 % issue and ~70 % alu-pipe utilisation (ncu, round 2), so
// the per-byte instruction count is what is left to win:
//  * GEC_DP4A: the table address  base + byte_p * 128  is ONE integer dot product,
//    dp4a(word, 0x80 << 8p, base) = base + 128 * byte_p, instead of PRMT (byte extract, alu pipe)
//    + IMAD (scale and add, fma pipe);
//  * GEC_XOR3: two sources are accumulated by one three-input LOP3 (a ^ b ^ c).
#ifndef GEC_DP4A
#define GEC_DP4A 1
#endif
#ifndef GEC_XOR3
#define GEC_XOR3 1
#endif
__device__ __forceinline__ uint32_t table_addr(uint32_t w, int p, uint32_t base, uint32_t row_bytes)
{
#if GEC_DP4A
    (void)row_bytes;
    return __dp4a(w, 0x80u << (8 * p), base);
#else
    const uint32_t x = __byte_perm(w, 0, 0x4440 + p);  // byte p, zero extended (alu pipe)
    return x * row_bytes + base;                        // IMAD (fma pipe)
#endif
}
__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
template <bool kFirst>
__device__ __forceinline__ void lookup16(uint32_t (&acc)[16], const uint4 &d, uint32_t base,
                                         uint32_t row_bytes)
{
    const uint32_t w[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
        for (int p = 0; p < 4; p++) {
            const uint32_t v = lds_u32(table_addr(w[i], p, base, row_bytes));
            if (kFirst) acc[4 * i + p] = v;
            else acc[4 * i + p] ^= v;
        }
    }
}
// two sources at once: acc = acc ^ T_a[..] ^ T_b[..] in one LOP3
template <bool kFirst>
__device__ __forceinline__ void lookup16x2(uint32_t (&acc)[16], const uint4 &da, uint32_t base_a, const uint4 &db,
                                           uint32_t base_b, uint32_t row_bytes)
{
    const uint32_t wa[4] = {da.x, da.y, da.z, da.w}, wb[4] = {db.x, db.y, db.z, db.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
        for (int p = 0; p < 4; p++) {
            const uint32_t va = lds_u32(table_addr(wa[i], p, base_a, row_bytes));
            const uint32_t vb = lds_u32(table_addr(wb[i], p, base_b, row_bytes));
            if (kFirst) acc[4 * i + p] = va ^ vb;
            else acc[4 * i + p] = xor3(acc[4 * i + p], va, vb);
        }
    }
}

__device__ __forceinline__ void rows_from_acc(const uint32_t (&acc)[16], uint4 (&r)[4])
{
    uint32_t o[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++)
        transpose4x4(acc[4 * i + 0], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3], o[0][i], o[1][i],
                     o[2][i], o[3][i]);
#pragma unroll
    for (int row = 0; row < 4; row++) r[row] = make_uint4(o[row][0], o[row][1], o[row][2], o[row][3]);
}

// Source shard read by this lane in slot u: slot u = phase p of group g; sub-warp q = lane / R
// of the group works on source base + (p xor q).
template <class CFG, int U> __device__ __forceinline__ uint32_t lane_source(uint32_t lane)
{
    constexpr TabLayout LAY = CFG::kLay;
    constexpr int g = slot_group(LAY, U);
    constexpr int lg = LAY.lg[g];
    constexpr int ph = U - LAY.base[g];
    return (uint32_t)LAY.base[g] + ((uint32_t)ph ^ (lg ? (lane >> (5 - lg)) : 0u));
}
template <class CFG, int U> __device__ __forceinline__ constexpr bool slot_may_pad()
{
    constexpr TabLayout LAY = CFG::kLay;
    constexpr int g = slot_group(LAY, U);
    return LAY.base[g] + (1 << LAY.lg[g]) > (int)CFG::kK;
}

// LDG: one 16-byte column of every source straight into registers.
//   sp     : address of this lane's column in source 0 (uniform modes) / shard 0 (plan mode)
//   kPlan  : source j lives at sp + src_off[j] (smem) instead of sp + j*stride
template <class CFG, bool kPlan>
__device__ __forceinline__ void column_load(const uint8_t *sp, uint32_t stride, const uint32_t *src_off,
                                            uint32_t lane, uint4 (&d)[CFG::S])
{
    static_for<0, CFG::S>([&](auto uc) {
        constexpr int u = decltype(uc)::value;
        const uint32_t j = lane_source<CFG, u>(lane);
        if (!slot_may_pad<CFG, u>() || j < (uint32_t)CFG::kK) d[u] = ldg_stream(sp + (kPlan ? src_off[j] : j * stride));
        else d[u] = make_uint4(0, 0, 0, 0);
    });
}
// TMA: the same vectors out of the warp's stage (row j = source j, 512 B per row)
template <class CFG>
__device__ __forceinline__ void stage_read(uint32_t stage_lane_addr /* stage + lane*16 */, uint32_t lane,
                                           uint4 (&d)[CFG::S])
{
    static_for<0, CFG::S>([&](auto uc) {
        constexpr int u = decltype(uc)::value;
        const uint32_t j = lane_source<CFG, u>(lane);
        if (!slot_may_pad<CFG, u>() || j < (uint32_t)CFG::kK) d[u] = lds_v4(stage_lane_addr + j * kStageRowBytes);
        else d[u] = make_uint4(0, 0, 0, 0);
    });
}

// look up + transpose -> r[row] (uint4) for the slots of one column
//   tab_addr : shared address of the table buffer
template <class CFG>
__device__ __forceinline__ void column_compute(uint4 (&d)[CFG::S], uint32_t tab_addr, uint32_t lane,
                                               uint32_t row_bytes, uint32_t tail_bytes, uint4 (&r)[4])
{
    constexpr TabLayout LAY = CFG::kLay;
    uint32_t acc[16];
    if (tail_bytes) {
#pragma unroll
        for (int u = 0; u < CFG::S; u++) d[u] = mask_tail(d[u], tail_bytes);
    }
    // this lane's bank at phase ph of group g: lane xor ph*R
    auto slot_base = [&](auto uc) -> uint32_t {
        constexpr int u = decltype(uc)::value;
        constexpr int g = slot_group(LAY, u);
        constexpr int lg = LAY.lg[g];
        constexpr int ph = u - LAY.base[g];
        return tab_addr + (uint32_t)g * kGroupBytes + ((lane ^ ((uint32_t)ph << (lg ? 5 - lg : 0))) << 2);
    };
#if GEC_XOR3
    static_for<0, CFG::S / 2>([&](auto pc) {
        constexpr int u = 2 * decltype(pc)::value;
        lookup16x2<u == 0>(acc, d[u], slot_base(std::integral_constant<int, u>{}), d[u + 1],
                           slot_base(std::integral_constant<int, u + 1>{}), row_bytes);
    });
    if constexpr (CFG::S % 2 == 1)
        lookup16<CFG::S == 1>(acc, d[CFG::S - 1], slot_base(std::integral_constant<int, CFG::S - 1>{}), row_bytes);
#else
    static_for<0, CFG::S>([&](auto uc) {
        constexpr int u = decltype(uc)::value;
        lookup16<u == 0>(acc, d[u], slot_base(uc), row_bytes);
    });
#endif
    rows_from_acc(acc, r);
}

// ---- one table group at a time (split staging): rows of group g sit at stage rows 0..size-1
template <class CFG, int G>
__device__ __forceinline__ void group_read(uint32_t stage_lane_addr, uint32_t lane, uint4 (&d)[16])
{
    constexpr TabLayout LAY = CFG::kLay;
    constexpr int lg = LAY.lg[G], n = 1 << lg;
    static_for<0, n>([&](auto pc) {
        constexpr int ph = decltype(pc)::value;
        const uint32_t row = (uint32_t)ph ^ (lg ? (lane >> (5 - lg)) : 0u);  // source base + row
        if (LAY.base[G] + n <= (int)CFG::kK || (uint32_t)LAY.base[G] + row < (uint32_t)CFG::kK)
            d[ph] = lds_v4(stage_lane_addr + row * kStageRowBytes);
        else d[ph] = make_uint4(0, 0, 0, 0);
    });
}
template <class CFG, int G>
__device__ __forceinline__ void group_lookup(uint32_t (&acc)[16], uint4 (&d)[16], uint32_t tab_addr, uint32_t lane,
                                             uint32_t row_bytes, uint32_t tail_bytes)
{
    constexpr TabLayout LAY = CFG::kLay;
    constexpr int lg = LAY.lg[G], n = 1 << lg;
    if (tail_bytes) {
#pragma unroll
        for (int u = 0; u < n; u++) d[u] = mask_tail(d[u], tail_bytes);
    }
    auto base_of = [&](int ph) -> uint32_t {
        return tab_addr + (uint32_t)G * kGroupBytes + ((lane ^ ((uint32_t)ph << (lg ? 5 - lg : 0))) << 2);
    };
    if constexpr (n == 1) {
        if (G == 0) lookup16<true>(acc, d[0], base_of(0), row_bytes);
        else lookup16<false>(acc, d[0], base_of(0), row_bytes);
    } else {
        static_for<0, n / 2>([&](auto pc) {
            constexpr int u = 2 * decltype(pc)::value;
            if (G == 0 && u == 0) lookup16x2<true>(acc, d[u], base_of(u), d[u + 1], base_of(u + 1), row_bytes);
            else lookup16x2<false>(acc, d[u], base_of(u), d[u + 1], base_of(u + 1), row_bytes);
        });
    }
}

// ------------------------------------------------------------------ the streaming kernel
template <int K, int MODE> struct KernelCfg : StreamCfg<K, MODE> {
    static constexpr int kK = K;
};

template <int K, int MODE>
__global__ void __launch_bounds__(StreamCfg<K, MODE>::kThreads, 1) rs_apply_kernel(const __grid_constant__ ApplyParams p)
{
    using CFG = KernelCfg<K, MODE>;
    constexpr int S = CFG::S;
    constexpr int NW = CFG::kWarps;  // consumer warps
    constexpr bool TMA = CFG::kTma;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *const tab = reinterpret_cast<uint32_t *>(smem_raw);
    const uint32_t tab_addr = (uint32_t)__cvta_generic_to_shared(smem_raw);
    const uint32_t stage_addr = tab_addr + CFG::kTabBytes + warp * (CFG::kStageRows * kStageRowBytes);
    PlanSlot *const slot = reinterpret_cast<PlanSlot *>(smem_raw + CFG::kTabBytes + CFG::kStageBytes);
    const uint32_t bars = tab_addr + CFG::kTabBytes + CFG::kStageBytes + 2 * (uint32_t)sizeof(PlanSlot);
    const uint32_t bar_full = bars, bar_empty = bars + 16, bar_stage = bars + 32 + warp * 8;  // full[2], empty[2], stage[NW]

    if (tid == 0) {
        mbar_init(bar_full, 32);
        mbar_init(bar_full + 8, 32);
        mbar_init(bar_empty, NW * 32);
        mbar_init(bar_empty + 8, NW * 32);
    }
    if (TMA && lane == 0 && warp < (uint32_t)NW) mbar_init(bar_stage, 1);
    mbar_fence_init();
    uint32_t stage_parity = 0;

    // TMA: lane 0 arms the warp's stage with `nrow` x `rb` bytes; the copies are issued by the caller
    if constexpr (MODE != kModePlan) {
        // ---- uniform coefficient matrix: build once, then warps stream items ----------------
        build_tables<CFG>(tab, p.coef, K, p.rows, warp, (uint32_t)NW, K);
        __syncthreads();

        const uint32_t ips = p.items_per_stripe;
        const uint32_t total = p.n * ips;  // host guarantees < 2^32
        const uint32_t gwarps = gridDim.x * NW;

        // position of this lane's column for a work item (stripe, 32-column chunk)
        struct Pos {
            const uint8_t *sp;  // this lane's column in source 0
            uint32_t s, col, tail, rb;
            bool valid, any;  // this lane has a column / the warp has at least one
        };
        auto locate = [&](uint32_t item) -> Pos {
            Pos z;
            z.s = item / ips;
            const uint32_t c = item - z.s * ips;
            const uint32_t len = p.shard_len ? __ldg(p.shard_len + z.s) : p.stride;
            const uint32_t nvec = (len + 15) >> 4;
            z.col = c * 32 + lane;
            z.valid = z.col < nvec;
            z.any = c * 32 < nvec;
            z.tail = (z.col == nvec - 1) ? (len & 15) : 0;
            z.rb = z.any ? min(kStageRowBytes, (nvec - c * 32) * 16) : 0;
            z.sp = p.src + (unsigned long long)z.s * p.src_pitch + (size_t)z.col * 16;
            return z;
        };
        // TMA: arm the stage and bring in the staged rows (lane 0): one 2-D tensor copy for the K source
        // rows when the host supplied a tensor map, else one 1-D bulk copy per row
        auto issue = [&](const Pos &z) {
            if (!z.any || lane != 0) return;  // lane 0's column is the first of the chunk
            constexpr int NR = CFG::kStageRows;
            const uint32_t prow = MODE == kModeVerify ? p.rows : 0u;  // stored parity rows staged behind the sources
            if (GEC_TMAP && K >= GEC_TMAP_FROM_K && p.use_tmap) {
                mbar_arrive_expect_tx(bar_stage, kStageRowBytes * K + z.rb * prow);
                tensor_g2s_2d(stage_addr, &p.tmap, (z.col >> 5) * (kStageRowBytes / 4), z.s * p.rows_per_stripe, bar_stage);
            } else {
                mbar_arrive_expect_tx(bar_stage, z.rb * ((uint32_t)K + prow));
#pragma unroll
                for (int j = 0; j < K; j++) bulk_g2s(stage_addr + j * kStageRowBytes, z.sp + (size_t)j * p.stride, z.rb, bar_stage);
            }
#pragma unroll
            for (int j = K; j < NR; j++)
                if ((uint32_t)(j - K) < prow)
                    bulk_g2s(stage_addr + j * kStageRowBytes, z.sp + (size_t)(j + p.row_off) * p.stride, z.rb, bar_stage);
        };
        auto finish = [&](const Pos &z, const uint4 (&r)[4], const uint4 (&st)[4]) {
            uint32_t mm = 0;
            if (MODE == kModeEncode) {
                if (z.valid) {
                    uint8_t *dp = p.dst + (unsigned long long)z.s * p.dst_pitch + (size_t)z.col * 16;
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        if (i < (int)p.rows) stg_stream(dp + (size_t)i * p.stride, r[i]);
                }
            } else {
                if (z.valid) {
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        if (i < (int)p.rows) {
                            uint4 sv = st[i];
                            if (z.tail) sv = mask_tail(sv, z.tail);
                            const uint32_t diff = (sv.x ^ r[i].x) | (sv.y ^ r[i].y) | (sv.z ^ r[i].z) | (sv.w ^ r[i].w);
                            if (diff) mm |= 1u << (p.row_off + i);
                        }
                    }
                }
                // warp-shuffle OR reduction of the per-lane mismatch bits, one atomic per warp
                mm = __reduce_or_sync(0xffffffffu, mm);
                if (mm && lane == 0) atomicOr(p.mismatch + z.s, mm);
            }
        };
        // stored parity rows of a verify item (they follow the k data shards of the same stripe)
        auto load_stored = [&](const Pos &z, uint4 (&st)[4]) {
            if (MODE != kModeVerify) return;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                st[i] = make_uint4(0, 0, 0, 0);
                if (i < (int)p.rows && z.valid) {
                    if (TMA) st[i] = lds_v4(stage_addr + lane * 16 + (CFG::kSrcRows + i) * kStageRowBytes);
                    else st[i] = ldg_stream(z.sp + (size_t)(K + p.row_off + i) * p.stride);
                }
            }
        };

        uint32_t item = blockIdx.x * NW + warp;
        if constexpr (CFG::kSplit) {
            // k > 16: one table group (<= 16 sources) per phase; the stage is refilled with the next group
            // (or the first group of the next item) as soon as the current one sits in registers
            constexpr TabLayout LAY = CFG::kLay;
            constexpr int NG = LAY.ngroups;
            auto issue_g = [&](const Pos &z, auto gc) {
                constexpr int g = decltype(gc)::value;
                constexpr int nrow = (LAY.base[g] + (1 << LAY.lg[g]) <= K) ? (1 << LAY.lg[g]) : (K - LAY.base[g]);
                if (!z.any || lane != 0) return;
                const uint32_t prow = (MODE == kModeVerify && g == NG - 1) ? p.rows : 0u;  // stored parity rides with the last group
                if (GEC_TMAP && p.use_tmap) {
                    // box = 16 rows: rows past this group are the next sources (or zero fill at the end of the
                    // tensor); they are fetched and ignored
                    mbar_arrive_expect_tx(bar_stage, kStageRowBytes * 16 + z.rb * prow);
                    tensor_g2s_2d(stage_addr, &p.tmap, (z.col >> 5) * (kStageRowBytes / 4),
                                  z.s * p.rows_per_stripe + LAY.base[g], bar_stage);
                } else {
                    mbar_arrive_expect_tx(bar_stage, z.rb * ((uint32_t)nrow + prow));
#pragma unroll 1  // fallback path (no tensor map: stride < 512 B): keep it out of the register budget
                    for (int r = 0; r < nrow; r++)
                        bulk_g2s(stage_addr + r * kStageRowBytes, z.sp + (size_t)(LAY.base[g] + r) * p.stride, z.rb, bar_stage);
                }
#pragma unroll 1
                for (uint32_t i = 0; i < prow; i++)
                    bulk_g2s(stage_addr + (CFG::kSrcRows + i) * kStageRowBytes, z.sp + (size_t)(K + p.row_off + i) * p.stride, z.rb,
                             bar_stage);
            };
            Pos nx;
            nx.valid = nx.any = false;
            if (item < total) {
                nx = locate(item);
                issue_g(nx, std::integral_constant<int, 0>{});
            }
            while (item < total) {
                const Pos cur = nx;
                if (!cur.any) {  // chunk past the end of a short stripe: nothing was staged for it
                    item += gwarps;
                    nx.valid = nx.any = false;
                    if (item < total) {
                        nx = locate(item);
                        issue_g(nx, std::integral_constant<int, 0>{});
                    }
                    continue;
                }
                uint32_t acc[16];
                uint4 st[4];
                static_for<0, NG>([&](auto gc) {
                    constexpr int g = decltype(gc)::value;
                    uint4 d[16];
                    mbar_wait(bar_stage, stage_parity);
                    stage_parity ^= 1;
                    group_read<CFG, g>(stage_addr + lane * 16, lane, d);
                    if (g == NG - 1) load_stored(cur, st);
                    __syncwarp();  // every lane has its vectors: the stage may be refilled
                    if constexpr (g + 1 < NG) {
                        issue_g(cur, std::integral_constant<int, g + 1>{});
                    } else {
                        item += gwarps;
                        nx.valid = nx.any = false;
                        if (item < total) {
                            nx = locate(item);
                            issue_g(nx, std::integral_constant<int, 0>{});
                        }
                    }
                    if (cur.valid) group_lookup<CFG, g>(acc, d, tab_addr, lane, p.row_bytes, cur.tail);
                });
                uint4 r[4];
                if (cur.valid) rows_from_acc(acc, r);
                finish(cur, r, st);
            }
        } else if constexpr (TMA) {
            Pos nx;
            nx.valid = nx.any = false;
            if (item < total) {
                nx = locate(item);
                issue(nx);
            }
            while (item < total) {
                const Pos cur = nx;
                uint4 d[S], st[4];
                if (cur.any) {
                    mbar_wait(bar_stage, stage_parity);
                    stage_parity ^= 1;
                    stage_read<CFG>(stage_addr + lane * 16, lane, d);
                    load_stored(cur, st);
                }
                __syncwarp();  // every lane has its vectors: the stage may be refilled
                item += gwarps;
                nx.valid = nx.any = false;
                if (item < total) {
                    nx = locate(item);
                    issue(nx);
                }
                uint4 r[4];
                if (cur.valid) column_compute<CFG>(d, tab_addr, lane, p.row_bytes, cur.tail, r);
                finish(cur, r, st);
            }
        } else {
            uint4 dn[S], stn[4];
            Pos nx;
            nx.valid = nx.any = false;
            if (item < total) {
                nx = locate(item);
                if (nx.valid) column_load<CFG, false>(nx.sp, p.stride, nullptr, lane, dn);
                load_stored(nx, stn);
            }
            while (item < total) {
                uint4 d[S], st[4];
#pragma unroll
                for (int u = 0; u < S; u++) d[u] = dn[u];
#pragma unroll
                for (int i = 0; i < 4; i++) st[i] = stn[i];
                const Pos cur = nx;
                item += gwarps;
                nx.valid = nx.any = false;
                if (item < total) {
                    nx = locate(item);
                    if (nx.valid) column_load<CFG, false>(nx.sp, p.stride, nullptr, lane, dn);
                    load_stored(nx, stn);
                }
                uint4 r[4];
                if (cur.valid) column_compute<CFG>(d, tab_addr, lane, p.row_bytes, cur.tail, r);
                finish(cur, r, st);
            }
        }
    } else {
        // ---- per-stripe matrices, no block-wide barrier after this one --------------------------
        __syncthreads();  // mbarriers initialised
        constexpr uint32_t kTabBuf = CFG::kTabBytes / 2;
        if (warp == (uint32_t)NW) {
            // ===== builder warp: claim stripes, stage their plans, build their tables one stripe
            // ahead of the consumers.  Stripe sequence number i uses buffer / slot i & 1.
            uint32_t claimed = 0;
            if (lane == 0) claimed = atomicAdd(p.counter, 1u);
            // pattern whose tables each buffer holds (scalars, not arrays: `b` is a run-time index)
            unsigned long long bp0 = ~0ull, bp1 = ~0ull, bo0 = ~0ull, bo1 = ~0ull;
            bool have0 = false, have1 = false;
            for (uint32_t i = 0;; i++) {
                const uint32_t b = i & 1, use = i >> 1;
                // every consumer warp has left the stripe that used this buffer and slot
                if (use >= 1) mbar_wait(bar_empty + 8 * b, (use - 1) & 1);
                PlanSlot &ps = slot[b];
                const uint32_t s = __shfl_sync(0xffffffffu, claimed, 0);
                if (lane == 0) claimed = atomicAdd(p.counter, 1u);  // consumed by the next iteration
                int rows = 0;
                unsigned long long kp = 0, ko = 0;
                if (s < p.n) {
                    const StripePlan *pl = p.plan + s;
                    rows = pl->unrecoverable ? 0 : min(kRowsPerPass, (int)pl->nrows - (int)p.row_off);
                    if (rows > 0) {
                        if (lane < (uint32_t)K) ps.src_off[lane] = (uint32_t)pl->surv[lane] * p.stride;
                        if (lane < (uint32_t)rows) ps.dst_off[lane] = (uint32_t)pl->out_idx[p.row_off + lane] * p.stride;
                        for (uint32_t e = lane; e < (uint32_t)rows * kMaxK; e += 32)
                            ps.coef[e] = pl->coef[p.row_off + e / kMaxK][e % kMaxK];
                        kp = pl->key_present;
                        ko = pl->key_out;
                    }
                }
                if (lane == 0) {
                    ps.sid = s;
                    ps.rows = rows;
                    ps.chunk_next = 0;
                    ps.len = s < p.n ? (p.shard_len ? __ldg(p.shard_len + s) : p.stride) : 0;
                }
                __syncwarp();
                const bool same = b ? (have1 && kp == bp1 && ko == bo1) : (have0 && kp == bp0 && ko == bo0);
                if (rows > 0 && !same) {
                    build_tables<CFG>(tab + b * (kTabBuf / 4), ps.coef, kMaxK, (uint32_t)rows, 0, 1, K);
                    if (b) {
                        bp1 = kp;
                        bo1 = ko;
                        have1 = true;
                    } else {
                        bp0 = kp;
                        bo0 = ko;
                        have0 = true;
                    }
                }
                mbar_arrive(bar_full + 8 * b);  // all 32 lanes: each lane's table stores are released by its own arrive
                if (s >= p.n) break;
            }
            return;
        }

        // ===== consumer warps
        constexpr uint32_t kNone = 0xffffffffu;
        uint32_t pos = 0;      // stripe sequence number the search is at
        bool entered = false;  // full[pos] has been waited for
        bool ended = false;    // the terminal slot (sid >= n) was seen
        uint32_t pend = kNone; // sequence number of the item whose lookups are still to run
        struct It {
            uint32_t seq, s, chunk, nvec, len;
            int rows;
            bool valid;
        };
        // this warp will not touch tables / slot of sequence i again (every lane arrives: each
        // lane's own reads are ordered before its own release)
        auto leave = [&](uint32_t i) { mbar_arrive(bar_empty + 8 * (i & 1)); };
        // next work item of this warp; never waits for full[j] with j > lim (the builder may need
        // this warp's `leave` of an older stripe first)
        auto find = [&](uint32_t lim, It &it) {
            it.valid = false;
            while (!ended) {
                if (!entered) {
                    if (pos > lim) return;
                    mbar_wait(bar_full + 8 * (pos & 1), (pos >> 1) & 1);
                    entered = true;
                }
                PlanSlot &ps = slot[pos & 1];
                const uint32_t s = ps.sid;
                if (s >= p.n) {
                    ended = true;
                    return;
                }
                const int rows = ps.rows;
                if (rows > 0) {
                    const uint32_t len = ps.len, nvec = (len + 15) >> 4;
                    uint32_t c = 0;
                    if (lane == 0) c = atomicAdd(&ps.chunk_next, 1u);
                    c = __shfl_sync(0xffffffffu, c, 0);
                    if (c * 32 < nvec) {
                        it.seq = pos;
                        it.s = s;
                        it.chunk = c;
                        it.nvec = nvec;
                        it.len = len;
                        it.rows = rows;
                        it.valid = true;
                        return;
                    }
                }
                if (pos != pend) leave(pos);  // else: deferred until the pending lookups are done
                pos++;
                entered = false;
            }
        };
        // start bringing in the columns of an item: TMA copies into the stage / LDG into dn
        uint4 dn[TMA ? 1 : S];
        // split staging: rows of table group g only (stage row r = source base_g + r)
        auto fetch_group = [&](const It &it, auto gc) {
            constexpr int g = decltype(gc)::value;
            constexpr TabLayout LAY = CFG::kLay;
            constexpr int nrow = (LAY.base[g] + (1 << LAY.lg[g]) <= K) ? (1 << LAY.lg[g]) : (K - LAY.base[g]);
            if (lane == 0) {
                const PlanSlot &ps = slot[it.seq & 1];
                const uint8_t *sbase = p.src + (unsigned long long)it.s * p.src_pitch + (size_t)it.chunk * kStageRowBytes;
                const uint32_t rb = min(kStageRowBytes, (it.nvec - it.chunk * 32) * 16);
                mbar_arrive_expect_tx(bar_stage, rb * nrow);
#pragma unroll
                for (int r = 0; r < nrow; r++)
                    bulk_g2s(stage_addr + r * kStageRowBytes, sbase + ps.src_off[LAY.base[g] + r], rb, bar_stage);
            }
        };
        auto fetch = [&](const It &it) {
            const PlanSlot &ps = slot[it.seq & 1];
            const uint8_t *sbase = p.src + (unsigned long long)it.s * p.src_pitch;
            if constexpr (CFG::kSplit) {
                fetch_group(it, std::integral_constant<int, 0>{});
            } else if constexpr (TMA) {
                if (lane == 0) {
                    const uint32_t rb = min(kStageRowBytes, (it.nvec - it.chunk * 32) * 16);
                    mbar_arrive_expect_tx(bar_stage, rb * K);
#pragma unroll
                    for (int j = 0; j < K; j++)
                        bulk_g2s(stage_addr + j * kStageRowBytes, sbase + ps.src_off[j] + (size_t)it.chunk * kStageRowBytes, rb,
                                 bar_stage);
                }
            } else {
                const uint32_t col = it.chunk * 32 + lane;
                if (col < it.nvec) column_load<CFG, true>(sbase + (size_t)col * 16, p.stride, ps.src_off, lane, dn);
            }
        };

        It nx;
        find(kNone, nx);
        if (nx.valid) fetch(nx);
        if constexpr (CFG::kSplit) {
            constexpr int NG = CFG::kLay.ngroups;
            while (nx.valid) {
                const It cur = nx;
                const uint32_t col = cur.chunk * 32 + lane;
                const bool have_col = col < cur.nvec;
                const uint32_t tail = (have_col && col == cur.nvec - 1) ? (cur.len & 15) : 0;
                uint32_t acc[16];
                static_for<0, NG>([&](auto gc) {
                    constexpr int g = decltype(gc)::value;
                    uint4 d[16];
                    mbar_wait(bar_stage, stage_parity);
                    stage_parity ^= 1;
                    group_read<CFG, g>(stage_addr + lane * 16, lane, d);
                    __syncwarp();  // every lane has its vectors: the stage may be refilled
                    if constexpr (g + 1 < NG) {
                        fetch_group(cur, std::integral_constant<int, g + 1>{});  // next group of the same item
                    } else {
                        pend = cur.seq;
                        find(cur.seq + 1, nx);
                        if (nx.valid) fetch(nx);  // first group of the next item
                    }
                    if (have_col) group_lookup<CFG, g>(acc, d, tab_addr + (cur.seq & 1) * kTabBuf, lane, p.row_bytes, tail);
                });
                if (have_col) {
                    const PlanSlot &ps = slot[cur.seq & 1];
                    uint4 r[4];
                    rows_from_acc(acc, r);
                    uint8_t *dbase = p.dst + (unsigned long long)cur.s * p.dst_pitch;
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        if (i < cur.rows) stg_stream(dbase + ps.dst_off[i] + (size_t)col * 16, r[i]);
                }
                if (pos != cur.seq) leave(cur.seq);
                pend = kNone;
                if (!nx.valid && !ended) {
                    find(kNone, nx);
                    if (nx.valid) fetch(nx);
                }
            }
            return;
        }
        while (nx.valid) {
            const It cur = nx;
            uint4 d[S];
            if constexpr (TMA) {
                mbar_wait(bar_stage, stage_parity);
                stage_parity ^= 1;
                stage_read<CFG>(stage_addr + lane * 16, lane, d);
                __syncwarp();  // every lane has its vectors: the stage may be refilled
            } else {
#pragma unroll
                for (int u = 0; u < S; u++) d[u] = dn[u];
            }
            pend = cur.seq;
            find(cur.seq + 1, nx);
            if (nx.valid) fetch(nx);
            {
                const PlanSlot &ps = slot[cur.seq & 1];
                const uint32_t col = cur.chunk * 32 + lane;
                if (col < cur.nvec) {
                    const uint32_t tail = (col == cur.nvec - 1) ? (cur.len & 15) : 0;
                    uint4 r[4];
                    column_compute<CFG>(d, tab_addr + (cur.seq & 1) * kTabBuf, lane, p.row_bytes, tail, r);
                    uint8_t *dbase = p.dst + (unsigned long long)cur.s * p.dst_pitch;
#pragma unroll
                    for (int i = 0; i < 4; i++)
                        if (i < cur.rows) stg_stream(dbase + ps.dst_off[i] + (size_t)col * 16, r[i]);
                }
            }
            if (pos != cur.seq) leave(cur.seq);  // the search moved on while these lookups were pending
            pend = kNone;
            if (!nx.valid && !ended) {  // the look-ahead was not allowed to go further: continue now
                find(kNone, nx);
                if (nx.valid) fetch(nx);
            }
        }
    }
}

// ------------------------------------------------------------------ decode planning
struct PlanParams {
    const uint8_t *present;  // n*(k+m)
    const uint8_t *want;     // nullable
    int32_t *status;         // nullable, n
    StripePlan *plan;        // n
    uint32_t *counter;       // reset to 0 for the apply kernel's scheduler
    uint32_t n, k, m;
    uint32_t present_is_bad;  // 1: `present` holds "bad" flags (scrub): a shard is present iff flag == 0
    alignas(16) uint8_t P[kMaxM * kMaxK];  // parity rows, P[i*k + j] (16-byte aligned: staged with uint4 loads)
};

constexpr int kPlanWarps = 4;

// One warp per stripe: pick the first k present shards, solve the a x a system that couples the
// a absent data shards to the a parity survivors (Gauss-Jordan, lanes own columns), compose the
// rows that map the survivors straight to every wanted absent shard.
__global__ void __launch_bounds__(kPlanWarps * 32) rs_plan_kernel(const __grid_constant__ PlanParams q)
{
    __shared__ __align__(16) uint8_t s_gf[sizeof(GfTables)];
    uint8_t *const s_exp = s_gf, *const s_log = s_gf + 512;
    __shared__ uint8_t s_A[kPlanWarps][kMaxK][2 * kMaxK];
    __shared__ uint8_t s_surv[kPlanWarps][kMaxK];
    __shared__ uint8_t s_out[kPlanWarps][kMaxM];
    __shared__ uint8_t s_col[kPlanWarps][kMaxK];
    __shared__ uint8_t s_dm[kPlanWarps][kMaxM];
    __shared__ __align__(16) uint8_t s_P[kMaxM * kMaxK];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    stage_gf_tables(s_gf);
    {  // parity rows: kernel parameter (constant bank) -> shared, warp-uniform 16-byte loads
        const uint4 *src = reinterpret_cast<const uint4 *>(q.P);
        for (uint32_t i = warp; i < sizeof(q.P) / 16; i += blockDim.x >> 5) {
            const uint4 v = src[i];
            if (lane < 4) reinterpret_cast<uint32_t *>(s_P)[i * 4 + lane] = lane == 0 ? v.x : (lane == 1 ? v.y : (lane == 2 ? v.z : v.w));
        }
    }
    if (blockIdx.x == 0 && tid == 0) *q.counter = 0;
    __syncthreads();
    auto mul = [&](uint32_t a, uint32_t b) -> uint32_t {
        return (a && b) ? s_exp[s_log[a] + s_log[b]] : 0u;
    };

    const uint32_t s = blockIdx.x * kPlanWarps + warp;
    if (s >= q.n) return;
    const uint32_t k = q.k, m = q.m, tot = k + m;
    StripePlan *pl = q.plan + s;
    const uint8_t *pr = q.present + (size_t)s * tot;
    const uint8_t *wn = q.want ? q.want + (size_t)s * tot : nullptr;

    // presence / wanted masks (tot <= 40: two ballot rounds)
    const bool inv = q.present_is_bad != 0;
    const bool p0 = lane < tot && ((pr[lane] != 0) != inv);
    const bool p1 = lane + 32 < tot && ((pr[lane + 32] != 0) != inv);
    const unsigned long long present =
        (unsigned long long)__ballot_sync(0xffffffffu, p0) |
        ((unsigned long long)__ballot_sync(0xffffffffu, p1) << 32);
    const bool w0 = lane < tot && !p0 && (!wn || wn[lane] != 0);
    const bool w1 = lane + 32 < tot && !p1 && (!wn || wn[lane + 32] != 0);
    unsigned long long outmask = (unsigned long long)__ballot_sync(0xffffffffu, w0) |
                                 ((unsigned long long)__ballot_sync(0xffffffffu, w1) << 32);
    const int npresent = __popcll(present);
    const bool bad = npresent < (int)k;
    if (bad) outmask = 0;
    int nrows = __popcll(outmask);

    if (lane == 0) {
        // survivors: first k present; outputs: wanted absent shards in index order
        unsigned long long pm = present;
        for (uint32_t r = 0; r < k && pm; r++) {
            const int i = __ffsll((long long)pm) - 1;
            s_surv[warp][r] = (uint8_t)i;
            pm &= pm - 1;
        }
        unsigned long long om = outmask;
        for (int r = 0; r < nrows; r++) {
            const int i = __ffsll((long long)om) - 1;
            s_out[warp][r] = (uint8_t)i;
            om &= om - 1;
        }
        pl->key_present = present;
        pl->key_out = outmask;
        pl->nrows = (uint8_t)nrows;
        pl->unrecoverable = bad ? 1 : 0;
        if (q.status) q.status[s] = bad ? -4 : 0;
    }
    __syncwarp();
    if (bad || nrows == 0) return;

    // The survivors are the present data shards (identity rows of the generator) followed by the
    // first `a` present parity shards, a = number of absent data shards.  Only an a x a system
    // couples the unknowns:   y_Pu = A x_Dm + B x_Dp,   A = P[Pu][Dm], B = P[Pu][Dp]
    //   =>  x_Dm = Ainv y_Pu + (Ainv B) x_Dp          (characteristic 2)
    // so a full k x k inversion is never needed (a <= m <= 8).
    uint8_t(*A)[2 * kMaxK] = s_A[warp];  // rows 0..7: [A | I] -> [I | Ainv]; rows 8..15: Ainv*B; rows 16..23: decode rows
    const unsigned long long datamask = (k >= 64 ? ~0ull : ((1ull << k) - 1));
    const unsigned long long mdmask = ~present & datamask;
    const uint32_t a = (uint32_t)__popcll(mdmask);
    const uint32_t nd = k - a;  // data survivors occupy positions [0, nd) of surv[], parity survivors [nd, k)
    if (lane == 0) {
        unsigned long long mm = mdmask;
        for (uint32_t t = 0; t < a; t++) {
            s_dm[warp][t] = (uint8_t)(__ffsll((long long)mm) - 1);
            mm &= mm - 1;
        }
    }
    __syncwarp();
    if (a) {
        for (uint32_t r = 0; r < a; r++) {
            const uint32_t prow = (uint32_t)s_surv[warp][nd + r] - k;
            if (lane < 2 * a) A[r][lane] = lane < a ? s_P[prow * k + s_dm[warp][lane]] : (uint8_t)(lane - a == r);
        }
        __syncwarp();
        for (uint32_t c = 0; c < a; c++) {
            const bool cand = lane < a && lane >= c && A[lane][c] != 0;  // pivot search: lanes are rows
            const uint32_t bal = __ballot_sync(0xffffffffu, cand);
            if (!bal) {  // singular: cannot happen for an MDS generator; report unrecoverable
                if (lane == 0) {
                    pl->nrows = 0;
                    pl->unrecoverable = 1;
                    if (q.status) q.status[s] = -4;
                }
                return;
            }
            const uint32_t piv = __ffs(bal) - 1;
            const uint32_t iv = s_exp[255 - s_log[A[piv][c]]];
            __syncwarp();
            if (lane < 2 * a) {
                const uint8_t x = A[piv][lane], y = A[c][lane];
                A[piv][lane] = y;                  // swap (no-op when piv == c)
                A[c][lane] = (uint8_t)mul(x, iv);  // scaled pivot row
            }
            __syncwarp();
            const uint32_t pv = lane < 2 * a ? A[c][lane] : 0;
            if (lane < a) s_col[warp][lane] = lane == c ? 0 : A[lane][c];
            __syncwarp();
            for (uint32_t r = 0; r < a; r++) {
                const uint32_t f = s_col[warp][r];  // broadcast; lanes own columns
                if (f && lane < 2 * a) A[r][lane] ^= (uint8_t)mul(f, pv);
            }
            __syncwarp();
        }
        // decode row of missing data shard dm[t] over the survivor positions:
        //   data survivors:   (Ainv B)[t][j] = XOR_r Ainv[t][r] * P[Pu_r][surv[j]]
        //   parity survivors: Ainv[t][j - nd]
        for (uint32_t t = 0; t < a; t++) {
            uint32_t v = 0;
            if (lane < nd) {
                const uint32_t col = s_surv[warp][lane];
                for (uint32_t r = 0; r < a; r++)
                    v ^= mul(A[t][a + r], s_P[((uint32_t)s_surv[warp][nd + r] - k) * k + col]);
            } else if (lane < k) {
                v = A[t][a + (lane - nd)];
            }
            if (lane < k) A[16 + t][lane] = (uint8_t)v;
        }
        __syncwarp();
    }
    // rows for the wanted outputs
    for (int r = 0; r < nrows; r++) {
        const uint32_t o = s_out[warp][r];
        if (lane < k) {
            uint32_t v = 0;
            if (o < k) {
                // rank of o among the absent data shards
                const uint32_t t = (uint32_t)__popcll(mdmask & ((1ull << o) - 1));
                v = A[16 + t][lane];
            } else {
                // absent parity row i: P[i][Dp] on the data survivors, plus P[i][Dm] through the rows above
                const uint32_t i = o - k;
                if (lane < nd) v = s_P[i * k + s_surv[warp][lane]];
                for (uint32_t t = 0; t < a; t++) v ^= mul(s_P[i * k + s_dm[warp][t]], A[16 + t][lane]);
            }
            pl->coef[r][lane] = (uint8_t)v;
        }
    }
    if (lane < k) pl->surv[lane] = s_surv[warp][lane];
    if (lane < (uint32_t)nrows) pl->out_idx[lane] = s_out[warp][lane];
}

// ------------------------------------------------------------------ synthetic data
// splitmix64 counter stream of SURVEY.md 8(d) (the CPU checker generates the same stream).
__global__ void fill_random_kernel(unsigned long long *dst, size_t nwords, unsigned long long seed,
                                   unsigned long long first_idx)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nwords;
         i += (size_t)gridDim.x * blockDim.x) {
        unsigned long long z = seed + (first_idx + i + 1) * 0x9E3779B97F4A7C15ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        dst[i] = z ^ (z >> 31);
    }
}

// ------------------------------------------------------------------ per-shard integrity (row f2)
// blake2sum (BLAKE2b-512 truncated to 32 bytes, src/util/data.rs:130-138) of every shard of a
// batch, one thread per shard.  BLAKE2b is sequential per message, so the parallelism is across
// the n * shards_per_stripe independent shards; compute-bound (~28 integer instructions per
// byte), not HBM-bound.  `expect` != NULL turns it into the scrub check: bad[i] = sum differs.
struct SumParams {
    const uint8_t *base;        // shard i at base + i * stride
    const uint32_t *shard_len;  // per stripe, nullable (=> stride)
    const uint8_t *expect;      // nullable: 32 bytes per shard to compare with
    uint8_t *sums;              // nullable: 32 bytes per shard out
    uint8_t *bad;               // nullable: 1 byte per shard out (only with expect)
    uint32_t stride;
    uint32_t per_stripe;        // shards per stripe (k, m or k+m)
    uint32_t n_shards;
    uint32_t out_per_stripe;    // sums/expect/bad are indexed (i / per_stripe) * out_per_stripe
    uint32_t out_off;           //                              + out_off + i % per_stripe
    // optional second segment (shards n_first.. of the launch): lets one launch hash the data
    // array AND the parity array of an encode batch (half the latency of two launches)
    const uint8_t *base2;
    uint32_t n_first;           // shards in the first segment (== n_shards when there is no second)
    uint32_t per_stripe2;
    uint32_t out_off2;
};

// where shard i of a launch lives, which stripe's length applies, and its slot in sums/expect/bad
__device__ __forceinline__ void locate_shard(const SumParams &q, uint32_t i, const uint8_t *&p, uint32_t &len,
                                             size_t &oi)
{
    uint32_t stripe;
    if (i < q.n_first) {
        stripe = i / q.per_stripe;
        p = q.base + (size_t)i * q.stride;
        oi = (size_t)stripe * q.out_per_stripe + q.out_off + (i - stripe * q.per_stripe);
    } else {
        const uint32_t j = i - q.n_first;
        stripe = j / q.per_stripe2;
        p = q.base2 + (size_t)j * q.stride;
        oi = (size_t)stripe * q.out_per_stripe + q.out_off2 + (j - stripe * q.per_stripe2);
    }
    len = q.shard_len ? __ldg(q.shard_len + stripe) : q.stride;
}

__global__ void __launch_bounds__(128) blake2sum_shards_kernel(const __grid_constant__ SumParams q)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q.n_shards) return;
    const uint8_t *p;
    uint32_t len;
    size_t oi;
    locate_shard(q, i, p, len, oi);
    Blake2bState S;
    blake2b_init512(S);
    uint64_t m[16];
    uint32_t off = 0;
    while (len - off > 128) {
#pragma unroll
        for (int w = 0; w < 8; w++) {
            const uint4 v = *reinterpret_cast<const uint4 *>(p + off + 16 * w);
            m[2 * w] = (uint64_t)v.x | ((uint64_t)v.y << 32);
            m[2 * w + 1] = (uint64_t)v.z | ((uint64_t)v.w << 32);
        }
        S.t += 128;
        blake2b_compress(S, m, false);
        off += 128;
    }
    const uint32_t rem = len - off;  // 0..128 bytes in the last block (0 only for an empty shard)
#pragma unroll
    for (int w = 0; w < 8; w++) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if ((uint32_t)(16 * w) < rem) {
            v = *reinterpret_cast<const uint4 *>(p + off + 16 * w);  // within roundup16(len): readable
            if (rem - 16 * w < 16) v = mask_tail(v, rem - 16 * w);
        }
        m[2 * w] = (uint64_t)v.x | ((uint64_t)v.y << 32);
        m[2 * w + 1] = (uint64_t)v.z | ((uint64_t)v.w << 32);
    }
    S.t += rem;
    blake2b_compress(S, m, true);
    if (q.sums) {
        uint4 *o = reinterpret_cast<uint4 *>(q.sums + oi * 32);
        o[0] = make_uint4((uint32_t)S.h[0], (uint32_t)(S.h[0] >> 32), (uint32_t)S.h[1], (uint32_t)(S.h[1] >> 32));
        o[1] = make_uint4((uint32_t)S.h[2], (uint32_t)(S.h[2] >> 32), (uint32_t)S.h[3], (uint32_t)(S.h[3] >> 32));
    }
    if (q.expect && q.bad) {
        const unsigned long long *e = reinterpret_cast<const unsigned long long *>(q.expect + oi * 32);
        q.bad[oi] = (e[0] != S.h[0]) | (e[1] != S.h[1]) | (e[2] != S.h[2]) | (e[3] != S.h[3]);
    }
}


// ---- the same hash with FOUR lanes per shard --------------------------------------------------
// With a few ten-thousand shards per batch the one-thread-per-shard kernel leaves most of the GPU
// idle (28 672 shards = 1.5 warps per scheduler).  BLAKE2b's four column G functions and four
// diagonal G functions are independent, so a quad of lanes shares one message: lane c owns
// column c of the 4x4 state (a,b,c,d = v[c], v[4+c], v[8+c], v[12+c]); the diagonal step is the
// column step after rotating rows 1,2,3 by 1,2,3 lanes inside the quad (quad-masked shuffles).
// The 128-byte message block sits in shared memory (32 B loaded per lane, coalesced per quad); the
// per-round word selection sigma[r] is four byte offsets packed in one register per round.
// ~1.5x the instructions of the scalar kernel for 4x the parallelism.
__constant__ uint8_t c_b2_sigma[12][16] = {
    {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3},
    {11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4}, {7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8},
    {9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13}, {2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9},
    {12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11}, {13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10},
    {6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5}, {10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0},
    {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15}, {14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3}};

__device__ __forceinline__ uint64_t shfl64(uint32_t mask, uint64_t v, uint32_t src)
{
    const uint32_t lo = __shfl_sync(mask, (uint32_t)v, src), hi = __shfl_sync(mask, (uint32_t)(v >> 32), src);
    return (uint64_t)lo | ((uint64_t)hi << 32);
}
__device__ __forceinline__ uint64_t lds_u64(uint32_t addr)
{
    uint64_t r;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(r) : "r"(addr));
    return r;
}

constexpr int kQuadThreads = 128;  // 32 shards per block

__global__ void __launch_bounds__(kQuadThreads) blake2sum_shards_quad_kernel(const __grid_constant__ SumParams q)
{
    // 144-byte pitch: consecutive quads start 4 banks apart (a 128-byte pitch puts the same word
    // of all 8 quads of a warp in the same bank: 8-way conflicts on every message load)
    __shared__ __align__(16) uint8_t s_msg[kQuadThreads / 4][144];
    const uint32_t tid = threadIdx.x, lane = tid & 31, c = tid & 3;
    const uint32_t i = blockIdx.x * (kQuadThreads / 4) + (tid >> 2);  // shard index
    if (i >= q.n_shards) return;                                      // whole quads leave together
    const uint32_t qmask = 0xFu << (lane & ~3u), qbase = lane & ~3u;
    const uint8_t *p;
    uint32_t len;
    size_t oi;
    locate_shard(q, i, p, len, oi);
    const uint32_t msg = (uint32_t)__cvta_generic_to_shared(&s_msg[tid >> 2][0]);

    // per-round message offsets for this lane: {col x, col y, diag x, diag y} * 8 bytes
    uint32_t off[12];
#pragma unroll
    for (int r = 0; r < 12; r++)
        off[r] = ((uint32_t)c_b2_sigma[r][2 * c] << 3) | ((uint32_t)c_b2_sigma[r][2 * c + 1] << 11) |
                 ((uint32_t)c_b2_sigma[r][8 + 2 * c] << 19) | ((uint32_t)c_b2_sigma[r][8 + 2 * c + 1] << 27);
    const uint64_t IV[8] = {0x6a09e667f3bcc908ull, 0xbb67ae8584caa73bull, 0x3c6ef372fe94f82bull, 0xa54ff53a5f1d36f1ull,
                            0x510e527fade682d1ull, 0x9b05688c2b3e6c1full, 0x1f83d9abfb41bd6bull, 0x5be0cd19137e2179ull};
    const uint64_t ivlo = c == 0 ? IV[0] : (c == 1 ? IV[1] : (c == 2 ? IV[2] : IV[3]));
    const uint64_t ivhi = c == 0 ? IV[4] : (c == 1 ? IV[5] : (c == 2 ? IV[6] : IV[7]));
    uint64_t h0 = ivlo ^ (c == 0 ? 0x01010040ull : 0ull), h1 = ivhi;  // h[c], h[4+c]

    // this lane's 32 bytes of the block starting at byte `o` (zero beyond len)
    auto load32 = [&](uint32_t o, uint4 &x, uint4 &y) {
        x = make_uint4(0, 0, 0, 0);
        y = make_uint4(0, 0, 0, 0);
        const uint32_t a0 = o + 32 * c;
        if (a0 < len) {
            x = *reinterpret_cast<const uint4 *>(p + a0);
            if (len - a0 < 16) x = mask_tail(x, len - a0);
        }
        if (a0 + 16 < len) {
            y = *reinterpret_cast<const uint4 *>(p + a0 + 16);
            if (len - a0 - 16 < 16) y = mask_tail(y, len - a0 - 16);
        }
    };
    uint4 nx, ny;
    load32(0, nx, ny);
    uint32_t o = 0;
    for (;;) {
        const bool last = len - o <= 128;  // also true for an empty shard
        __syncwarp(qmask);                  // previous block's words are no longer needed
        *reinterpret_cast<uint4 *>(&s_msg[tid >> 2][32 * c]) = nx;
        *reinterpret_cast<uint4 *>(&s_msg[tid >> 2][32 * c + 16]) = ny;
        __syncwarp(qmask);
        if (!last) load32(o + 128, nx, ny);  // prefetch the next block
        const uint64_t t = last ? (uint64_t)len : (uint64_t)o + 128;
        uint64_t va = h0, vb = h1, vc = ivlo, vd = ivhi;
        if (c == 0) vd ^= t;
        if (c == 2 && last) vd = ~vd;
#pragma unroll
        for (int r = 0; r < 12; r++) {
            const uint32_t f = off[r];
            uint64_t mx = lds_u64(msg + (f & 0xff)), my = lds_u64(msg + ((f >> 8) & 0xff));
            GEC_B2_G(va, vb, vc, vd, mx, my);
            vb = shfl64(qmask, vb, qbase + ((c + 1) & 3));
            vc = shfl64(qmask, vc, qbase + ((c + 2) & 3));
            vd = shfl64(qmask, vd, qbase + ((c + 3) & 3));
            mx = lds_u64(msg + ((f >> 16) & 0xff));
            my = lds_u64(msg + (f >> 24));
            GEC_B2_G(va, vb, vc, vd, mx, my);
            vb = shfl64(qmask, vb, qbase + ((c + 3) & 3));
            vc = shfl64(qmask, vc, qbase + ((c + 2) & 3));
            vd = shfl64(qmask, vd, qbase + ((c + 1) & 3));
        }
        h0 ^= va ^ vc;
        h1 ^= vb ^ vd;
        if (last) break;
        o += 128;
    }
    if (q.sums) *reinterpret_cast<unsigned long long *>(q.sums + oi * 32 + 8 * c) = h0;
    if (q.expect && q.bad) {
        const unsigned long long e = *reinterpret_cast<const unsigned long long *>(q.expect + oi * 32 + 8 * c);
        const uint32_t diff = __ballot_sync(qmask, e != h0) & qmask;
        if (c == 0) q.bad[oi] = diff ? 1 : 0;
    }
}

// ------------------------------------------------------------------ block -> shard framing on the device
// rpc_put_block hands over a contiguous block (bytes::Bytes); the streaming kernels want k shards,
// `stride` apart and 16-byte aligned, the last one zero padded (DataBlock::from_buffer framing,
// src/block/block.rs:85-96; short last block src/api/s3/put.rs:583-617).  The block crosses PCIe as
// ONE contiguous copy (a pitched 2-D copy with an odd row width -- shard_len is rarely a multiple of
// 16 -- runs far below the link rate) and this kernel cuts it up at HBM speed: every thread
// produces one 16-byte vector of one shard from an arbitrarily aligned source position (five
// aligned 32-bit loads + funnel shifts), zero beyond the shard / the block.
struct SplitParams {
    const uint8_t *blocks;       // block s at blocks + s*block_pitch (16-byte aligned)
    const uint32_t *block_len;   // per block
    uint8_t *shards;             // shard j of block s at shards + (s*k + j)*stride
    unsigned long long block_pitch;
    uint32_t stride, k, n;
    uint32_t parts;              // CTAs per block: a dispatcher batch of a dozen blocks still has to fill 148 SMs
};
__global__ void __launch_bounds__(256) split_blocks_kernel(const __grid_constant__ SplitParams q)
{
    for (uint32_t w = blockIdx.x; w < q.n * q.parts; w += gridDim.x) {
        const uint32_t s = w / q.parts, part = w - s * q.parts;
        const uint32_t len = __ldg(q.block_len + s);
        const uint32_t L = (len + q.k - 1) / q.k, nvec = (L + 15) >> 4;
        const uint8_t *src = q.blocks + (unsigned long long)s * q.block_pitch;
        uint8_t *dst = q.shards + (unsigned long long)s * q.k * q.stride;
        const uint32_t total = q.k * nvec, per = ((total + q.parts - 1) / q.parts + 255u) & ~255u;
        const uint32_t lo = part * per, hi = min(total, lo + per);
#pragma unroll 4
        for (uint32_t idx = lo + threadIdx.x; idx < hi; idx += 256) {
            const uint32_t j = idx / nvec, v = idx - j * nvec;
            const uint32_t pos = j * L + v * 16;  // first source byte of this vector
            // valid bytes: inside the shard and inside the block
            uint32_t nvalid = min(16u, L - v * 16);
            nvalid = pos >= len ? 0 : min(nvalid, len - pos);
            uint4 o = make_uint4(0, 0, 0, 0);
            if (nvalid) {
                const uint32_t a = pos & ~3u, sh = (pos & 3u) * 8;
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(src + a);
                // words a .. a+16 hold bytes pos .. pos+15 (+ up to 3 on either side); the staging buffer is
                // padded so that reading one word past the block is always inside the allocation
                const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = sh ? wp[4] : 0;
                o = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                               __funnelshift_r(w3, w4, sh));
                if (nvalid < 16) o = mask_tail(o, nvalid);
            }
            *reinterpret_cast<uint4 *>(dst + (size_t)j * q.stride + (size_t)v * 16) = o;
        }
    }
}

// ---- fast per-shard integrity tag: 8 x Adler-32 ("adler8") -----------------------------------
// BLAKE2b is compute-bound on CUDA cores (~20 integer instructions per byte: at most ~1.3 TB/s,
// round 1 measured 0.45-0.6 TB/s), which capped the scrub sweep at 7 % of HBM bandwidth.  Scrub
// only has to catch bit rot (the block's content address stays Garage's blake2sum), so the shard
// files may carry a cheap tag instead: the shard is cut in 8 segments of
// seg = roundup16(ceil(len / 8)) bytes and the tag is the 8 little-endian zlib Adler-32 values of
// the segments (an empty segment has Adler-32 = 1) -- 32 bytes, the size of Garage's `Hash`.
// Adler-32 is a = 1 + sum d_i, b = n + sum (n - i) d_i (mod 65521): plain byte sums, 4 DP4A per 16
// bytes for each, so the kernel streams at HBM speed; one warp per shard, four 16-byte loads per
// lane in flight.  Pinned by python's zlib.adler32 (tests/test_blake2.py).
constexpr uint32_t kAdlerMod = 65521;
__host__ __device__ inline uint32_t adler8_seg_bytes(uint32_t len)
{
    return (((len + 7) / 8) + 15) / 16 * 16;
}

__global__ void __launch_bounds__(256) adler8_shards_kernel(const __grid_constant__ SumParams q)
{
    // (a block-per-segment variant, 256 threads on one contiguous ~20 KB region + a shared-memory reduction, measured
    // SLOWER: 2.2-2.9 TB/s against 4.0 TB/s, profiles/r02_summary.md)
    // work unit = one SEGMENT of one shard per warp (8 units per shard): 8x the units of a warp-per-shard
    // split, so the persistent grid stays balanced down to a few hundred shards (ncu of the warp-per-shard
    // version: 50 % of DRAM peak with a 2-wave tail at 18 432 shards).  `bad` must be zero on entry when
    // `expect` is given (the host memsets it): segments OR their verdict into the shard's flag byte.
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t wpb = blockDim.x >> 5;
    const uint32_t units = q.n_shards * 8u;  // host guarantees n_shards < 2^29
    for (uint32_t u = blockIdx.x * wpb + (threadIdx.x >> 5); u < units; u += gridDim.x * wpb) {
        const uint32_t i = u >> 3, sgi = u & 7;
        const uint8_t *p;
        uint32_t len;
        size_t oi;
        locate_shard(q, i, p, len, oi);
        const uint32_t seg = adler8_seg_bytes(len);
        const uint32_t start = sgi * seg;
        uint32_t tag = 1;  // Adler-32 of an empty segment
        if (start < len) {
            const uint32_t end = min(len, start + seg), n = end - start;
            unsigned long long A = 0, B = 0, T = 0;
            // 8 vectors per lane in flight: rel = byte offset of the vector inside the segment
            for (uint32_t r0 = lane * 16; r0 < n; r0 += 8 * 512) {
                uint4 v[8];
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const uint32_t rel = r0 + k * 512;
                    v[k] = make_uint4(0, 0, 0, 0);
                    if (rel < n) {
                        v[k] = ldg_stream(p + start + rel);  // within roundup16(len): readable
                        if (n - rel < 16) v[k] = mask_tail(v[k], n - rel);
                    }
                }
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const uint32_t rel = r0 + k * 512;
                    uint32_t sm = __dp4a(v[k].x, 0x01010101u, 0u);
                    sm = __dp4a(v[k].y, 0x01010101u, sm);
                    sm = __dp4a(v[k].z, 0x01010101u, sm);
                    sm = __dp4a(v[k].w, 0x01010101u, sm);
                    uint32_t t = __dp4a(v[k].x, 0x03020100u, 0u);  // sum_j j * byte_j
                    t = __dp4a(v[k].y, 0x07060504u, t);
                    t = __dp4a(v[k].z, 0x0b0a0908u, t);
                    t = __dp4a(v[k].w, 0x0f0e0d0cu, t);
                    A += sm;
                    if (rel < n) B += (unsigned long long)(n - rel) * sm;
                    T += t;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                A += __shfl_xor_sync(0xffffffffu, A, o);
                B += __shfl_xor_sync(0xffffffffu, B, o);
                T += __shfl_xor_sync(0xffffffffu, T, o);
            }
            const uint32_t a = (uint32_t)((1 + A) % kAdlerMod);
            const uint32_t b = (uint32_t)((n + B - T) % kAdlerMod);  // B >= T: (n - rel) >= j + 1 for every byte
            tag = (b << 16) | a;
        }
        if (lane == 0) {
            if (q.sums) reinterpret_cast<uint32_t *>(q.sums + oi * 32)[sgi] = tag;
            if (q.expect && q.bad && reinterpret_cast<const uint32_t *>(q.expect + oi * 32)[sgi] != tag) {
                // set byte `oi` of bad[] to 1 through the aligned 32-bit word that contains it
                const unsigned long long addr = reinterpret_cast<unsigned long long>(q.bad + oi);
                atomicOr(reinterpret_cast<unsigned int *>(addr & ~3ull), 1u << (8 * (unsigned)(addr & 3ull)));
            }
        }
    }
}

// ------------------------------------------------------------------ error-locating decode (garage_ec_correct)
// Both built-in matrices (and any matrix that passes h_grs_multipliers) define a generalized RS code: the
// parity-check rows H[l][r] = v_r X_r^l, l < m, annihilate every codeword.  Locator X_r = r xor kLocShift
// (shifting every evaluation point by one constant keeps the code and the v_r; the shift keeps X_r != 0).
// Pipeline (DESIGN.md section 4, "Error-locating decode"):
//   1. check:  rs_apply_kernel<kModeVerify> -- the streaming verify, unchanged: mismatch[s] != 0 iff some
//      column of stripe s is not a codeword;
//   2. list:   rs_correct_list_kernel -- status / fixed of every stripe; stripes with an absent shard or a
//      mismatch go to a compacted list (device side: no host round trip, graph-capturable);
//   3. scan:   rs_correct_scan_kernel<M> -- every byte column of every listed stripe: GRS syndromes,
//      errors-and-erasures decoding; writes nothing but the per-stripe union of error positions and an
//      "uncorrectable" flag;
//   4. apply:  rs_correct_apply_kernel<M> -- listed stripes whose every column decoded: decode again and
//      write the erased and the wrong shards (zero padding to roundup16); the rest only get status -7.
constexpr uint32_t kLocShift = 0x80;
constexpr int kCorrectThreads = 256;  // one byte column per thread

struct CorrectParams {
    uint8_t *shards;              // stripe s, shard r at (s*(k+m) + r) * stride
    const uint8_t *present;       // nullable (= all present)
    const uint32_t *shard_len;    // nullable (= stride)
    const uint32_t *mismatch;     // check pass result
    int32_t *status;              // nullable
    uint8_t *fixed;               // nullable, n*(k+m)
    uint32_t *list;               // compacted stripe indices, list[0 .. *count)
    uint32_t *count;
    unsigned long long *err_mask;  // per list entry: union of the error positions of its columns
    uint32_t *bad;                 // per list entry: != 0 if some column had more than t errors
    uint32_t stride, n, k, m;
    uint32_t items_per_stripe;    // ceil(stride / kCorrectThreads)
    uint8_t logx[kMaxK + kMaxM];  // log X_r
    uint8_t logv[kMaxK + kMaxM];  // log v_r
};

// one thread per stripe: presence, status, fixed row; stripes that need the decoder are listed
__global__ void rs_correct_list_kernel(const __grid_constant__ CorrectParams p)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    const uint32_t tot = p.k + p.m;
    uint32_t absent = 0;
    if (p.present)
        for (uint32_t r = 0; r < tot; r++) absent += p.present[(size_t)s * tot + r] ? 0u : 1u;
    if (p.fixed)
        for (uint32_t r = 0; r < tot; r++) p.fixed[(size_t)s * tot + r] = 0;
    if (absent > p.m) {
        if (p.status) p.status[s] = -4;  // GARAGE_EC_E_UNRECOVERABLE
        return;
    }
    if (p.status) p.status[s] = 0;
    if (absent || p.mismatch[s]) {
        const uint32_t q = atomicAdd(p.count, 1u);
        p.list[q] = s;
        p.err_mask[q] = 0;
        p.bad[q] = 0;
    }
}

struct GfSmem {
    uint8_t exp[512];
    uint8_t log[256];
};
__device__ __forceinline__ uint32_t gf_mul_s(const GfSmem &g, uint32_t a, uint32_t b)
{
    return (a && b) ? g.exp[g.log[a] + g.log[b]] : 0u;
}
// a * alpha^lb, lb in [0, 255]
__device__ __forceinline__ uint32_t gf_mul_l(const GfSmem &g, uint32_t a, uint32_t lb)
{
    return a ? g.exp[g.log[a] + lb] : 0u;
}

// Errors-and-erasures decoding of one byte column from its m GRS syndromes S (S_l = sum_r y_r v_r X_r^l,
// erased y_r taken as 0) and the erasure locator gam = prod_{r in E} (1 + X_r x) of degree e:
// Forney syndromes -> Berlekamp-Massey -> errata locator psi = lambda * gam and evaluator
// omg = S * psi mod x^M.  Returns L = deg lambda, or -1 if 2L > m - e (more errors than t).
// Every index is a compile-time constant, so the polynomials stay in registers.
template <int M>
__device__ __forceinline__ int correct_decode(const GfSmem &g, const uint32_t (&S)[M], const uint32_t (&gam)[M + 1], int e,
                                              uint32_t (&psi)[M + 1], uint32_t (&omg)[M])
{
    uint32_t F[M];
#pragma unroll
    for (int i = 0; i < M; i++) {
        uint32_t v = 0;
#pragma unroll
        for (int j = 0; j <= i; j++) v ^= gf_mul_s(g, S[j], gam[i - j]);
        F[i] = v;
    }
    // Forney syndromes F[e .. M) moved down to F[0 .. M-e)
#pragma unroll
    for (int q = 0; q < M; q++) {
        if (q < e) {
#pragma unroll
            for (int i = 0; i + 1 < M; i++) F[i] = F[i + 1];
            F[M - 1] = 0;
        }
    }
    const int N = M - e;
    uint32_t C[M + 1], B[M + 1];  // B = x^shift * (previous connection polynomial)
#pragma unroll
    for (int i = 0; i <= M; i++) {
        C[i] = i == 0 ? 1u : 0u;
        B[i] = i == 1 ? 1u : 0u;
    }
    int L = 0;
    uint32_t b = 1;
#pragma unroll
    for (int i = 0; i < M; i++) {
        if (i < N) {
            uint32_t d = F[i];
#pragma unroll
            for (int j = 1; j <= i; j++) d ^= gf_mul_s(g, C[j], F[i - j]);
            if (d) {
                const uint32_t lc = (uint32_t)g.log[d] + 255u - g.log[b];  // log(d / b), < 510
                uint32_t T[M + 1];
#pragma unroll
                for (int j = 0; j <= M; j++) T[j] = C[j] ^ (B[j] ? g.exp[g.log[B[j]] + (lc % 255u)] : 0u);
                if (2 * L <= i) {
#pragma unroll
                    for (int j = 0; j <= M; j++) B[j] = C[j];
                    L = i + 1 - L;
                    b = d;
                }
#pragma unroll
                for (int j = 0; j <= M; j++) C[j] = T[j];
            }
#pragma unroll
            for (int j = M; j > 0; j--) B[j] = B[j - 1];
            B[0] = 0;
        }
    }
    if (2 * L > N) return -1;
#pragma unroll
    for (int i = 0; i <= M; i++) {
        uint32_t v = 0;
#pragma unroll
        for (int j = 0; j <= i; j++) v ^= gf_mul_s(g, C[j], gam[i - j]);
        psi[i] = v;
    }
#pragma unroll
    for (int i = 0; i < M; i++) {
        uint32_t v = 0;
#pragma unroll
        for (int j = 0; j <= i; j++) v ^= gf_mul_s(g, S[j], psi[i - j]);
        omg[i] = v;
    }
    return L;
}

// errata value at position r (log X_r = lx, log v_r = lv): psi(1/X_r) == 0 marks an errata position;
// value y_r xor c_r = X_r omg(1/X_r) / (v_r psi'(1/X_r)).  Returns false where psi has no simple root.
template <int M>
__device__ __forceinline__ bool correct_value(const GfSmem &g, const uint32_t (&psi)[M + 1], const uint32_t (&omg)[M], uint32_t lx,
                                              uint32_t lv, bool &errata, uint32_t &val)
{
    const uint32_t li = lx ? 255u - lx : 0u;  // log (1/X_r)
    uint32_t ps = psi[M];
#pragma unroll
    for (int i = M - 1; i >= 0; i--) ps = gf_mul_l(g, ps, li) ^ psi[i];
    errata = ps == 0;
    val = 0;
    if (!errata) return true;
    uint32_t om = omg[M - 1];
#pragma unroll
    for (int i = M - 2; i >= 0; i--) om = gf_mul_l(g, om, li) ^ omg[i];
    // psi'(x) = sum over odd i of psi[i] x^(i-1) (characteristic 2)
    uint32_t dp = 0;
#pragma unroll
    for (int i = M - (M % 2 == 0 ? 1 : 0); i >= 1; i -= 2) dp = gf_mul_l(g, gf_mul_l(g, dp, li), li) ^ psi[i];
    if (!dp) return false;
    if (om) val = g.exp[(g.log[om] + lx + 2u * 255u - g.log[dp] - lv) % 255u];
    return true;
}

// per work item: presence mask, erasure count and erasure locator of the stripe, staged by warp 0
struct CorrectStripe {
    unsigned long long pm;
    uint32_t s, len, e, pad;
    uint32_t gam[kMaxM + 1];
};

template <int M>
__device__ __forceinline__ void correct_stage_stripe(const CorrectParams &p, const GfSmem &g, uint32_t s, CorrectStripe &cs)
{
    const uint32_t tid = threadIdx.x, tot = p.k + M;
    if (tid >= 32) return;
    const bool p0 = tid < tot && (!p.present || p.present[(size_t)s * tot + tid]);
    const bool p1 = tid + 32 < tot && (!p.present || p.present[(size_t)s * tot + tid + 32]);
    const unsigned long long pm =
        (unsigned long long)__ballot_sync(0xffffffffu, p0) | ((unsigned long long)__ballot_sync(0xffffffffu, p1) << 32);
    if (tid != 0) return;
    cs.pm = pm;
    cs.s = s;
    cs.len = p.shard_len ? p.shard_len[s] : p.stride;
    cs.e = tot - (uint32_t)__popcll(pm);
    uint32_t gam[kMaxM + 1] = {1};
    for (uint32_t r = 0; r < tot; r++) {
        if ((pm >> r) & 1) continue;
        for (int j = kMaxM; j > 0; j--) gam[j] ^= gf_mul_l(g, gam[j - 1], p.logx[r]);  // gam *= (1 + X_r x)
    }
    for (int j = 0; j <= kMaxM; j++) cs.gam[j] = gam[j];
}

// syndromes of byte column x of the stripe (x < len); absent shards count as zero
template <int M>
__device__ __forceinline__ void correct_syndromes(const CorrectParams &p, const GfSmem &g, const uint8_t *s_logh,
                                                  const CorrectStripe &cs, uint32_t x, uint32_t (&S)[M])
{
    const uint32_t tot = p.k + M;
    const uint8_t *col = p.shards + (size_t)cs.s * tot * p.stride + x;
#pragma unroll
    for (int l = 0; l < M; l++) S[l] = 0;
#pragma unroll 2
    for (uint32_t r = 0; r < tot; r++) {
        if (!((cs.pm >> r) & 1)) continue;
        const uint32_t y = __ldg(col + (size_t)r * p.stride);
        if (!y) continue;
        const uint32_t ly = g.log[y];
#pragma unroll
        for (int l = 0; l < M; l++) S[l] ^= g.exp[ly + s_logh[l * (kMaxK + kMaxM) + r]];
    }
}

template <int M>
__device__ __forceinline__ void correct_setup(const CorrectParams &p, GfSmem &g, uint8_t *s_logh)
{
    stage_gf_tables(reinterpret_cast<uint8_t *>(&g));
    const uint32_t tot = p.k + M;
    for (uint32_t i = threadIdx.x; i < M * tot; i += blockDim.x) {
        const uint32_t l = i / tot, r = i - l * tot;
        s_logh[l * (kMaxK + kMaxM) + r] = (uint8_t)((p.logv[r] + l * (uint32_t)p.logx[r]) % 255u);  // log(v_r X_r^l)
    }
}

template <int M>
__global__ void __launch_bounds__(kCorrectThreads) rs_correct_scan_kernel(const __grid_constant__ CorrectParams p)
{
    __shared__ __align__(16) GfSmem g;
    __shared__ uint8_t s_logh[M * (kMaxK + kMaxM)];
    __shared__ CorrectStripe cs;
    correct_setup<M>(p, g, s_logh);
    const uint32_t tid = threadIdx.x, lane = tid & 31, tot = p.k + M;
    const unsigned long long total = (unsigned long long)*p.count * p.items_per_stripe;
    for (unsigned long long item = blockIdx.x; item < total; item += gridDim.x) {
        const uint32_t q = (uint32_t)(item / p.items_per_stripe), c = (uint32_t)(item - (unsigned long long)q * p.items_per_stripe);
        __syncthreads();  // tables staged / previous item done with `cs`
        correct_stage_stripe<M>(p, g, p.list[q], cs);
        __syncthreads();
        const uint32_t x = c * kCorrectThreads + tid;
        unsigned long long errs = 0;
        bool fail = false;
        if (x < cs.len) {
            uint32_t S[M];
            correct_syndromes<M>(p, g, s_logh, cs, x, S);
            uint32_t any = 0;
#pragma unroll
            for (int l = 0; l < M; l++) any |= S[l];
            if (any) {  // clean columns (all-zero syndromes) of a listed stripe need nothing more
                uint32_t gam[M + 1], psi[M + 1], omg[M];
#pragma unroll
                for (int j = 0; j <= M; j++) gam[j] = cs.gam[j];
                const int L = correct_decode<M>(g, S, gam, (int)cs.e, psi, omg);
                if (L < 0) {
                    fail = true;
                } else {
                    // L distinct roots among the present positions, simple errata roots, and the errata pattern
                    // must reproduce the syndromes: then y minus the pattern is the codeword within radius t
                    uint32_t chk[M];
#pragma unroll
                    for (int l = 0; l < M; l++) chk[l] = 0;
                    int roots = 0;
                    for (uint32_t r = 0; r < tot && !fail; r++) {
                        bool errata;
                        uint32_t val;
                        if (!correct_value<M>(g, psi, omg, p.logx[r], p.logv[r], errata, val)) fail = true;
                        if (!errata) continue;
                        const bool erased = !((cs.pm >> r) & 1);
                        if (!erased) {
                            roots++;
                            if (val) errs |= 1ull << r;
                        }
                        if (val) {
                            const uint32_t lv = g.log[val];
#pragma unroll
                            for (int l = 0; l < M; l++) chk[l] ^= g.exp[lv + s_logh[l * (kMaxK + kMaxM) + r]];
                        }
                    }
                    if (roots != L) fail = true;
#pragma unroll
                    for (int l = 0; l < M; l++) fail |= chk[l] != S[l];
                }
            }
        }
        const uint32_t lo = __reduce_or_sync(0xffffffffu, (uint32_t)errs);
        const uint32_t hi = __reduce_or_sync(0xffffffffu, (uint32_t)(errs >> 32));
        const bool wfail = __any_sync(0xffffffffu, fail);
        if (lane == 0) {
            if (lo | hi) atomicOr(p.err_mask + q, ((unsigned long long)hi << 32) | lo);
            if (wfail) atomicOr(p.bad + q, 1u);
        }
    }
}

template <int M>
__global__ void __launch_bounds__(kCorrectThreads) rs_correct_apply_kernel(const __grid_constant__ CorrectParams p)
{
    __shared__ __align__(16) GfSmem g;
    __shared__ uint8_t s_logh[M * (kMaxK + kMaxM)];
    __shared__ CorrectStripe cs;
    correct_setup<M>(p, g, s_logh);
    const uint32_t tid = threadIdx.x, tot = p.k + M;
    const unsigned long long total = (unsigned long long)*p.count * p.items_per_stripe;
    for (unsigned long long item = blockIdx.x; item < total; item += gridDim.x) {
        const uint32_t q = (uint32_t)(item / p.items_per_stripe), c = (uint32_t)(item - (unsigned long long)q * p.items_per_stripe);
        __syncthreads();
        correct_stage_stripe<M>(p, g, p.list[q], cs);
        __syncthreads();
        const uint32_t s = cs.s;
        if (p.bad[q]) {  // uniform over the block: nothing of this stripe is written
            if (c == 0 && tid == 0 && p.status) p.status[s] = -7;  // GARAGE_EC_E_UNCORRECTABLE
            continue;
        }
        const unsigned long long errs = p.err_mask[q], absent = ~cs.pm & ((tot >= 64 ? 0ull : 1ull << tot) - 1ull);
        if (c == 0 && p.fixed && tid < tot && ((errs >> tid) & 1)) p.fixed[(size_t)s * tot + tid] = 1;
        const unsigned long long wr = errs | absent;  // shards to write
        const uint32_t x = c * kCorrectThreads + tid;
        if (!wr || x >= ((cs.len + 15u) & ~15u)) continue;
        uint8_t *col = p.shards + (size_t)s * tot * p.stride + x;
        if (x >= cs.len) {  // output padding
            for (unsigned long long w = wr; w; w &= w - 1) col[(size_t)(__ffsll((long long)w) - 1) * p.stride] = 0;
            continue;
        }
        uint32_t S[M];
        correct_syndromes<M>(p, g, s_logh, cs, x, S);
        uint32_t any = 0;
#pragma unroll
        for (int l = 0; l < M; l++) any |= S[l];
        uint32_t gam[M + 1], psi[M + 1], omg[M];
        if (any) {
#pragma unroll
            for (int j = 0; j <= M; j++) gam[j] = cs.gam[j];
            correct_decode<M>(g, S, gam, (int)cs.e, psi, omg);  // succeeded in the scan pass
        }
        for (unsigned long long w = wr; w; w &= w - 1) {
            const uint32_t r = (uint32_t)(__ffsll((long long)w) - 1);
            const bool erased = (absent >> r) & 1;
            uint32_t val = 0;
            if (any) {
                bool errata;
                correct_value<M>(g, psi, omg, p.logx[r], p.logv[r], errata, val);
            }
            uint8_t *dst = col + (size_t)r * p.stride;
            if (erased) *dst = (uint8_t)val;
            else if (val) *dst = (uint8_t)(*dst ^ val);
        }
    }
}

}  // namespace garage_ec
