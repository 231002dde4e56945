// mapf_env_kernel.cuh -- env-per-thread step kernel (sm_100a) of the batched MAPF transition.
//
// Reference semantics: src/environments/reference_model_multi_agent.py ("ENV:line").
//
// Why a second mapping.  The lane-per-agent kernel (mapf_kernels.cuh) spends ~1 900 warp
// instructions per 32 agent-steps: every lane re-executes the env-level coordination (ballots,
// candidate loops that run to the longest lane, predicated single-lane blocks) and ncu shows it
// bound by instruction issue, not by HBM.  Here ONE THREAD owns ONE ENV and walks its agents in
// index order exactly like the reference's python loop (ENV:502-563), so the sequential
// semantics need no cross-lane protocol at all and nothing is computed redundantly:
//   * the occupancy and goal owner grids (ENV:102-103) are two bitboards (one 32-bit word per map
//     row, map width <= 32) in shared memory, laid out [row][lane] so a warp's accesses never
//     conflict; a move is "test one bit, clear one bit, set one bit";
//   * staggered observations (ENV:528-536, SURVEY F3) fall out of the walk itself: agent i's window rows are
//     read right after its own move, when the boards are exactly snapshot i;
//   * a window row is ONE table lookup: the (obstacle | goal) and (agent | goal) bits of the row, side by
//     side, index a 4^V-entry table of V nibbles, and PRMT turns 4 nibbles into 4 output bytes;
//   * the walk is software-pipelined by hand over the 4 agents of a quad: phase A does the moves and
//     collects the raw window rows (the only part that must see the evolving board), phase B the table
//     lookups and the byte rows of all four agents at once (independent chains that overlap);
//   * rare per-env events -- a lifelong goal reassignment, an episode end with its in-launch reset -- are
//     served by the whole warp working on that ONE env (lane = agent / map row), not by 32 lanes walking
//     along for the sake of one: the launch is a single wave, its time is the slowest warp's;
//   * lock neighbourhoods, intent blocking, co-location and the wait-for graph use per-row /
//     per-column agent masks (their AND is the owner set of a cell) built in the board memory
//     once the boards are dead; wait-for cycles are found by stripping leaves off the functional
//     graph with agent bitmasks;
//   * state is read and written with 128-bit accesses (4 agents per access); the byte channels
//     (local_obs, action_mask) go through a per-warp staging tile and leave coalesced.
// No tensor cores: there is no dense contraction on this path.
#pragma once

#include "mapf_kernels.cuh"

namespace mapf {

// Shared-memory carve-up of the env-per-thread kernel.  Everything the hot loops address is at a
// compile-time offset (folded into the LDS/STS immediates); only the per-warp stride is a run-time value.
// The CTA-wide tables [0, tables_bytes) are built once on the host (mapf_set_map) and copied in.
constexpr int ENV_MAX_ROWS = 64;       // map rows the env-per-thread kernel accepts (columns: 32)
constexpr int ENV_T1_OFF = 0;          // u32[1 << V]: bit j -> nibble j
constexpr int ENV_KTH_OFF = 512;       // u8[32*8]: position of the (k+1)-th set bit of a 5-bit mask
constexpr int ENV_FREEROW_OFF = 768;   // u32[R]: bit c = cell (r, c) is free
constexpr int ENV_FREEBITS_OFF = 1024; // u32[fw]: cell-linear free bitmap (reset draws, ENV:267-282)
constexpr int ENV_GDT_OFF = 1280;      // float[(2R-1)+(2C-1)] goal-delta quotients (ENV:330-335)
constexpr int ENV_LUT_OFF = 2048;      // obstacle window of every cell: u32[R*32] (V <= 5) or u64[R*32] (V = 7)
constexpr int ENV_ROW_PAD = 2;         // zero rows around the owner masks of the epilogue (lock_nearby_manhattan <= 2)

// stage row of one env and quad: 4 * V2 observation bytes + 20 action-mask bytes, odd word stride
__host__ __device__ constexpr int env_stage_stride(int V2) { return ((4 * V2 + 20 + 3) / 4) | 1; }
// the stage also lands the 64-byte env-word rows of the warp's 32 envs after the walk: at least 2 KB
__host__ __device__ constexpr int env_stage_bytes(int V2) {
    return 32 * env_stage_stride(V2) * 4 > 32 * 64 ? 32 * env_stage_stride(V2) * 4 : 32 * 64;
}

struct EnvLayout {
    int tables_bytes;  // multiple of 16
    int pre_off;       // prefix counts of the free-cell bitmap (reset draws)
    int warp_bytes;    // per-warp block: [stage][occupancy boards][goal boards][agent records]
    int board_rows;    // max(R, C, N) + 2 * ENV_ROW_PAD
    int nq;            // ceil(N / 4)
    int total_bytes;
};

__host__ __device__ inline EnvLayout make_env_layout(int N, int R, int C, int SR, int fw, int warps) {
    const int V = 2 * SR + 1, V2 = V * V;
    EnvLayout E;
    E.pre_off = (ENV_LUT_OFF + R * 32 * (V > 5 ? 8 : 4) + 15) & ~15;
    E.tables_bytes = E.pre_off + 65 * 4 + 12;                     // u32[fw + 1]: free cells in front of bitmap word w (fw <= 64)
    E.board_rows = R > C ? R : C;
    if (N > E.board_rows) E.board_rows = N;
    E.board_rows += 2 * ENV_ROW_PAD;
    E.nq = (N + 3) / 4;
    int w = env_stage_bytes(V2);             // stage: one row per lane
    w += E.board_rows * 32 * 4;              // occupancy boards: u32 [row][lane]
    w += E.board_rows * 32 * 4;              // goal boards: u32 [row][lane]
    w += 4 * E.nq * 32 * 4;                  // agent records: u32 [agent][lane]
    w = (w + 15) & ~15;
    E.warp_bytes = w;
    // window rows above / below the map read up to 3 board rows beyond a warp's boards: keep that inside the allocation
    E.total_bytes = E.tables_bytes + w * warps + 1024;
    (void)fw;
    return E;
}

// quad (4 consecutive agents of one env) loads / stores; VEC = N % 4 == 0 => one 128-bit access
template <bool VEC>
__device__ __forceinline__ uint4 ldq32(const uint32_t *a, size_t i, int i0, int N, bool ok, uint32_t d) {
    uint4 v = make_uint4(d, d, d, d);
    if (VEC) { if (ok) v = *reinterpret_cast<const uint4 *>(a + i); }
    else if (ok) {
        if (i0 + 0 < N) v.x = a[i + 0];
        if (i0 + 1 < N) v.y = a[i + 1];
        if (i0 + 2 < N) v.z = a[i + 2];
        if (i0 + 3 < N) v.w = a[i + 3];
    }
    return v;
}
template <bool VEC>
__device__ __forceinline__ void stq32(uint32_t *a, size_t i, int i0, int N, bool ok, uint4 v) {
    if (!ok) return;
    if (VEC) *reinterpret_cast<uint4 *>(a + i) = v;
    else {
        if (i0 + 0 < N) a[i + 0] = v.x;
        if (i0 + 1 < N) a[i + 1] = v.y;
        if (i0 + 2 < N) a[i + 2] = v.z;
        if (i0 + 3 < N) a[i + 3] = v.w;
    }
}
template <bool VEC>
__device__ __forceinline__ uint32_t ldq8(const uint8_t *a, size_t i, int i0, int N, bool ok) {
    uint32_t v = 0;
    if (VEC) { if (ok) v = *reinterpret_cast<const uint32_t *>(a + i); }
    else if (ok) {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (i0 + k < N) v |= (uint32_t)a[i + k] << (8 * k);
    }
    return v;
}
template <bool VEC>
__device__ __forceinline__ void stq8(uint8_t *a, size_t i, int i0, int N, bool ok, uint32_t v) {
    if (!ok) return;
    if (VEC) *reinterpret_cast<uint32_t *>(a + i) = v;
    else {
#pragma unroll
        for (int k = 0; k < 4; ++k) if (i0 + k < N) a[i + k] = (uint8_t)(v >> (8 * k));
    }
}
template <bool VEC>
__device__ __forceinline__ uint2 ldq16(const int16_t *a, size_t i, int i0, int N, bool ok) {
    uint2 v = make_uint2(0, 0);
    if (VEC) { if (ok) v = *reinterpret_cast<const uint2 *>(a + i); }
    else if (ok) {
        if (i0 + 0 < N) v.x |= (uint32_t)(uint16_t)a[i + 0];
        if (i0 + 1 < N) v.x |= (uint32_t)(uint16_t)a[i + 1] << 16;
        if (i0 + 2 < N) v.y |= (uint32_t)(uint16_t)a[i + 2];
        if (i0 + 3 < N) v.y |= (uint32_t)(uint16_t)a[i + 3] << 16;
    }
    return v;
}
template <bool VEC>
__device__ __forceinline__ void stq16(int16_t *a, size_t i, int i0, int N, bool ok, uint2 v) {
    if (!ok) return;
    if (VEC) *reinterpret_cast<uint2 *>(a + i) = v;
    else {
        if (i0 + 0 < N) a[i + 0] = (int16_t)(v.x & 0xFFFFu);
        if (i0 + 1 < N) a[i + 1] = (int16_t)(v.x >> 16);
        if (i0 + 2 < N) a[i + 2] = (int16_t)(v.y & 0xFFFFu);
        if (i0 + 3 < N) a[i + 3] = (int16_t)(v.y >> 16);
    }
}

__device__ __forceinline__ uint32_t qget(const uint4 &v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }
__device__ __forceinline__ void qset(uint4 &v, int k, uint32_t x) { if (k == 0) v.x = x; else if (k == 1) v.y = x; else if (k == 2) v.z = x; else v.w = x; }
// u16 lane k of a 4 x u16 pack
__device__ __forceinline__ uint32_t hget(const uint2 &v, int k) { const uint32_t w = (k < 2) ? v.x : v.y; return (k & 1) ? (w >> 16) : (w & 0xFFFFu); }
__device__ __forceinline__ void hset(uint2 &v, int k, uint32_t x) {
    uint32_t &w = (k < 2) ? v.x : v.y;
    w = (k & 1) ? ((w & 0x0000FFFFu) | (x << 16)) : ((w & 0xFFFF0000u) | (x & 0xFFFFu));
}
// cell code = row * 32 + col (map width <= 32); the state tensors hold int16 (row, col) pairs
__device__ __forceinline__ uint32_t code_of(uint32_t packed) { return ((packed & 0xFFFFu) << 5) | (packed >> 16); }
__device__ __forceinline__ uint32_t packed_of(uint32_t code) { return (code >> 5) | ((code & 31u) << 16); }

// One Philox call serves the 4 agents of a quad (scripts/benchmark_multi_agent_env.py:38-57).
__device__ __forceinline__ uint4 sample_quad(unsigned long long seed, long long env_global, int quad,
                                             unsigned long long counter) {
    Philox ph(seed ^ 0xA511E9B3ull, env_global);
    return ph((uint32_t)counter, (uint32_t)(counter >> 32), (uint32_t)quad, 0x41435421u);
}

// Host-side image of the CTA-wide tables (mapf_set_map); `rows` are the padded obstacle bit-rows of
// the lane-per-agent kernel (bit c + PAD of row r + PAD = obstacle or out of bounds, ENV:718).
inline void build_env_tables(int SR, int R, int C, int wpr, int fw, const uint32_t *rows,
                             const uint32_t *free_bits, int normalize, float den0, float den1, unsigned char *img,
                             int pre_off) {
    const int V = 2 * SR + 1;
    {
        uint32_t *pre = reinterpret_cast<uint32_t *>(img + pre_off);
        uint32_t acc = 0;
        for (int w = 0; w <= 64; ++w) {
            pre[w] = acc;
            if (w < fw) acc += (uint32_t)__builtin_popcount(free_bits[w]);
        }
    }
    auto rowbits = [&](int r, int c0, int n) {  // n bits starting at map column c0 of map row r (padding = 1)
        unsigned long long x = 0;
        for (int j = 0; j < n; ++j) {
            const int bit = c0 + j + PAD;
            if ((rows[(r + PAD) * wpr + (bit >> 5)] >> (bit & 31)) & 1u) x |= 1ull << j;
        }
        return x;
    };
    uint32_t *t1 = reinterpret_cast<uint32_t *>(img + ENV_T1_OFF);
    for (int x = 0; x < (1 << V); ++x) {
        uint32_t s = 0;
        for (int j = 0; j < V; ++j) s |= ((uint32_t)(x >> j) & 1u) << (4 * j);
        t1[x] = s;
    }
    uint8_t *kth = img + ENV_KTH_OFF;
    for (int m = 0; m < 32; ++m)
        for (int k = 0; k < 8; ++k) {
            int pos = 0, seen = 0;
            for (int b = 0; b < 5; ++b)
                if ((m >> b) & 1) { if (seen == k) pos = b; ++seen; }
            kth[m * 8 + k] = (uint8_t)(k < seen ? pos : 0);
        }
    for (int cell = 0; cell < R * 32; ++cell) {
        const int r = cell >> 5, c = cell & 31;
        unsigned long long w = 0;
        if (c < C)
            for (int wr = 0; wr < V; ++wr) w |= rowbits(r - SR + wr, c - SR, V) << (wr * V);
        if (V > 5) reinterpret_cast<unsigned long long *>(img + ENV_LUT_OFF)[cell] = w;
        else reinterpret_cast<uint32_t *>(img + ENV_LUT_OFF)[cell] = (uint32_t)w;
    }
    uint32_t *freerow = reinterpret_cast<uint32_t *>(img + ENV_FREEROW_OFF);
    for (int r = 0; r < R; ++r) freerow[r] = (uint32_t)(~rowbits(r, 0, C) & (C >= 32 ? 0xFFFFFFFFull : ((1ull << C) - 1ull)));
    uint32_t *fb = reinterpret_cast<uint32_t *>(img + ENV_FREEBITS_OFF);
    for (int i = 0; i < fw; ++i) fb[i] = free_bits[i];
    float *gdt = reinterpret_cast<float *>(img + ENV_GDT_OFF);
    const int nr = 2 * R - 1, n = nr + 2 * C - 1;
    for (int i = 0; i < n; ++i) {   // ENV:330-335: one IEEE division per distinct (goal - pos) value
        const bool row = i < nr;
        const float d = (float)(row ? i - (R - 1) : i - nr - (C - 1));
        gdt[i] = normalize ? d / (row ? den0 : den1) : d;
    }
}

// nibble j of `sel` (values 0..4) -> byte j: one PRMT against the byte table {0,1,2,3,4}
__device__ __forceinline__ uint32_t nibbles_to_bytes(uint32_t sel) {
    uint32_t w;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(w) : "r"(0x03020100u), "r"(0x00000004u), "r"(sel));
    return w;
}
// nibble j of `sel` (values 0..3) -> byte j of {0, 1, 2, 4}: the two-plane window rows of the walk (3 = both planes = OTHER_GOAL)
__device__ __forceinline__ uint32_t nibbles_to_bytes_0124(uint32_t sel) {
    uint32_t w;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(w) : "r"(0x04020100u), "r"(0u), "r"(sel));
    return w;
}
// bits 0..3 of m -> bytes 0/1
__device__ __forceinline__ uint32_t spread4(uint32_t m) { return ((m & 15u) * 0x00204081u) & 0x01010101u; }
// bit `b` of each of the 4 bytes of w -> nibble
__device__ __forceinline__ uint32_t gather4(uint32_t w, int b) { return ((((w >> b) & 0x01010101u) * 0x01020408u) >> 24) & 15u; }
// cell delta of an action {0, -32, +1, +32, -1} (ENV:104-113 on cell codes)
__device__ __forceinline__ int action_delta(uint32_t a) { return (int)(int8_t)__byte_perm(0x2001E000u, 0x000000FFu, a); }
// Loads from the CTA-wide immutable tables (and, inside one walk, the goal boards) as non-volatile asm without a
// memory clobber: the compiler may order them freely against the stores around them, which is what lets the
// look-ups of four agents overlap.  `tag` is an artificial dependency (the round number) that keeps a load from
// being merged with its twin in another round, where the goal boards may differ.  Addresses are shared-window bytes.
__device__ __forceinline__ uint32_t lds_pure(uint32_t saddr) {
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint32_t lds_pure(uint32_t saddr, uint32_t tag) {
    uint32_t v;
    asm("{ .reg .b32 t; mov.b32 t, %2; ld.shared.u32 %0, [%1]; }" : "=r"(v) : "r"(saddr), "r"(tag));
    return v;
}
__device__ __forceinline__ uint32_t lds_pure_u8(uint32_t saddr) {
    uint32_t v;
    asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
template <typename WB> __device__ __forceinline__ WB lut_ld(uint32_t saddr);
template <> __device__ __forceinline__ uint32_t lut_ld<uint32_t>(uint32_t saddr) { return lds_pure(saddr); }
template <> __device__ __forceinline__ unsigned long long lut_ld<unsigned long long>(uint32_t saddr) {
    unsigned long long v;
    asm("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(saddr));
    return v;
}
// stage-row store: volatile (kept, and kept in order with the other stage stores) but no memory clobber -- the stage
// is only read after the __syncwarp() in front of the flush, so board loads may move across it
__device__ __forceinline__ void sts_stage(uint32_t saddr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(saddr), "r"(v));
}

__device__ __forceinline__ void sts_stage_u8(uint32_t saddr, uint32_t v) {   // byte patch behind the word stores (same ordering class)
    asm volatile("st.shared.u8 [%0], %1;" ::"r"(saddr), "r"(v));
}

// agent record in shared memory, rec[agent * EPW] per env:
//   bits 0..10 cell code | 11..13 action | 14 target blocked (obstacle / out of bounds) | 16..31 int16 distance delta
constexpr uint32_t REC_CODE = 0x7FFu;

// One thread owns one env (32 envs per warp) and walks its agents in index order, a quad (4 agents = one 128-bit
// state access) at a time.
// FAST: the benchmark's configuration (lifelong goals, lock metrics on) as compile-time constants -- the other
// branches and their uniform tests drop out of the hot loops (smaller instruction footprint); same results.
// One CTA of 14 warps per SM (shared memory allows no more).  The register file is split four ways (16 K registers per
// scheduler) and two of the schedulers hold 4 of the 14 warps: 4 x 32 x 128 registers is all there is, so 128 it is
// (144 would fit the 64 K total but not the partitions: "too many resources requested for launch").
// MANY: mapf_step_many -- `p.inner_steps` consecutive env steps in ONE launch, every warp on its own tile from the first step
// to the last (no grid-wide dependency between steps: the tail of the one-wave launch is paid once, and what a step
// reads is what the step before just wrote, in L2).  Step it > 0 takes the actions the fused sampler drew in step
// it - 1 and writes its outputs `p.out_step_stride` envs further into the caller's [K, B, ...] buffers.
template <int SR, bool VEC, bool FAST = false, bool MANY = false>
__global__ void __launch_bounds__(448, 1) mapf_step_env_kernel(const KParams p, const EnvLayout E) {
    const bool kLifelong = FAST ? true : p.lifelong;
    const bool kLock = FAST ? true : p.lock_enabled;
    constexpr int V = 2 * SR + 1, V2 = V * V;
    constexpr uint32_t VM = (1u << V) - 1u;
    constexpr uint32_t M4 = VM << 2;          // a window row, pre-scaled by 4 (byte offset into the tables)
    constexpr int OBS_W = V2;                 // observation words per quad and env (4 * V2 bytes)
    constexpr int STRIDE = env_stage_stride(V2);
    constexpr int STAGE_BYTES = env_stage_bytes(V2);
    constexpr int CTR = SR * V + SR;
    constexpr int PADR = ENV_ROW_PAD;
    using WB = typename WinBits<V>::type;
    extern __shared__ __align__(16) unsigned char esm[];
    const unsigned full = 0xFFFFFFFFu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    const int N = p.N, R = p.R, C = p.C, NQ = E.nq;

    // ------------------------------------------------------------------ CTA-wide tables (built on the host)
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(p.env_tables);
        uint4 *dst = reinterpret_cast<uint4 *>(esm);
        for (int i = tid; i < (E.tables_bytes >> 4); i += blockDim.x) dst[i] = src[i];
    }
    // Programmatic dependent launch: the next launch in the stream may place its CTAs as ours exit and run the
    // table copy above (the tables are immutable between launches) while the slowest CTAs of this launch finish;
    // everything that touches env state waits here for the previous launch to complete and flush.
    asm volatile("griddepcontrol.launch_dependents;");
    // While the previous launch drains: ask L2 for the state rows of my first tile (a hint -- L2 is the coherence point,
    // whatever the previous launch still writes there is what the loads behind the wait will see).  With a working set
    // beyond L2 (several env batches stepped in turn) the first loads of a warp would otherwise all miss to HBM at the
    // same moment, with nothing to overlap them with.
    if (p.env_prefetch) {
        const int tile0 = blockIdx.x * (blockDim.x >> 5) + (tid >> 5);
        const int left = p.B - tile0 * 32;
        if (left > 0) {
            const size_t a0 = (size_t)tile0 * 32 * (size_t)p.N;
            const uint32_t agents = (uint32_t)(left < 32 ? left : 32) * (uint32_t)p.N;
            const void *ptr = nullptr;
            uint32_t bytes = agents * 4u;
            switch (tid & 31) {
                case 0: ptr = p.positions + a0; break;
                case 1: ptr = p.goals + a0; break;
                case 2: ptr = p.lock_gp + a0; break;
                case 3: ptr = p.lock_mv + a0; break;
                case 4: ptr = p.lock_fm + a0; break;
                case 5: ptr = p.actions ? p.actions + a0 : nullptr; bytes = agents; break;
                case 6: ptr = p.agent_flags + a0; bytes = agents; break;
                case 7: ptr = p.env_words + (size_t)tile0 * 32 * 4; bytes = (uint32_t)(left < 32 ? left : 32) * 64u; break;
                default: break;
            }
            bytes &= ~15u;
            if (ptr && bytes && (reinterpret_cast<uintptr_t>(ptr) & 15) == 0)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"(bytes) : "memory");
        }
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
    __syncthreads();
    const char *t1b = reinterpret_cast<const char *>(esm + ENV_T1_OFF);
    const uint8_t *kth = esm + ENV_KTH_OFF;
    const WB *lut = reinterpret_cast<const WB *>(esm + ENV_LUT_OFF);
    const uint32_t *freerow = reinterpret_cast<const uint32_t *>(esm + ENV_FREEROW_OFF);
    const uint32_t *freebits = reinterpret_cast<const uint32_t *>(esm + ENV_FREEBITS_OFF);
    const float *gdt = reinterpret_cast<const float *>(esm + ENV_GDT_OFF);
    const uint32_t esm_s = (uint32_t)__cvta_generic_to_shared(esm);
    const uint32_t t1_s = esm_s + ENV_T1_OFF, kth_s = esm_s + ENV_KTH_OFF, lut_s = esm_s + ENV_LUT_OFF;
    const uint32_t *freepre = reinterpret_cast<const uint32_t *>(esm + E.pre_off);
    // k-th free cell (cell-linear order, ENV:82) by binary search over the prefix counts
    auto kth_free = [&](int k) -> int {
        int lo = 0;
#pragma unroll
        for (int stp = 32; stp >= 1; stp >>= 1)
            if (lo + stp < p.fw && (int)freepre[lo + stp] <= k) lo += stp;
        return lo * 32 + (int)__fns(freebits[lo], 0, k - (int)freepre[lo] + 1);
    };

    unsigned char *wsm = esm + E.tables_bytes + warp * E.warp_bytes;
    uint32_t *stage_w = reinterpret_cast<uint32_t *>(wsm);                              // [lane][STRIDE] words
    uint32_t *my_stage = stage_w + lane * STRIDE;
    const uint32_t my_stage_s = (uint32_t)__cvta_generic_to_shared(my_stage);
    uint32_t *occ_w = reinterpret_cast<uint32_t *>(wsm + STAGE_BYTES);                  // occupancy boards [row][lane]
    uint32_t *goal_w = occ_w + E.board_rows * 32;                                       // goal boards [row][lane]
    uint32_t *rec_w = goal_w + E.board_rows * 32;                                       // agent records [agent][lane]
    uint32_t *occ = occ_w + lane, *goalb = goal_w + lane, *rec = rec_w + lane;          // mine: row r at occ[r * 32]
    const uint32_t goalb_s = (uint32_t)__cvta_generic_to_shared(goalb);
    // owner masks of the epilogue (dead board memory, row stride 32 words): bit a of rowm[r] / colm[c] = agent a's row / column
    uint32_t *rowm = occ, *colm = goalb;
    const int ntiles = (p.B + 31) / 32;
    uint32_t errs = 0;
    const uint32_t mdw = p.dw >= 32 ? full : ((1u << p.dw) - 1u);
    const uint32_t mlw = p.lw >= 32 ? full : ((1u << p.lw) - 1u);
    const uint32_t allN = (N >= 32) ? full : ((1u << N) - 1u);

    // Final-state observation of agent `lane` of ONE env, the whole warp on that env (ENV:565-575 after a goal
    // reassignment, ENV:459-468 after a reset): window, mask, goal delta, pressure flag, next action -- straight to
    // global memory.  occ_e / goal_e: the env's boards (row r at [r * 32]); ctr2: my own cell belongs to another agent.
    auto emit_final = [&](size_t abe, size_t oo, unsigned long long sctr, long long eg, const uint32_t *occ_e,
                          const uint32_t *goal_e, uint32_t code, uint32_t gcode, uint32_t bp_bit, bool ctr2) {
        if (lane >= N) return;
        const int r = (int)(code >> 5), c = (int)(code & 31u);
        const WB obst = lut[code];
        const int sa = c > SR ? c - SR : 0, sb2 = (c < SR ? SR - c : 0) + 2;
        const uint32_t *orow = occ_e + (r - SR) * 32, *grow = goal_e + (r - SR) * 32;
        uint32_t acc[(4 * V2 + 31) / 32 + 1];
#pragma unroll
        for (int j = 0; j < (int)(sizeof(acc) / sizeof(acc[0])); ++j) acc[j] = 0;
        uint32_t blk_up = 0, blk_mid = 0, blk_dn = 0;
#pragma unroll
        for (int wr = 0; wr < V; ++wr) {
            const uint32_t bx = orow[wr * 32], by = grow[wr * 32];
            const uint32_t o4 = (wr * V >= 2 ? (uint32_t)(obst >> (wr * V - 2)) : (uint32_t)(obst << 2)) & M4;
            const uint32_t MC = (wr == SR) ? (M4 & ~(4u << SR)) : M4;
            const uint32_t occ4 = ((bx >> sa) << sb2) & MC;
            const uint32_t agent4 = occ4 & ~o4, blk4 = occ4 | o4;
            const uint32_t g4 = ((by >> sa) << sb2) & M4 & ~blk4;
            if (wr == SR - 1) blk_up = blk4;
            if (wr == SR) blk_mid = blk4;
            if (wr == SR + 1) blk_dn = blk4;
            const uint32_t t = *reinterpret_cast<const uint32_t *>(t1b + o4) +
                               (*reinterpret_cast<const uint32_t *>(t1b + agent4) << 1) +
                               (*reinterpret_cast<const uint32_t *>(t1b + g4) << 2);
            const int bitpos = 4 * V * wr, wi = bitpos >> 5, sh = bitpos & 31;
            acc[wi] |= t << sh;
            if (sh + 4 * V > 32) acc[wi + 1] |= t >> (32 - sh);
        }
        const uint32_t am = 1u | ((~blk_up >> (2 + SR)) & 1u) << 1 | ((~blk_mid >> (2 + SR + 1)) & 1u) << 2 |
                            ((~blk_dn >> (2 + SR)) & 1u) << 3 | ((~blk_mid >> (2 + SR - 1)) & 1u) << 4;
        if (p.o_local_obs) {
            uint8_t *ob = p.o_local_obs + (abe + oo + lane) * V2;
#pragma unroll
            for (int n = 0; n < V2; ++n) ob[n] = (uint8_t)((acc[n >> 3] >> (4 * (n & 7))) & 0xFu);
            const int dr = (int)(gcode >> 5) - r + SR, dc = (int)(gcode & 31u) - c + SR;
            if ((unsigned)dr < (unsigned)V && (unsigned)dc < (unsigned)V) {   // own goal: code 3
                const int ci = dr * V + dc;
                const bool occ_other = (ci != CTR) && ((occ_e[(gcode >> 5) * 32] >> (gcode & 31u)) & 1u);
                if (!((obst >> ci) & 1) && !occ_other) ob[ci] = 3;
            }
            if (ctr2) ob[CTR] = 2;   // injected co-location (ENV:737-739)
        }
        if (p.o_action_mask) {
#pragma unroll
            for (int k = 0; k < 5; ++k) p.o_action_mask[(abe + oo + lane) * 5 + k] = (int8_t)((am >> k) & 1u);
        }
        if (p.o_goal_delta) {
            const int gi0 = (int)(gcode >> 5) - r + (R - 1), gi1 = (int)(gcode & 31u) - c + (C - 1) + 2 * R - 1;
            p.o_goal_delta[abe + oo + lane] = make_float2(gdt[gi0], gdt[gi1]);
        }
        if (p.o_blocking_prev) p.o_blocking_prev[abe + oo + lane] = (uint8_t)bp_bit;
        if (p.sample_mode) {
            const uint4 rnd = sample_quad(p.seed, eg, lane >> 2, sctr);
            const uint32_t x = qget(rnd, lane & 3);
            const uint32_t na = p.sample_mode == 1 ? kth[am * 8 + __umulhi(x, (uint32_t)__popc(am))] : __umulhi(x, 5u);
            p.o_next_actions[abe + lane] = (int8_t)na;
        }
    };

    for (int tile = blockIdx.x * warps + warp; tile < ntiles; tile += gridDim.x * warps) {
    const int env = tile * 32 + lane;
    const bool ok = env < p.B;
    const size_t ab = (size_t)(ok ? env : 0) * N;
    const long long env_global = p.env_id_base + env;
    const size_t env0 = (size_t)tile * 32;
    for (int it = 0; it < (MANY ? p.inner_steps : 1); ++it) {
    const size_t so = MANY ? (size_t)it * (size_t)p.out_step_stride : 0, oo = so * (size_t)N;   // this step's output rows
    const unsigned long long sctr = p.sample_counter + (MANY ? (unsigned long long)it : 0ull);
    const int8_t *acts_in = (MANY && it > 0) ? p.o_next_actions : p.actions;

    // ---------------------------------------------------------------- the two env words the walk needs (the rest: epilogue)
    int lock_count = 0, lock_head = 0;
    if (ok) {
        const int *ew1 = reinterpret_cast<const int *>(p.env_words + (size_t)env * 4);
        lock_count = ew1[MAPF_W_LOCK_COUNT];
        lock_head = ew1[MAPF_W_LOCK_HEAD];
    }
    const int count_after = lock_count + 1;
    if (lock_head < 0 || lock_head >= p.lw) lock_head = 0;
    const int slot_new = lock_head;
    const int slot_next = (lock_head + 1 == p.lw) ? 0 : lock_head + 1;
    const bool use_ring = kLock && count_after >= p.lw && p.lw > 1;

    uint32_t reached_m = 0, completed_m = 0, bprev_m = 0;   // agent_flags of the previous step (MAPF_AF_*), one bit per agent
    // Injected states with several agents on one cell (the only way ENV:658-666 fires).  A set bit of the occupancy
    // board is exactly "_occupancy_owner != -1" (ENV:516-526), so moves need nothing extra; the observation of a
    // co-located agent does: the owner of a shared cell is its highest index (ENV:200-205) and everybody else sees
    // OTHER_AGENT in the centre of its own window (ENV:737-739).  solo_m: bit a = agent a owns the cell it stands on.
    bool degen = false;
    uint32_t solo_m = 0xFFFFFFFFu;
    // ---------------------------------------------------------------- pre-pass: agent records and owner boards of the state before the step
    for (int r = 0; r < E.board_rows; ++r) { occ[r * 32] = 0u; goalb[r * 32] = 0u; }
    uint32_t dup = 0;
    auto prepass_quad = [&](int i0, const uint4 &pq, const uint4 &gq, uint32_t act4, uint32_t fl4) {
        reached_m |= gather4(fl4, 0) << i0;      // MAPF_AF_REACHED
        completed_m |= gather4(fl4, 1) << i0;    // MAPF_AF_COMPLETED_ONCE
        bprev_m |= gather4(fl4, 2) << i0;        // MAPF_AF_BLOCKING_PREV
        solo_m &= ~(gather4(fl4, 3) << i0);      // MAPF_AF_NOT_OWNER (injected co-location, carried over from earlier steps)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (VEC || i0 + k < N) {   // VEC: N is a multiple of 4, every quad is full
                const uint32_t code = code_of(qget(pq, k)), gcode = code_of(qget(gq, k));
                int a = (int)(int8_t)(act4 >> (8 * k));
                if (a < 0 || a > 4) { errs |= MAPF_DEV_ERR_INVALID_ACTION; a = 0; }
                // target obstacle / bounds from the cell's obstacle window (ENV:516-521)
                const uint32_t nbi = __byte_perm((uint32_t)CTR | ((uint32_t)(CTR - V) << 8) | ((uint32_t)(CTR + 1) << 16) |
                                                 ((uint32_t)(CTR + V) << 24), (uint32_t)(CTR - 1), (uint32_t)a) & 0xFFu;
                const uint32_t tblocked = ((uint32_t)lut[code] >> nbi) & 1u;
                rec[(i0 + k) * 32] = code | ((uint32_t)a << 11) | (tblocked << 14) | (gcode << 16);   // goal rides in the (still unused) delta half
                if (ok) {
                    // shared-memory atomics instead of read-modify-write chains: the 2N board updates of the pre-pass
                    // are independent instructions in flight together (the returned word is only looked at afterwards)
                    if (!((fl4 >> (8 * k + 3)) & 1u)) {   // only the owner of a cell marks it (always, in legal states)
                        const uint32_t cb0 = 1u << (code & 31u);
                        dup |= atomicOr(&occ[(code >> 5) * 32], cb0) & cb0;   // two agents on one cell: an injected state (ENV:658-666)
                    } else degen = true;
                    atomicOr(&goalb[(gcode >> 5) * 32], 1u << (gcode & 31u));
                }
            }
        }
    };
    for (int q = 0; q < NQ; q += 2) {   // two quads per turn: eight state loads in flight before the first is needed
        const int i0 = 4 * q, i1 = i0 + 4;
        const bool two = q + 1 < NQ;
        const uint4 pq0 = ldq32<VEC>(p.positions, ab + i0, i0, N, ok, 0u);
        const uint4 gq0 = ldq32<VEC>(p.goals, ab + i0, i0, N, ok, 0u);
        const uint32_t ac0 = acts_in ? ldq8<VEC>(reinterpret_cast<const uint8_t *>(acts_in), ab + i0, i0, N, ok) : 0u;
        const uint32_t fl0 = ldq8<VEC>(p.agent_flags, ab + i0, i0, N, ok);
        const uint4 pq1 = ldq32<VEC>(p.positions, ab + i1, i1, N, ok && two, 0u);
        const uint4 gq1 = ldq32<VEC>(p.goals, ab + i1, i1, N, ok && two, 0u);
        const uint32_t ac1 = acts_in ? ldq8<VEC>(reinterpret_cast<const uint8_t *>(acts_in), ab + i1, i1, N, ok && two) : 0u;
        const uint32_t fl1 = ldq8<VEC>(p.agent_flags, ab + i1, i1, N, ok && two);
        prepass_quad(i0, pq0, gq0, ac0, fl0);
        if (two) prepass_quad(i1, pq1, gq1, ac1, fl1);
    }
    degen |= dup != 0;
    if (degen) {   // rare: among agents that claim the same cell the highest index owns it (ENV:200-205)
        const uint32_t claim = solo_m;
        for (int i = 0; i < N; ++i)
            for (int j = i + 1; j < N; ++j)
                if (((claim >> j) & 1u) && ((rec[i * 32] ^ rec[j * 32]) & REC_CODE) == 0u) { solo_m &= ~(1u << i); break; }
    }

    uint32_t moved_m = 0, failed_m = 0, gstep_m = 0, ongoal_m = 0;
    uint32_t Gd = 0, Md = 0, Fd = 0, Gl = 0, Ml = 0;
    const unsigned act_w = __ballot_sync(full, ok);
    const bool masked_sampler = p.sample_mode == 1;

    // ---------------------------------------------------------------- the agent walk (ENV:502-563), a quad at a time
    // lock history of the quad AFTER the one being walked: its loads are issued behind phase A and land during
    // phase B and the flush (one warp has ~3 others to hide a DRAM round trip behind -- not enough)
    uint4 gp_n = make_uint4(0, 0, 0, 0), mv_n = gp_n, fm_n = gp_n;
    uint2 ring_n = make_uint2(0u, 0u);
    auto load_lock = [&](int i0) {
        if (!kLock) return;
        gp_n = ldq32<VEC>(p.lock_gp, ab + i0, i0, N, ok, 0u);
        mv_n = ldq32<VEC>(p.lock_mv, ab + i0, i0, N, ok, 0u);
        fm_n = ldq32<VEC>(p.lock_fm, ab + i0, i0, N, ok, 0u);
        if (use_ring) ring_n = ldq16<VEC>(p.lock_dist, ((size_t)(ok ? env : 0) * p.lw + slot_next) * N + i0, i0, N, ok);
    };
    load_lock(0);
    for (int q = 0; q < NQ; ++q) {
        const int i0 = 4 * q;
        uint32_t rv4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) rv4[k] = (VEC || i0 + k < N) ? rec[(i0 + k) * 32] : 0u;
        uint4 gpq = gp_n, mvq = mv_n, fmq = fm_n;
        const uint2 ringq = ring_n;
        uint4 rnd = make_uint4(0, 0, 0, 0);
        if (p.sample_mode) rnd = sample_quad(p.seed, env_global, q, sctr);
        uint32_t ds[4] = {0, 0, 0, 0}, cd[4] = {0, 0, 0, 0}, gc[4] = {0, 0, 0, 0};
        uint32_t masks4 = 0, next4 = 0;
        int patch[4];
        // Phase A -- everything that has to see the occupancy board as it is right after agent k's own move
        // (snapshot k, ENV:528-536): the move itself and the raw window rows.  Nothing here waits for a table
        // look-up or writes the stage, so the board accesses of the four agents sit back to back in program
        // order and the arithmetic of agent k overlaps the shared-memory latency of agent k + 1.
        // win[k][wr]: row wr of agent k's window as V nibbles (codes 1 / 2 / 3, see below).
        uint32_t win[4][V];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            patch[k] = 4 * V2 + 20;
#pragma unroll
            for (int wr = 0; wr < V; ++wr) win[k][wr] = 0;
            if (!VEC && i0 + k >= N) continue;
            const uint32_t bit = 1u << (i0 + k);
            uint32_t code = rv4[k] & REC_CODE;
            const uint32_t gcode = rv4[k] >> 16;
            const uint32_t ocode = code;
            const uint32_t a = (rv4[k] >> 11) & 7u;
            // ENV:512-526: target cell; obstacle / bounds were resolved by the pre-pass, occupancy comes from the board
            const uint32_t tcode = code + (uint32_t)action_delta(a);
            const bool wants = ok && a != 0 && !(rv4[k] & 0x4000u);
            // No branches in here: the body of the k loop is meant to be ONE basic block, so that the scheduler can
            // interleave the arithmetic of the four agents around the board accesses.  The target row is read
            // whether or not the agent wants to move (a blocked target may lie one row outside the board: inside
            // the allocation, ignored), the two board updates are predicated shared-memory reductions.
            const uint32_t tb = 1u << (tcode & 31u);
            const uint32_t tv = occ[(tcode >> 5) * 32];
            const bool moves = wants & ((tv & tb) == 0u);
            atomicAnd(&occ[(code >> 5) * 32], moves ? ~(1u << (code & 31u)) : 0xFFFFFFFFu);   // neutral when the agent stays
            atomicOr(&occ[(tcode >> 5) * 32], moves ? tb : 0u);
            const bool failed = ok && a != 0 && !moves;  // ENV:583
            moved_m |= moves ? bit : 0u;
            failed_m |= failed ? bit : 0u;
            code = moves ? tcode : code;
            // ENV:538-563.  A lifelong arrival gets its new goal after the walk, in agent order.
            const bool on_goal = ok && code == gcode;
            bool gstep = false, cur_on_goal = on_goal;
            if (!kLifelong) {
                if (on_goal && !(reached_m & bit)) { reached_m |= bit; completed_m |= bit; gstep = true; }
            } else if (on_goal) {
                gstep = true;
                completed_m |= bit; reached_m &= ~bit;
                cur_on_goal = false;   // ENV:555
            }
            gstep_m |= gstep ? bit : 0u;
            ongoal_m |= cur_on_goal ? bit : 0u;
            // ENV:581-594 lock history
            uint32_t delta16 = 0;
            if (kLock) {
                const bool prev_on_goal = kLifelong ? false : (ocode == gcode);
                const bool gp = kLifelong ? gstep : (!prev_on_goal && cur_on_goal);
                const uint32_t g2 = (qget(gpq, k) << 1) | (gp ? 1u : 0u);
                const uint32_t m2 = (qget(mvq, k) << 1) | (moves ? 1u : 0u);
                const uint32_t f2 = (qget(fmq, k) << 1) | (failed ? 1u : 0u);
                qset(gpq, k, g2); qset(mvq, k, m2); qset(fmq, k, f2);
                const uint32_t okbit = ok ? bit : 0u;
                Gd |= (g2 & mdw) ? okbit : 0u;
                Md |= (m2 & mdw) ? okbit : 0u;
                Fd |= (f2 & mdw) ? okbit : 0u;
                Gl |= (g2 & mlw) ? okbit : 0u;
                Ml |= (m2 & mlw) ? okbit : 0u;
                const int dist = abs((int)(gcode >> 5) - (int)(code >> 5)) + abs((int)(gcode & 31u) - (int)(code & 31u));
                ds[k] = (uint32_t)dist;
                delta16 = (use_ring && ok) ? (uint32_t)((int)(int16_t)hget(ringq, k) - dist) << 16 : 0u;
            }
            rec[(i0 + k) * 32] = code | (rv4[k] & 0x7800u) | delta16;
            cd[k] = code;
            gc[k] = gcode;
            // ---------------------------------------------------- window rows of agent i on the boards as they are now
            const int r = (int)(code >> 5), c = (int)(code & 31u);
            const WB obst = lut_ld<WB>(lut_s + code * (uint32_t)sizeof(WB));
            const int sa = c > SR ? c - SR : 0, sb2 = (c < SR ? SR - c : 0) + 2;   // window columns start at c - SR
            const uint32_t *orow = &occ[(r - SR) * 32];
            const uint32_t grow_s = goalb_s + (uint32_t)((r - SR) * 128);
            uint32_t blk_up = 0, blk_mid = 0, blk_dn = 0;
#pragma unroll
            for (int wr = 0; wr < V; ++wr) {
                // rows outside the map read neighbouring shared memory: masked by the obstacle plane
                const uint32_t bx = orow[wr * 32];
                const uint32_t by = lds_pure(grow_s + (uint32_t)(wr * 128), (uint32_t)tile);   // goals do not change inside the walk
                const uint32_t o4 = (wr * V >= 2 ? (uint32_t)(obst >> (wr * V - 2)) : (uint32_t)(obst << 2)) & M4;
                const uint32_t MC = (wr == SR) ? (M4 & ~(4u << SR)) : M4;   // my own cell is not "another agent" (ENV:737)
                const uint32_t occ4 = ((bx >> sa) << sb2) & MC;
                const uint32_t agent4 = occ4 & ~o4;
                const uint32_t blk4 = occ4 | o4;
                const uint32_t g4 = ((by >> sa) << sb2) & M4 & ~blk4;
                if (wr == SR - 1) blk_up = blk4;
                if (wr == SR) blk_mid = blk4;
                if (wr == SR + 1) blk_dn = blk4;
                // plane 0 = obstacle | other's goal, plane 1 = other agent | other's goal (the three sets are disjoint,
                // ENV:730-745): spread(plane 0) + 2 * spread(plane 1) is the nibble row with codes 1 / 2 / 3, and the
                // nibble -> byte PRMT of phase B maps 3 to OTHER_GOAL (4).  t1 has one word per bank for V <= 5: lanes that
                // share a bank share the address, so these data-dependent look-ups never conflict (a single 4^V-entry
                // table would: ~3.5 wavefronts per access, measured).  The loads are free to float down to phase B.
                win[k][wr] = lds_pure(t1_s + (o4 | g4)) + (lds_pure(t1_s + (agent4 | g4)) << 1);
            }
            // ENV:761-771: a direction is valid iff its neighbour is neither obstacle nor agent
            const uint32_t am = 1u | ((~blk_up >> (2 + SR)) & 1u) << 1 | ((~blk_mid >> (2 + SR + 1)) & 1u) << 2 |
                                ((~blk_dn >> (2 + SR)) & 1u) << 3 | ((~blk_mid >> (2 + SR - 1)) & 1u) << 4;
            masks4 |= am << (8 * k);
            // own goal (code 3): the goal plane wrote 4 there; patched after the quad's words are stored
            {
                const int dr = (int)(gcode >> 5) - r + SR, dc = (int)(gcode & 31u) - c + SR;
                const bool in = (unsigned)dr < (unsigned)V && (unsigned)dc < (unsigned)V;
                const int ci = in ? dr * V + dc : 0;
                const bool occ_other = (ci != CTR) && ((occ[(gcode >> 5) * 32] >> (gcode & 31u)) & 1u);
                // byte 4 * V2 + 20 of the stage row is padding: the harmless target of a patch that does not apply
                patch[k] = (in && !((obst >> ci) & 1) && !occ_other) ? V2 * k + ci : 4 * V2 + 20;
            }
            {   // both samplers, selected afterwards (stored only when the sampler is fused in)
                const uint32_t x = qget(rnd, k);
                const uint32_t na_masked = lds_pure_u8(kth_s + am * 8u + __umulhi(x, (uint32_t)__popc(am)));
                const uint32_t na = masked_sampler ? na_masked : __umulhi(x, 5u);
                next4 |= na << (8 * k);
            }
        }
        stq32<VEC>(p.positions, ab + i0, i0, N, ok,
                   make_uint4(packed_of(cd[0]), packed_of(cd[1]), packed_of(cd[2]), packed_of(cd[3])));
        if (kLock) {
            stq32<VEC>(p.lock_gp, ab + i0, i0, N, ok, gpq);
            stq32<VEC>(p.lock_mv, ab + i0, i0, N, ok, mvq);
            stq32<VEC>(p.lock_fm, ab + i0, i0, N, ok, fmq);
            stq16<VEC>(p.lock_dist, ((size_t)(ok ? env : 0) * p.lw + slot_new) * N + i0, i0, N, ok,
                       make_uint2(ds[0] | (ds[1] << 16), ds[2] | (ds[3] << 16)));
        }
        if (q + 1 < NQ) load_lock(i0 + 4);
        // Phase B -- the byte rows of the four agents into my stage row (the table look-ups feeding it were issued in
        // phase A and, being loads from immutable tables, are free to complete anywhere in between).
        uint32_t carry = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!VEC && i0 + k >= N) continue;
            uint32_t acc[(4 * (V2 + 3) + 31) / 32 + 1];
#pragma unroll
            for (int j = 0; j < (int)(sizeof(acc) / sizeof(acc[0])); ++j) acc[j] = 0;
#pragma unroll
            for (int wr = 0; wr < V; ++wr) {
                const uint32_t t = win[k][wr];
                const int bitpos = 4 * (V * wr + (k & 3));  // agent k's bytes start k bytes into its first stage word
                const int wi = bitpos >> 5, sh = bitpos & 31;
                acc[wi] |= t << sh;
                if (sh + 4 * V > 32) acc[wi + 1] |= t >> (32 - sh);
            }
            // words of this agent: first word index (V2 * k) / 4; its k leading bytes belong to agent k-1
            constexpr int NWMAX = (V2 + 3 + 3) / 4;
            const int j0 = (V2 * k) >> 2;
            const int nw = ((k & 3) + V2 + 3) >> 2;
#pragma unroll
            for (int m = 0; m < NWMAX; ++m) {
                if (m >= nw) continue;
                uint32_t w = nibbles_to_bytes_0124((m & 1) ? (acc[m >> 1] >> 16) : acc[m >> 1]);
                if (m == 0 && (k & 3) != 0) w |= carry;                                  // leading partial word shared with agent k-1
                if (m == nw - 1 && (((k & 3) + V2) & 3) != 0) carry = w;                 // trailing partial word: stored by agent k+1
                else sts_stage(my_stage_s + (uint32_t)((j0 + m) * 4), w);   // lanes beyond the batch fill rows nobody flushes
            }
            if (!VEC && i0 + k == N - 1 && (((k & 3) + V2) & 3) != 0) sts_stage(my_stage_s + (uint32_t)((j0 + nw - 1) * 4), carry);
        }
        {
#pragma unroll
            for (int k = 0; k < 4; ++k) sts_stage_u8(my_stage_s + (uint32_t)patch[k], 3u);
            // action masks of the quad: 4 x 5 bytes = 5 words after the observation words
            uint32_t lo[4], hi[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t m = (masks4 >> (8 * k)) & 0x1Fu;
                lo[k] = spread4(m);
                hi[k] = m >> 4;
            }
            my_stage[OBS_W + 0] = lo[0];
            my_stage[OBS_W + 1] = hi[0] | (lo[1] << 8);
            my_stage[OBS_W + 2] = (lo[1] >> 24) | (hi[1] << 8) | (lo[2] << 16);
            my_stage[OBS_W + 3] = (lo[2] >> 16) | (hi[2] << 16) | (lo[3] << 24);
            my_stage[OBS_W + 4] = (lo[3] >> 8) | (hi[3] << 24);
        }
        if (ok) {
            if (p.o_goal_delta) {
                float2 gd[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {   // ENV:330-335
                    const int gi0 = (int)(gc[k] >> 5) - (int)(cd[k] >> 5) + (R - 1);
                    const int gi1 = (int)(gc[k] & 31u) - (int)(cd[k] & 31u) + (C - 1) + 2 * R - 1;
                    gd[k] = (VEC || i0 + k < N) ? make_float2(gdt[gi0], gdt[gi1]) : make_float2(0.f, 0.f);
                }
                if (VEC) {   // one 256-bit store per quad (sm_100 STG.256): half the L1 tag look-ups of two 128-bit stores
                    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p.o_goal_delta + ab + oo + i0),
                                 "f"(gd[0].x), "f"(gd[0].y), "f"(gd[1].x), "f"(gd[1].y), "f"(gd[2].x), "f"(gd[2].y),
                                 "f"(gd[3].x), "f"(gd[3].y) : "memory");
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) if (i0 + k < N) p.o_goal_delta[ab + oo + i0 + k] = gd[k];
                }
            }
            if (p.o_blocking_prev) stq8<VEC>(p.o_blocking_prev, ab + oo + i0, i0, N, true, spread4(bprev_m >> i0));
            if (p.sample_mode) stq8<VEC>(reinterpret_cast<uint8_t *>(p.o_next_actions), ab + i0, i0, N, true, next4);
        }
        // ------------------------------------------------ coalesced flush of the stage rows (one per lane)
        // row `e` holds quad q of env env0 + e: agent index (env0 + e) * N + 4 * q
        __syncwarp();
        if (VEC) {
            const size_t agent0 = env0 * N + oo + (size_t)i0;
            for (int w = lane; w < OBS_W + 5; w += 32) {
                const bool is_obs = w < OBS_W;
                unsigned char *gp = is_obs ? (p.o_local_obs ? p.o_local_obs + agent0 * V2 + 4 * w : nullptr)
                                           : (p.o_action_mask ? reinterpret_cast<unsigned char *>(p.o_action_mask) +
                                                                    agent0 * 5 + 4 * (w - OBS_W) : nullptr);
                const uint32_t gstride = (uint32_t)N * (uint32_t)(is_obs ? V2 : 5);
                const uint32_t *src = stage_w + w;
                if (gp) {
                    if (act_w == full) {
#pragma unroll
                        for (int e = 0; e < 32; ++e)
                            *reinterpret_cast<uint32_t *>(gp + (size_t)e * gstride) = src[e * STRIDE];
                    } else {
#pragma unroll 1
                        for (int e = 0; e < 32; ++e)
                            if ((act_w >> e) & 1u)
                                *reinterpret_cast<uint32_t *>(gp + (size_t)e * gstride) = src[e * STRIDE];
                    }
                }
            }
        } else {
            const int na = (N - i0) < 4 ? (N - i0) : 4;
            for (int e = 0; e < 32; ++e) {
                if (!((act_w >> e) & 1u)) continue;
                const uint8_t *src = reinterpret_cast<const uint8_t *>(stage_w + e * STRIDE);
                if (p.o_local_obs) {
                    uint8_t *dst = p.o_local_obs + ((env0 + e) * N + oo + i0) * V2;
                    for (int b = lane; b < na * V2; b += 32) dst[b] = src[b];
                }
                if (p.o_action_mask) {
                    uint8_t *dst = reinterpret_cast<uint8_t *>(p.o_action_mask) + ((env0 + e) * N + oo + i0) * 5;
                    for (int b = lane; b < na * 5; b += 32) dst[b] = src[4 * OBS_W + b];
                }
            }
        }
        __syncwarp();
    }

    // ---------------------------------------------------------------- the rest of the env words: needed behind the epilogue
    // Copied global -> shared with cp.async: no registers held while in flight (a row loaded into registers during the
    // walk stays live through every quad and spills).  16 bytes k of my env's row at ew_s + 512 k: a slot in the stage, which is
    // dead from here -- the __syncwarp closing the last flush says every lane has drained it -- to the next step's phase
    // B, behind the __syncwarp that ends this step.  Only this lane touches its slot, after its own wait.
    const uint32_t ew_s = (uint32_t)__cvta_generic_to_shared(stage_w) + (uint32_t)lane * 16u;
    {
        const int4 *src = p.env_words + (size_t)(ok ? env : 0) * 4;
#pragma unroll
        for (int k = 0; k < 4; ++k)   // lanes beyond the batch land zeros, as the register loads they replace left them
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(ew_s + 512u * k), "l"(src + k),
                         "r"(ok ? 16 : 0) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    int *ew_slot = reinterpret_cast<int *>(stage_w) + lane * 4;   // word w at ew_slot[128 * (w >> 2) + (w & 3)]
    auto ew_ld = [&](int word) -> int { return ew_slot[128 * (word >> 2) + (word & 3)]; };

    // ---------------------------------------------------------------- injected co-location (ENV:658-666), kept off the walk
    // Replays who owns which cell through the moves of this step (ENV:523: a leaving agent clears the owner for
    // everybody on its cell; ENV:525: a mover owns its new cell) and marks OTHER_AGENT in the centre of the window
    // of every agent that stood on a cell owned by somebody else when its observation was taken (ENV:737-739).
    if (__any_sync(full, degen)) {
        __syncwarp();   // the flush above wrote those windows
        if (degen && ok) {
            for (int i = 0; i < N; ++i) {
                const uint32_t rvi = rec[i * 32], newc = rvi & REC_CODE, biti = 1u << i;
                const bool mvd = (moved_m >> i) & 1u;
                const uint32_t oldc = mvd ? newc - (uint32_t)action_delta((rvi >> 11) & 7u) : newc;
                bool owned_by_other = false;
                for (int a2 = 0; a2 < N; ++a2) {
                    if (a2 == i) continue;
                    const uint32_t rva = rec[a2 * 32];
                    uint32_t ca = rva & REC_CODE;   // where a2 stands at agent i's turn: moved already only if a2 < i
                    if (a2 > i && ((moved_m >> a2) & 1u)) ca -= (uint32_t)action_delta((rva >> 11) & 7u);
                    if (ca == oldc) {
                        if (mvd) solo_m &= ~(1u << a2);                       // ENV:523
                        else if ((solo_m >> a2) & 1u) owned_by_other = true;  // the cell has an owner, and it is not me
                    }
                }
                if (mvd) solo_m |= biti;                                       // ENV:525
                else if (!(solo_m & biti) && owned_by_other && p.o_local_obs)
                    p.o_local_obs[(ab + oo + i) * V2 + CTR] = 2;
            }
        }
        __syncwarp();
    }

    // ---------------------------------------------------------------- lifelong goal reassignment (ENV:284-304, 547-556)
    if (kLock) lock_head = slot_next;
    const int arrivals = __popc(gstep_m);
    const uint32_t pend = kLifelong ? gstep_m : 0u;
    const bool reassigned = pend != 0;
    {
        // An arrival is rare per env (once in a few hundred steps) but not per warp of 32 envs, and the kernel is
        // one wave: the slowest warp sets the launch time.  So the WARP serves each of its reassigned envs
        // together -- lane = agent for the roll-back / re-emission, lane = map row for the candidate scan --
        // instead of 32 lanes re-walking their own env for the sake of one.
        unsigned rw = __ballot_sync(full, pend != 0);
        // the Philox counters of the envs served here come from the env-word slots (each lane reads and updates its own)
        if (rw) asm volatile("cp.async.wait_all;" ::: "memory");
        const uint32_t rng_counter0 = rw ? (uint32_t)ew_ld(MAPF_W_RNG_COUNTER) : 0u;
        while (rw) {
            const int e = __ffs(rw) - 1;
            rw &= rw - 1;
            uint32_t pe = __shfl_sync(full, pend, e);
            const uint32_t mv_e = __shfl_sync(full, moved_m, e), bp_e = __shfl_sync(full, bprev_m, e);
            const uint32_t solo_e = __shfl_sync(full, degen ? solo_m : 0xFFFFFFFFu, e);
            const uint32_t rc_e = __shfl_sync(full, rng_counter0, e);
            const int slot_new_e = __shfl_sync(full, slot_new, e), slot_next_e = __shfl_sync(full, slot_next, e);
            const bool use_ring_e = __shfl_sync(full, (int)use_ring, e) != 0;
            const long long eg = p.env_id_base + (long long)(env0 + e);
            const size_t abe = (env0 + e) * (size_t)N, enve = env0 + e;
            uint32_t *occ_e = occ_w + e, *goal_e = goal_w + e, *rec_e = rec_w + e;
            uint32_t rng_inc = 0, err_e = 0, ongoal_fix = 0;
            while (pe) {   // arrivals in agent order (ENV:284-304)
                const int i = __ffs(pe) - 1;
                pe &= pe - 1;
                // roll the env's occupancy board back to snapshot i: later movers leave their new cell, then re-take the old one
                const uint32_t later = mv_e & ~((2u << i) - 1u);
                const bool und = lane < N && ((later >> lane) & 1u);
                uint32_t nc = 0, oc = 0;
                if (und) {
                    const uint32_t rv = rec_e[lane * 32];
                    nc = rv & REC_CODE;
                    oc = nc - (uint32_t)action_delta((rv >> 11) & 7u);
                    atomicAnd(&occ_e[(nc >> 5) * 32], ~(1u << (nc & 31u)));
                }
                const uint32_t gold = code_of(p.goals[abe + i]);
                if (lane == 0) goal_e[(gold >> 5) * 32] &= ~(1u << (gold & 31u));   // ENV:288
                __syncwarp();
                if (und) atomicOr(&occ_e[(oc >> 5) * 32], 1u << (oc & 31u));
                __syncwarp();
                uint32_t ng = 0xFFFFFFFFu;
                if (p.goal_override) {
                    const uint32_t ov = p.goal_override[abe + i];
                    if (prow(ov) >= 0) ng = code_of(ov);
                }
                if (ng == 0xFFFFFFFFu) {   // candidates = free, unoccupied, nobody's goal; rows lane and lane + 32
                    const uint32_t c0 = lane < R ? (freerow[lane] & ~occ_e[lane * 32] & ~goal_e[lane * 32]) : 0u;
                    const uint32_t c1 = lane + 32 < R ? (freerow[lane + 32] & ~occ_e[(lane + 32) * 32] & ~goal_e[(lane + 32) * 32]) : 0u;
                    const int n0 = __popc(c0), n1 = __popc(c1);
                    int pre0 = n0, pre1 = n1;   // inclusive prefix sums over the lanes
#pragma unroll
                    for (int sft = 1; sft < 32; sft <<= 1) {
                        const int v0 = __shfl_up_sync(full, pre0, sft), v1 = __shfl_up_sync(full, pre1, sft);
                        if (lane >= sft) { pre0 += v0; pre1 += v1; }
                    }
                    const int tot0 = __shfl_sync(full, pre0, 31), n = tot0 + __shfl_sync(full, pre1, 31);
                    int kk = -1;
                    if (p.goal_rank) kk = p.goal_rank[abe + i];
                    if (kk < 0 && n > 0) {
                        const Philox ph(p.seed, eg);
                        const uint4 x = ph(rc_e + rng_inc, (uint32_t)i, 0x474F414Cu /* "GOAL" */, 0);
                        kk = (int)__umulhi(x.x, (uint32_t)n);
                        rng_inc++;
                    }
                    if (n > 0 && kk < n) {   // row-major order: rows 0..31, then 32..63
                        const bool hit0 = kk >= pre0 - n0 && kk < pre0;
                        const bool hit1 = kk >= tot0 + pre1 - n1 && kk < tot0 + pre1;
                        uint32_t mine = 0;
                        if (hit0) mine = (uint32_t)(lane * 32) + __fns(c0, 0, kk - (pre0 - n0) + 1);
                        if (hit1) mine = (uint32_t)((lane + 32) * 32) + __fns(c1, 0, kk - tot0 - (pre1 - n1) + 1);
                        const unsigned hb = __ballot_sync(full, hit0 || hit1);
                        ng = __shfl_sync(full, mine, __ffs(hb) - 1);
                    } else {
                        err_e |= MAPF_DEV_ERR_NO_GOAL_CELL;
                    }
                }
                if (ng == 0xFFFFFFFFu) { ng = gold; ongoal_fix |= 1u << i; }   // no cell: the old goal stays, the agent is on it
                if (lane == 0) {
                    goal_e[(ng >> 5) * 32] |= 1u << (ng & 31u);
                    p.goals[abe + i] = packed_of(ng);
                    if (kLock) {   // ENV:591: distance to the NEW goal
                        const uint32_t rv = rec_e[i * 32], code = rv & REC_CODE;
                        const int dist = abs((int)(ng >> 5) - (int)(code >> 5)) + abs((int)(ng & 31u) - (int)(code & 31u));
                        p.lock_dist[((size_t)enve * p.lw + slot_new_e) * N + i] = (int16_t)dist;
                        if (use_ring_e) {
                            const int ring_old = (int)p.lock_dist[((size_t)enve * p.lw + slot_next_e) * N + i];
                            rec_e[i * 32] = (rv & 0xFFFFu) | ((uint32_t)(ring_old - dist) << 16);
                        }
                    }
                }
                // roll forward again
                if (und) atomicAnd(&occ_e[(oc >> 5) * 32], ~(1u << (oc & 31u)));
                __syncwarp();
                if (und) atomicOr(&occ_e[(nc >> 5) * 32], 1u << (nc & 31u));
                __syncwarp();
            }
            // ENV:565-575: everybody of this env shows the final state; lane = agent
            {
                const uint32_t code = lane < N ? (rec_e[lane * 32] & REC_CODE) : 0u;
                const uint32_t gcode = lane < N ? code_of(p.goals[abe + lane]) : 0u;
                const bool ctr2 = !((solo_e >> lane) & 1u) && ((occ_e[(code >> 5) * 32] >> (code & 31u)) & 1u);
                emit_final(abe, oo, sctr, eg, occ_e, goal_e, code, gcode, (bp_e >> lane) & 1u, ctr2);
            }
            if (lane == e) {
                ew_slot[128 * (MAPF_W_RNG_COUNTER >> 2) + (MAPF_W_RNG_COUNTER & 3)] = (int)(rc_e + rng_inc);
                errs |= err_e; ongoal_m |= ongoal_fix;
            }
            __syncwarp();
        }
    }

    // ---------------------------------------------------------------- epilogue: owner masks, locks, blocking, wait-for graph
    // The boards are dead: rowm[r + PADR] / colm[c + PADR] get bit a for agent a's final row / column
    // (PADR zero rows on both sides).
    __syncwarp();
    // PK (the FAST instantiation, N <= 16): both masks share one word -- low half rows, high half columns -- in the goal
    // board's memory, and the occupancy board stays alive for a cheap pre-test: an agent with nobody within Manhattan
    // distance 2 on the final board and no failed move has nothing to do below (no neighbour set, no owner to look
    // up), and that is most agents -- the loop then runs over the few that do, not over all N.
    constexpr bool PK = FAST;
    uint32_t todo = ok ? allN : 0u;
    if (PK) {
        for (int r = 0; r < E.board_rows; ++r) goalb[r * 32] = 0u;
        uint32_t near_m = 0;
        if (ok) {
#pragma unroll 1
            for (int i = 0; i < N; ++i) {
                const uint32_t code = rec[i * 32] & REC_CODE;
                const int r = (int)(code >> 5);
                atomicOr(&goalb[(r + PADR) * 32], 1u << i);
                atomicOr(&goalb[((code & 31u) + PADR) * 32], 0x10000u << i);
                // rows above the map read neighbouring shared memory: a false "near" costs a look below, never a result
                const uint32_t *orow = &occ[(r - 2) * 32];
                const uint32_t b = 1u << (code & 31u);
                const uint32_t m1 = (b << 1) | (b >> 1), mB = m1 | b, mA = m1 | (b << 2) | (b >> 2);
                const uint32_t nr = (orow[64] & mA) | ((orow[32] | orow[96]) & mB) | ((orow[0] | orow[128]) & b);
                near_m |= nr ? (1u << i) : 0u;
            }
        }
        todo = (p.nearby == 2 && !degen && reached_m == 0u) ? (near_m | failed_m) & todo : todo;
    } else {
        for (int r = 0; r < E.board_rows; ++r) { occ[r * 32] = 0u; goalb[r * 32] = 0u; }
        if (ok) {
#pragma unroll 1
            for (int i = 0; i < N; ++i) {
                const uint32_t code = rec[i * 32] & REC_CODE;
                atomicOr(&rowm[((code >> 5) + PADR) * 32], 1u << i);   // reductions without a return value: no dependent chain
                atomicOr(&colm[((code & 31u) + PADR) * 32], 1u << i);
            }
        }
    }
    // agents of row / column idx (idx already padded)
    auto rowset = [&](int idx) -> uint32_t { return PK ? (goalb[idx * 32] & 0xFFFFu) : rowm[idx * 32]; };
    auto colset = [&](int idx) -> uint32_t { return PK ? (goalb[idx * 32] >> 16) : colm[idx * 32]; };
    uint32_t coloc_any = 0, wf_alive = 0, flags_any = 0;   // flags_any: bit 0 deadlock, bit 1 livelock participant set found
    uint32_t wf_m = 0, blocking_m = 0;
    const uint32_t intent_m = allN & ~reached_m;  // ENV:619-621: only agents that have not (sticky-)reached press
    // a rolled loop on purpose: the launch is one pass over the code per warp, the instruction cache is a
    // contended resource (stall_no_inst was 18 % with this loop unrolled by four)
#pragma unroll 1
    while (todo) {
        const int i = __ffs(todo) - 1;
        todo &= todo - 1;
        const uint32_t bit = 1u << i;
        const uint32_t rv = rec[i * 32];
        const uint32_t code = rv & REC_CODE;
        const int r = (int)(code >> 5), c = (int)(code & 31u);
        const int pr = r + PADR, pc = c + PADR;
        const uint32_t row0 = rowset(pr), col0 = colset(pc);
        const uint32_t here = row0 & col0;   // agents on my cell (me included)
        if (here & ~bit) coloc_any |= bit;
        // ENV:389-438 neighbours within Manhattan distance `nearby`, via the row / column masks
        if (kLock && !(ongoal_m & bit)) {
            uint32_t nb = 0;
            if (p.nearby == 2) {
                const uint32_t c1 = col0 | colset(pc - 1) | colset(pc + 1);
                const uint32_t c2 = c1 | colset(pc - 2) | colset(pc + 2);
                nb = (row0 & c2) | ((rowset(pr - 1) | rowset(pr + 1)) & c1) | ((rowset(pr - 2) | rowset(pr + 2)) & col0);
            } else {
                uint32_t u = 0;
                for (int w = 0; w <= p.nearby; ++w) {
                    const int dd = p.nearby - w;
                    if (c - w >= 0) u |= colset(pc - w);
                    if (c + w < C) u |= colset(pc + w);
                    uint32_t rm = 0;
                    if (r - dd >= 0) rm |= rowset(pr - dd);
                    if (r + dd < R) rm |= rowset(pr + dd);
                    nb |= rm & u;
                }
            }
            nb &= ~here;
            if (__popc(nb) >= p.min_nb) {
                const uint32_t P = nb | bit;
                if (!(P & Gd) && !(P & Md) && (P & Fd)) flags_any |= 1u;
                if (!(P & Gl) && (P & Ml)) {
                    uint32_t rest = nb;
                    int red = (int)rv >> 16;
                    while (rest) {
                        const int a = __ffs(rest) - 1;
                        rest &= rest - 1;
                        red += (int)rec[a * 32] >> 16;
                    }
                    if (red <= p.eps_floor) flags_any |= 2u;
                }
            }
        }
        // intended cell (kept even when invalid, ENV:514-515) -> who stands there.  A blocked target is an
        // obstacle or out of bounds: nobody can stand there.
        // (needed for ENV:609-623 only while some agent has sticky-reached -- never in lifelong mode -- and for the
        // wait-for edge of an agent whose move failed)
        uint32_t owner = here & ~bit;
        if (!(moved_m & bit)) {
            owner = 0;
            if (!(rv & 0x4000u) && (reached_m != 0u || (failed_m & bit))) {
                const uint32_t tcode = code + (uint32_t)action_delta((rv >> 11) & 7u);
                owner = rowset((int)(tcode >> 5) + PADR) & colset((int)(tcode & 31u) + PADR) & ~bit;
            }
        }
        if (intent_m & bit) blocking_m |= owner;   // ENV:609-623 (filtered below)
        if ((failed_m & bit) && owner) {   // wait-for edge i -> owner (kept in the action bits of the record)
            rec[i * 32] = (rv & ~0xF800u) | ((uint32_t)(31 - __clz(owner)) << 11);
            wf_alive |= bit;
        }
    }
    const bool dl_any = flags_any & 1u, ll_any = (flags_any & 2u) != 0;
    blocking_m &= reached_m & ~moved_m;
    // wait-for cycles: strip agents whose target is gone or that nobody waits for, until stable
    if (__any_sync(full, wf_alive != 0)) {
        uint32_t alive = wf_alive;
        for (;;) {
            uint32_t keep = 0, targets = 0, rest = alive;
            while (rest) {
                const int i = __ffs(rest) - 1;
                rest &= rest - 1;
                const uint32_t t = (rec[i * 32] >> 11) & 31u;
                if ((alive >> t) & 1u) { keep |= 1u << i; targets |= 1u << t; }
            }
            keep &= targets;
            const bool changed = keep != alive;
            alive = keep;
            if (!__any_sync(full, changed)) break;
        }
        wf_m = alive;
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    int step_count = ew_ld(MAPF_W_STEP_COUNT) + 1;  // ENV:475
    int lock_prev = ew_ld(MAPF_W_LOCK_PREV);
    int goals_total = ew_ld(MAPF_W_GOALS_TOTAL) + arrivals;  // lifelong: every arrival; else first arrivals (ENV:545,562)
    int blocking_total = ew_ld(MAPF_W_BLOCKING_TOTAL), dl_events = ew_ld(MAPF_W_DEADLOCK_EVENTS);
    int ll_events = ew_ld(MAPF_W_LIVELOCK_EVENTS), dl_steps = ew_ld(MAPF_W_DEADLOCK_STEPS);
    int ll_steps = ew_ld(MAPF_W_LIVELOCK_STEPS);
    uint32_t rng_counter = (uint32_t)ew_ld(MAPF_W_RNG_COUNTER);
    int ep_return_x2 = ew_ld(MAPF_W_EPISODE_RETURN_X2), wfg_steps = ew_ld(MAPF_W_WFG_CYCLE_STEPS);
    int episodes = ew_ld(MAPF_W_EPISODES);
    const bool wf_any = wf_m != 0;
    wfg_steps += wf_any;
    const int blocking_step = __popc(blocking_m);
    blocking_total += blocking_step;

    // ---------------------------------------------------------------- lock detection result, ENV:595-606
    bool dl_step = false, ll_step = false, dl_event = false, ll_event = false;
    if (kLock) {
        dl_step = count_after >= p.dw && dl_any;
        ll_step = !dl_step && count_after >= p.lw && ll_any;
        dl_event = dl_step && !(lock_prev & 1);
        ll_event = ll_step && !(lock_prev & 2);
        lock_prev = (dl_step ? 1 : 0) | (ll_step ? 2 : 0);
        dl_steps += dl_step; ll_steps += ll_step; dl_events += dl_event; ll_events += ll_event;
        lock_count = count_after;
    }

    // ---------------------------------------------------------------- rewards & termination, ENV:658-690
    bool terminated = false, truncated = false;
    const uint32_t scratch_on = kLifelong ? 0u : ongoal_m;   // reached_goal scratch (ENV:555)
    uint32_t bonus_m = 0, penalty_m = 0;
    if (!kLifelong && __popc(scratch_on) == N) { terminated = true; bonus_m = allN; }
    else if (step_count >= p.steps_per_episode) {
        terminated = true; truncated = true;  // F6
        if (!kLifelong) penalty_m = allN & ~scratch_on;
    }
    const bool done = ok && (terminated || truncated);
    int rsum = __popc(gstep_m) + 2 * __popc(bonus_m) - 2 * __popc(penalty_m);
    uint32_t coloc_pairs2 = 0;   // 2 * (co-located others), summed over my agents
    for (int q = 0; q < NQ; ++q) {
        const int i0 = 4 * q;
        const uint32_t gs = spread4(gstep_m >> i0), bl = spread4(blocking_m >> i0);
        const uint32_t asf4 = spread4(moved_m >> i0) * MAPF_ASF_MOVED + spread4(failed_m >> i0) * MAPF_ASF_FAILED_MOVE +
                              gs * MAPF_ASF_GOAL_REACHED + bl * MAPF_ASF_BLOCKING +
                              spread4(wf_m >> i0) * MAPF_ASF_WFG_CYCLE + spread4(ongoal_m >> i0) * MAPF_ASF_ON_GOAL;
        uint32_t af4 = spread4(reached_m >> i0) * MAPF_AF_REACHED + spread4(completed_m >> i0) * MAPF_AF_COMPLETED_ONCE +
                       bl * MAPF_AF_BLOCKING_PREV;
        if (degen) af4 += spread4(~solo_m >> i0) * MAPF_AF_NOT_OWNER;   // the owner grid outlives the step (ENV:102)
        // reward * 2 per agent (exact small integers): +1 arrival, +2 all-on-goal bonus, -2 truncation penalty
        const uint32_t pos4 = gs + 2u * spread4(bonus_m >> i0), neg4 = 2u * spread4(penalty_m >> i0);
        float rw[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int rx2 = (int)((pos4 >> (8 * k)) & 0xFFu) - (int)((neg4 >> (8 * k)) & 0xFFu);
            if ((coloc_any >> (i0 + k)) & 1u) {   // ENV:658-666, -1 per co-located pair member (injected states only)
                const uint32_t code = rec[(i0 + k) * 32] & REC_CODE;
                const int others = __popc(rowset((int)(code >> 5) + PADR) & colset((int)(code & 31u) + PADR)) - 1;
                rx2 -= 2 * others;
                coloc_pairs2 += 2u * (uint32_t)others;
            }
            rw[k] = 0.5f * (float)rx2;
        }
        if (ok) {
            if (p.o_reward) {
                if (VEC) *reinterpret_cast<float4 *>(p.o_reward + ab + oo + i0) = make_float4(rw[0], rw[1], rw[2], rw[3]);
                else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) if (i0 + k < N) p.o_reward[ab + oo + i0 + k] = rw[k];
                }
            }
            if (p.o_agent_step_flags) stq8<VEC>(p.o_agent_step_flags, ab + oo + i0, i0, N, true, asf4);
            stq8<VEC>(p.agent_flags, ab + i0, i0, N, true, af4);
        }
    }
    rsum -= (int)coloc_pairs2;
    ep_return_x2 += rsum;
    const int n_comp = __popc(completed_m), n_reach = __popc(reached_m);
    if (ok) {
        if (p.o_info) {  // integer sources of info["__all__"], ENV:639-656
            int4 *io = p.o_info + ((size_t)env + so) * 4;
            io[0] = make_int4(arrivals, kLifelong ? goals_total : n_reach, blocking_step, blocking_total);
            io[1] = make_int4(dl_step, ll_step, dl_event, ll_event);
            io[2] = make_int4(dl_events, ll_events, dl_steps, ll_steps);
            io[3] = make_int4(n_comp, step_count, n_reach, wfg_steps);
        }
        if (p.o_terminated) p.o_terminated[env + so] = terminated;
        if (p.o_truncated) p.o_truncated[env + so] = truncated;
        if (p.o_step_flags)
            p.o_step_flags[env + so] = (uint8_t)((terminated ? MAPF_SF_TERMINATED : 0) | (truncated ? MAPF_SF_TRUNCATED : 0) |
                                            (dl_step ? MAPF_SF_DEADLOCK_STEP : 0) | (ll_step ? MAPF_SF_LIVELOCK_STEP : 0) |
                                            (dl_event ? MAPF_SF_DEADLOCK_EVENT : 0) | (ll_event ? MAPF_SF_LIVELOCK_EVENT : 0) |
                                            (reassigned ? MAPF_SF_GOAL_REASSIGNED : 0) | (wf_any ? MAPF_SF_WFG_CYCLE : 0));
    }

    // ---------------------------------------------------------------- episode end: metrics, auto-reset
    if (done) {   // episode-end metric sums, src/trainers/callbacks.py:152,173,335-345
        double *m = p.env_metrics + (size_t)env * MAPF_METRIC_COUNT;
        const double gt = kLifelong ? (double)goals_total : (double)n_reach;  // ENV:630-633
        m[MAPF_M_EPISODES] += 1.0;
        m[MAPF_M_RETURN_SUM] += 0.5 * (double)ep_return_x2;
        m[MAPF_M_LENGTH_SUM] += (double)step_count;
        m[MAPF_M_SUCCESS_SUM] += (terminated && !truncated) ? 1.0 : 0.0;
        m[MAPF_M_GOALS_REACHED_SUM] += gt;
        m[MAPF_M_BLOCKING_COUNT_SUM] += (double)blocking_total;
        m[MAPF_M_DEADLOCK_COUNT_SUM] += (double)dl_events;
        m[MAPF_M_LIVELOCK_COUNT_SUM] += (double)ll_events;
        m[MAPF_M_DEADLOCK_STEPS_SUM] += (double)dl_steps;
        m[MAPF_M_LIVELOCK_STEPS_SUM] += (double)ll_steps;
        m[MAPF_M_THROUGHPUT_SUM] += gt / (double)(step_count > 1 ? step_count : 1);  // ENV:655
        m[MAPF_M_COMPLETION_RATIO_SUM] += (double)n_comp / (double)N;                 // ENV:638
        m[MAPF_M_WFG_CYCLE_STEPS_SUM] += (double)wfg_steps;
        episodes += 1;
    }
    // ENV:440-472 inside the launch (benchmark loop semantics: `if done: reset()`).  Like a goal reassignment an
    // episode end is rare per env and common per warp (in steady state 1 / steps_per_episode of the envs per step),
    // so the WARP resets each of its finished envs together, lane = agent: the layout draw (ENV:267-282) as
    // symmetric rejection with one Philox block per agent and round, the state rows, the boards of the new layout
    // and the first observation of the new episode (final state, no staggering at reset, ENV:459-468).
    unsigned rsw = __ballot_sync(full, done && p.auto_reset);
    if (rsw) {
        const int F = p.num_free[0];
        __syncwarp();
        while (rsw) {
            const int e = __ffs(rsw) - 1;
            rsw &= rsw - 1;
            const size_t enve = env0 + e, abe = enve * (size_t)N;
            const long long eg = p.env_id_base + (long long)enve;
            const uint32_t rc_e = __shfl_sync(full, rng_counter, e);
            uint32_t *occ_e = occ_w + e, *goal_e = goal_w + e, *rec_e = rec_w + e;
            const bool mine = lane < N;
            uint32_t rounds = 0, err_e = 0;
            bool sample = !p.deterministic;
            if (sample && F < 2 * N) { err_e |= MAPF_DEV_ERR_TOO_FEW_CELLS; sample = false; }
            uint32_t st = 0, gg = 0;   // cell codes of agent `lane`
            if (sample) {
                // every slot (starts 0..N-1, then goals) draws a uniform free cell; a slot equal to a lower-numbered
                // slot redraws in the next round (same rule and same Philox counters as draw_layout<G>)
                const Philox ph(p.seed, eg);
                int cs = -1 - lane, cg = -33 - lane;   // distinct placeholders for the lanes beyond N
                bool rs = mine, rgn = mine;
                while (__any_sync(full, rs || rgn)) {
                    if (rs || rgn) {
                        const uint4 x = ph(rc_e + rounds, (uint32_t)lane, 0x52455345u /* "RESE" */, 0);
                        if (rs) cs = kth_free((int)__umulhi(x.x, (uint32_t)F));
                        if (rgn) cg = kth_free((int)__umulhi(x.y, (uint32_t)F));
                    }
                    rs = false; rgn = false;
                    if (N <= 16) {
                        // all 2N slots side by side (starts in lanes 0..15, goals in lanes 16..31): one match tells every
                        // slot whether a lower-numbered one holds the same cell
                        const int gv = __shfl_sync(full, cg, (lane - 16) & 31);
                        const unsigned same = __match_any_sync(full, lane < 16 ? cs : gv);
                        const bool dupl = (same & ((1u << lane) - 1u)) != 0;
                        const bool dupg = __shfl_sync(full, (int)dupl, (lane + 16) & 31) != 0;
                        rs = mine && dupl;
                        rgn = mine && dupg;
                    } else {
                        for (int a = 0; a < N; ++a) {
                            const int os = __shfl_sync(full, cs, a), og = __shfl_sync(full, cg, a);
                            if (mine) {
                                if (a < lane && os == cs) rs = true;   // lower start slot
                                if (os == cg) rgn = true;              // every start slot is lower than a goal slot
                                if (a < lane && og == cg) rgn = true;  // lower goal slot
                            }
                        }
                    }
                    rounds++;
                }
                if (mine) {
                    st = (uint32_t)((cs / C) * 32 + cs % C);
                    gg = (uint32_t)((cg / C) * 32 + cg % C);
                }
            } else if (mine) {
                st = p.deterministic ? code_of(p.starts[abe + lane]) : (rec_e[lane * 32] & REC_CODE);   // F7: goals stay
                gg = code_of(p.goals[abe + lane]);
            }
            if (mine) {
                p.positions[abe + lane] = packed_of(st);
                if (sample) { p.starts[abe + lane] = packed_of(st); p.goals[abe + lane] = packed_of(gg); }
                p.agent_flags[abe + lane] = 0;
                if (kLock) { p.lock_gp[abe + lane] = 0u; p.lock_mv[abe + lane] = 0u; p.lock_fm[abe + lane] = 0u; }
            }
            // boards of the new layout
            for (int r = lane; r < E.board_rows; r += 32) { occ_e[r * 32] = 0u; goal_e[r * 32] = 0u; }
            __syncwarp();
            if (mine) {
                atomicOr(&occ_e[(st >> 5) * 32], 1u << (st & 31u));
                atomicOr(&goal_e[(gg >> 5) * 32], 1u << (gg & 31u));
            }
            __syncwarp();
            emit_final(abe, oo, sctr, eg, occ_e, goal_e, st, gg, 0u, false);
            if (lane == e) {
                rng_counter += rounds; errs |= err_e;
                step_count = 0; lock_count = 0; lock_head = 0; lock_prev = 0; goals_total = 0; blocking_total = 0;
                dl_events = ll_events = dl_steps = ll_steps = 0; ep_return_x2 = 0; wfg_steps = 0;
            }
            __syncwarp();
        }
    }

    // ---------------------------------------------------------------- env words write-back
    if (ok) {
        int4 *ew4 = p.env_words + (size_t)env * 4;
        ew4[0] = make_int4(step_count, lock_count, lock_prev, goals_total);
        ew4[1] = make_int4(blocking_total, dl_events, ll_events, dl_steps);
        ew4[2] = make_int4(ll_steps, (int)rng_counter, ep_return_x2, wfg_steps);
        ew4[3] = make_int4(episodes, lock_head, ew_ld(MAPF_W_RESERVED1), ew_ld(MAPF_W_RESERVED2));
    }
    __syncwarp();
    }  // inner steps
    }  // tile loop
    errs = __reduce_or_sync(full, errs);
    if (errs && lane == 0) atomicOr(p.err_bits, errs);
}

}  // namespace mapf
