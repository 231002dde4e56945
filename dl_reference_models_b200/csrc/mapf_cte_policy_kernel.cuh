// mapf_cte_policy_kernel.cuh -- the centralised (CTE) policy on the single-agent view's outputs, in ONE launch per
// step: obs_grid (the R*C grid codes of mapf_cte_kernel) -> Linear(R*C, 64)-ReLU-Linear(64, 64)-ReLU -> {5N logits,
// value} -> per agent a masked 5-way softmax and draw (RLlib's multi-categorical over MultiDiscrete([5] * N)).
// cte_rollout.CteActionMaskPolicy is the specification.
//
//   * a warp takes 32 envs (two m16 tiles); layer 1 is a K = R*C bf16 m16n8k16 mma.sync GEMM with f32 accumulation.
//     The grid codes are <= 2N + 1 <= 65, exact in bf16; a code byte b is turned into bf16(128 + b) by one byte
//     permute (0x4300 | b, b < 128) and 128 is subtracted exactly in bf16x2;
//   * W1 is resident in shared memory (bf16, row stride S1 = K padded to 32 (+32 when that is a multiple of 64):
//     conflict-free 128-bit fragment loads).  The grid bytes of the warp's 32 rows are staged per warp in chunks of
//     CTE_KC columns, double-buffered with cp.async (16-, 8- or 4-byte copies, the widest the row length and the
//     base address allow; byte loads for other shapes);
//   * inside a k32 block the lane of thread-in-group t holds the grid columns 8t .. 8t + 7 of its rows: columns
//     8t .. 8t + 3 are the k16 chunk 0 operand (k = 2t, 2t + 1, 2t + 8, 2t + 9), 8t + 4 .. 8t + 7 chunk 1's, so one
//     64-bit load gives a row's A operand of both chunks and one 128-bit load a W1 row's B operand of both;
//   * layer 2 is mapf_policy_act_kernel's (pol_layer2); the head is 5N + 1 columns (5N logits, then the value) in
//     n8 tiles, evaluated in groups of five tiles (40 columns = 8 agents) into a per-warp [32][41] float buffer that
//     reuses the grid staging; lane e then runs env e's agents of the group in agent order: mask, stable softmax,
//     an inverse-CDF draw from one Philox word (pol_draw: key (seed ^ "CTEP", env_id_base + env), counter
//     (counter, agent)), and adds the agent's log-probability to the env's joint one.  In greedy mode (the template
//     parameter GREEDY, from a.greedy) the action is the first index of the largest masked logit instead, no Philox.
//
// Layers 1-2 and the heads + draws are written in mapf_cte_trunk.inc / mapf_cte_heads.inc, which the recurrent CTE
// kernels (mapf_cte_lstm_policy_kernel.cuh) include as well.
// Supported: 1 <= N <= MAPF_MAX_AGENTS, 1 <= R*C <= MAPF_CTE_POLICY_MAX_CELLS (1024: W1 of 64 x 1056 bf16, 132 KB,
// stays resident next to the 8 warps' 6 KB staging buffers within the 227 KB of one block).
#pragma once

#include "mapf_policy_kernel.cuh"

namespace mapf {

constexpr int CTE_THREADS = 256;           // 8 warps, one 32-env tile each at a time
constexpr int CTE_KC = 64;                 // grid columns per staged chunk
constexpr int CTE_STAGE_STRIDE = CTE_KC + 32;   // bytes per staged row (96: conflict-free 64-bit fragment loads)
constexpr int CTE_WARP_BYTES = 2 * 32 * CTE_STAGE_STRIDE;   // two stages; the head buffer [32][41] f32 reuses them
constexpr int CTE_OS = 41;                 // f32 row stride of the head buffer (odd: conflict-free row reads)
static_assert(32 * CTE_OS * 4 <= CTE_WARP_BYTES, "head buffer must fit the staging buffers");

__host__ __device__ constexpr int cte_kpad(int cells) { return (cells + 31) & ~31; }
__host__ __device__ constexpr int cte_s1(int cells) { return cte_kpad(cells) + (cte_kpad(cells) % 64 == 0 ? 32 : 0); }
__host__ __device__ constexpr int cte_head_tiles(int n) { return (5 * n + 1 + 7) / 8; }
// packed weight block (bytes), also its shared-memory image: w1 [64][S1] | w2 [64][72] | w3 [8 NT][72] (rows 0 .. 5N-1
// logits, 5N value, the rest zero) | f32 b1[64] b2[64] b3[8 NT]
__host__ __device__ constexpr long long cte_weight_bytes(int cells, int n) {
    return (long long)(POL_H * cte_s1(cells) + POL_H * POL_W2_STRIDE + 8 * cte_head_tiles(n) * POL_W2_STRIDE) * 2 +
           (2 * POL_H + 8 * cte_head_tiles(n)) * 4;
}

__device__ __forceinline__ uint32_t cte_code_pair(uint32_t w, uint32_t sel) {   // two code bytes of w -> bf16x2
    uint32_t v = __byte_perm(w, 0x43434343u, sel);
    __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162 *>(&v);
    h = __hsub2(h, __floats2bfloat162_rn(128.f, 128.f));
    return *reinterpret_cast<uint32_t *>(&h);
}

// stage columns [k0, k0 + CTE_KC) of the tile's rows r < na (row r at obs + r * cells) into st[r][0 .. CTE_KC);
// W = 16 / 8 / 4: cp.async of W bytes (row length and base are W-aligned), 1: plain byte loads
__device__ __forceinline__ void cte_stage(const uint8_t *obs, int cells, int na, int k0, int W, uint8_t *st, int lane) {
    const int ncol = min(CTE_KC, cells - k0);
    if (ncol <= 0) return;
    const int segs = CTE_KC / W;
    for (int i = lane; i < 32 * segs; i += 32) {
        const int r = i / segs, c = (i - r * segs) * W;
        if (r >= na || c >= ncol) continue;
        const uint8_t *src = obs + (long long)r * cells + k0 + c;
        uint8_t *dst = st + r * CTE_STAGE_STRIDE + c;
        const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
        if (W == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src));
        else if (W == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(src));
        else if (W == 4) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src));
        else *dst = *src;
    }
}

// GREEDY = a.greedy: the first argmax of each agent's masked logits instead of the draw (mapf_cte_heads.inc)
template <bool GREEDY>
__global__ void __launch_bounds__(CTE_THREADS, 1) mapf_cte_policy_act_kernel(const mapf_cte_policy_args a) {
    extern __shared__ __align__(16) unsigned char psm[];
    const int cells = a.cells, N = a.num_agents, S1 = cte_s1(cells), KP = cte_kpad(cells), NT = cte_head_tiles(N);
    __nv_bfloat16 *w1 = reinterpret_cast<__nv_bfloat16 *>(psm);                 // [64][S1]
    __nv_bfloat16 *w2 = w1 + POL_H * S1;                                        // [64][72]
    __nv_bfloat16 *w3 = w2 + POL_H * POL_W2_STRIDE;                             // [8 NT][72]
    float *bias = reinterpret_cast<float *>(w3 + 8 * NT * POL_W2_STRIDE);       // b1[64] b2[64] b3[8 NT]
    const float *b3 = bias + 2 * POL_H;
    unsigned char *wsm0 = reinterpret_cast<unsigned char *>(bias + 2 * POL_H + 8 * NT);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    {   // weights: already bf16 and padded on the host side (mapf_cte_policy_pack_weights)
        const uint4 *src = reinterpret_cast<const uint4 *>(a.weights);
        uint4 *dst = reinterpret_cast<uint4 *>(psm);
        const int n16 = (int)((wsm0 - psm) >> 4);
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    uint8_t *stg = wsm0 + warp * CTE_WARP_BYTES;                                // [2][32][96] grid bytes
    float *os = reinterpret_cast<float *>(stg);                                 // [32][41] head outputs (after layer 1)
    const int g = lane >> 2, t = lane & 3;
    // copy width: the widest of 16 / 8 / 4 bytes that divides the row length and the base address
    const unsigned long long al = (unsigned long long)cells | reinterpret_cast<uintptr_t>(a.obs_grid);
    const int W = (al & 15) == 0 ? 16 : (al & 7) == 0 ? 8 : (al & 3) == 0 ? 4 : 1;
    const int nst = (KP + CTE_KC - 1) / CTE_KC;
    const long long ntiles = ((long long)a.num_envs + 31) >> 5;
    constexpr unsigned long long draw_tag = 0x43544550ull;   // "CTEP"
    for (long long tile = (long long)blockIdx.x * warps + warp; tile < ntiles; tile += (long long)gridDim.x * warps) {
        const long long e0 = tile << 5;
        const int na = a.num_envs - e0 < 32 ? (int)(a.num_envs - e0) : 32;
        const uint8_t *obs = a.obs_grid + e0 * cells;
#include "mapf_cte_trunk.inc"
#include "mapf_cte_heads.inc"
    }
}

}  // namespace mapf
