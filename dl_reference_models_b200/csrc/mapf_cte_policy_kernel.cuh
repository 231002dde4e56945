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
//     (counter, agent)), and adds the agent's log-probability to the env's joint one.
//
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
    for (long long tile = (long long)blockIdx.x * warps + warp; tile < ntiles; tile += (long long)gridDim.x * warps) {
        const long long e0 = tile << 5;
        const int na = a.num_envs - e0 < 32 ? (int)(a.num_envs - e0) : 32;
        const uint8_t *obs = a.obs_grid + e0 * cells;
        // ------------------------------------------------------------ layer 1: K = R*C, double-buffered staging
        float d[2][POL_H / 8][4];
#pragma unroll
        for (int j = 0; j < POL_H / 8; ++j) {
            const float2 bb = *reinterpret_cast<const float2 *>(bias + 8 * j + 2 * t);
#pragma unroll
            for (int m = 0; m < 2; ++m) { d[m][j][0] = bb.x; d[m][j][1] = bb.y; d[m][j][2] = bb.x; d[m][j][3] = bb.y; }
        }
        cte_stage(obs, cells, na, 0, W, stg, lane);
        asm volatile("cp.async.commit_group;" ::: "memory");
        for (int s = 0; s < nst; ++s) {
            if (s + 1 < nst) cte_stage(obs, cells, na, (s + 1) * CTE_KC, W, stg + ((s + 1) & 1) * 32 * CTE_STAGE_STRIDE, lane);
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 1;" ::: "memory");
            __syncwarp();
            const uint8_t *st = stg + (s & 1) * 32 * CTE_STAGE_STRIDE;
#pragma unroll
            for (int sc = 0; sc < CTE_KC / 32; ++sc) {
                const int kb = s * CTE_KC + 32 * sc;
                if (kb >= KP) break;
                uint32_t af[2][2][4];   // [m-tile][k16 chunk]
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    const uint2 v0 = *reinterpret_cast<const uint2 *>(st + (16 * m + g) * CTE_STAGE_STRIDE + 32 * sc + 8 * t);
                    const uint2 v1 = *reinterpret_cast<const uint2 *>(st + (16 * m + g + 8) * CTE_STAGE_STRIDE + 32 * sc + 8 * t);
                    af[m][0][0] = cte_code_pair(v0.x, 0x4140u); af[m][0][1] = cte_code_pair(v1.x, 0x4140u);
                    af[m][0][2] = cte_code_pair(v0.x, 0x4342u); af[m][0][3] = cte_code_pair(v1.x, 0x4342u);
                    af[m][1][0] = cte_code_pair(v0.y, 0x4140u); af[m][1][1] = cte_code_pair(v1.y, 0x4140u);
                    af[m][1][2] = cte_code_pair(v0.y, 0x4342u); af[m][1][3] = cte_code_pair(v1.y, 0x4342u);
                }
#pragma unroll
                for (int j = 0; j < POL_H / 8; ++j) {
                    const uint4 wb = *reinterpret_cast<const uint4 *>(w1 + (8 * j + g) * S1 + kb + 8 * t);
#pragma unroll
                    for (int m = 0; m < 2; ++m) {
                        mma_bf16_16816(d[m][j], af[m][0], wb.x, wb.y);
                        mma_bf16_16816(d[m][j], af[m][1], wb.z, wb.w);
                    }
                }
            }
            __syncwarp();   // every lane is done with this stage before it is refilled
        }
        // ------------------------------------------------------------ layer 2
        uint32_t h2[2][POL_H / 16][4];
#pragma unroll
        for (int m = 0; m < 2; ++m) {
            uint32_t h1[POL_H / 16][4];
#pragma unroll
            for (int j = 0; j < POL_H / 8; ++j) {
                h1[j >> 1][(j & 1) * 2 + 0] = pack_relu_bf16(d[m][j][0], d[m][j][1]);   // row g,   cols 8j + 2t, +1
                h1[j >> 1][(j & 1) * 2 + 1] = pack_relu_bf16(d[m][j][2], d[m][j][3]);   // row g+8
            }
            pol_layer2(h1, w2, bias + POL_H, g, t, h2[m]);
        }
        // ------------------------------------------------------------ heads in groups of 5 n8 tiles, then the draws
        const long long env = e0 + lane;
        float lsum = 0.f;
        for (int j0 = 0; j0 < NT; j0 += 5) {
            for (int j = j0; j < j0 + 5 && j < NT; ++j) {
                const float2 bb = *reinterpret_cast<const float2 *>(b3 + 8 * j + 2 * t);
#pragma unroll
                for (int m = 0; m < 2; ++m) {
                    float o[4] = {bb.x, bb.y, bb.x, bb.y};
#pragma unroll
                    for (int kk = 0; kk < POL_H / 16; ++kk) {
                        const uint32_t *wb = reinterpret_cast<const uint32_t *>(w3 + (8 * j + g) * POL_W2_STRIDE + 16 * kk + 2 * t);
                        mma_bf16_16816(o, h2[m][kk], wb[0], wb[4]);
                    }
                    float *r0 = os + (16 * m + g) * CTE_OS + 8 * (j - j0) + 2 * t, *r1 = r0 + 8 * CTE_OS;
                    r0[0] = o[0]; r0[1] = o[1]; r1[0] = o[2]; r1[1] = o[3];
                }
            }
            __syncwarp();
            if (lane < na) {
                const float *row = os + lane * CTE_OS;
                const int ag1 = min(N, j0 / 5 * 8 + 8);
                for (int ag = j0 / 5 * 8; ag < ag1; ++ag) {
                    const float *lr = row + 5 * ag - 8 * j0;
                    const long long idx = env * N + ag;
                    float l[5];
                    const int8_t *mk = a.action_mask + idx * 5;
#pragma unroll
                    for (int k = 0; k < 5; ++k) l[k] = lr[k] + (mk[k] ? 9.99999e-07f : -13.815511f);   // action_mask_model.py:57-61
                    float mx = l[0];
#pragma unroll
                    for (int k = 1; k < 5; ++k) mx = fmaxf(mx, l[k]);
                    float pr[5], sum = 0.f;
#pragma unroll
                    for (int k = 0; k < 5; ++k) { pr[k] = __expf(l[k] - mx); sum += pr[k]; }
                    const int act = pol_draw(a.seed ^ 0x43544550ull /* "CTEP" */, a.env_id_base + env, a.counter, ag, pr, sum);
                    float la = l[0];   // l[act] without a local-memory array
#pragma unroll
                    for (int k = 1; k < 5; ++k) la = act == k ? l[k] : la;
                    lsum += la - mx - __logf(sum);
                    if (a.actions) a.actions[idx] = (int8_t)act;
                    if (a.actions64) a.actions64[idx] = (long long)act;
                    if (a.logits_out) {
#pragma unroll
                        for (int k = 0; k < 5; ++k) a.logits_out[idx * 5 + k] = l[k];
                    }
                }
                if (a.value && 5 * N >= 8 * j0 && 5 * N < 8 * j0 + 40) a.value[env] = row[5 * N - 8 * j0];
            }
            __syncwarp();
        }
        if (a.logp && lane < na) a.logp[env] = lsum;
    }
}

}  // namespace mapf
