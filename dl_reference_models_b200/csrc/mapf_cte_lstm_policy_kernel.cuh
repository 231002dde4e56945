// mapf_cte_lstm_policy_kernel.cuh -- the recurrent centralised (CTE) policy: the grid codes -> the 64-64 ReLU trunk of
// mapf_cte_policy_act -> LSTMCell(64 + 5N + 1, 64) fed with [trunk output | one-hot of the previous joint action |
// previous reward] -> {5N logits, value} from the new h -> per agent a masked 5-way draw.  cte_rollout.CteRecurrentPolicy
// is the specification, RecurrentCteCollector's reset cut the episode-start rule.
//
// Two launches per call, because the resident weights do not fit one block together: at 1 024 cells W1 alone is 132 KB,
// and the gate weights at N = 32 are 148 KB.
//   1. mapf_cte_lstm_trunk_kernel: layers 1 and 2 exactly as mapf_cte_policy_act_kernel (mapf_cte_trunk.inc), storing the bf16
//      trunk output y to the caller's [B, 64] workspace (128 B per env, read back from L2 by the second launch);
//   2. mapf_cte_lstm_step_kernel: a warp takes 32 envs (two m16 tiles, one after the other).  The gate GEMM is one
//      bf16 m16n8k16 mma.sync product of depth K = 64 (y) + KH (the one-hot, 5N padded to 16; exact in bf16) + 64
//      (bf16 h) against [W_ih without its reward column | 0 | W_hh], rows [i; f; g; o] as torch's LSTMCell.  The
//      reward is not exact in bf16 (the CTE penalties -0.2 / -0.05), so its term is added with f32 FMAs from an f32
//      copy of that W_ih column.  As in mapf_lstm_policy_act_kernel the four gate tiles of an 8-column block are
//      accumulated side by side and the cell update runs in registers with c in f32 (lstm_gate_chunk, lstm_sigmoid,
//      the accurate tanhf).  The previous actions of the warp's 32 envs are staged in shared memory, and each lane
//      turns its rows' into a bit mask of the one-hot columns it holds (4 bits per k16 chunk); the A fragments of the
//      one-hot chunks are rebuilt from that mask in every column block.  Every A fragment of an m-tile (y, one-hot,
//      h) is read before the first h / c of that m-tile is written, so the state may be updated in place.  The heads
//      and the draws (or, GREEDY, the argmax) are mapf_cte_policy_act_kernel's (mapf_cte_heads.inc), with the Philox
//      tag "CTEL".
// Shared memory of the step kernel at N = 32: 148 KB of gate weights, 24 KB of heads, 3 KB of f32 vectors and 8 warps'
// [32][41] f32 head buffers (41 KB, which also hold the staged previous actions): 215 KB.
#pragma once

#include "mapf_cte_policy_kernel.cuh"
#include "mapf_policy_lstm_kernel.cuh"

namespace mapf {

constexpr int CTEL_THREADS = 256;                      // 8 warps: 16 would not fit the head buffers at N = 32
constexpr int CTEL_WARP_BYTES = 32 * CTE_OS * 4;       // [32][41] f32 head buffer; the staged actions [32][N] reuse it
static_assert(32 * MAPF_MAX_AGENTS <= CTEL_WARP_BYTES, "the staged previous actions must fit the head buffer");

__host__ __device__ constexpr int ctel_kh(int n) { return (5 * n + 15) & ~15; }            // one-hot columns, padded
__host__ __device__ constexpr int ctel_sg(int n) { return 2 * POL_H + ctel_kh(n) + 8; }   // gate row stride (bf16)
// packed weight block (bytes) in two parts, each also the shared-memory image of its kernel:
//   trunk: w1 [64][S1] | w2 [64][72] | f32 b1[64] b2[64]
//   step:  wg [256][SG] (cols 0..63 W_ih y part, 64..64+5N-1 its one-hot part, then zero, then W_hh at 64 + KH) |
//          w3 [8 NT][72] (5N logits, the value, zero rows) | f32 bg[256] (b_ih + b_hh) wr[256] (W_ih reward column) b3[8 NT]
__host__ __device__ constexpr long long ctel_trunk_bytes(int cells) {
    return (long long)(POL_H * cte_s1(cells) + POL_H * POL_W2_STRIDE) * 2 + 2 * POL_H * 4;
}
__host__ __device__ constexpr long long ctel_step_bytes(int n) {
    return (long long)(4 * POL_H * ctel_sg(n) + 8 * cte_head_tiles(n) * POL_W2_STRIDE) * 2 + (8 * POL_H + 8 * cte_head_tiles(n)) * 4;
}

__global__ void __launch_bounds__(CTE_THREADS, 1) mapf_cte_lstm_trunk_kernel(const mapf_cte_lstm_policy_args a) {
    extern __shared__ __align__(16) unsigned char psm[];
    const int cells = a.cells, S1 = cte_s1(cells), KP = cte_kpad(cells);
    __nv_bfloat16 *w1 = reinterpret_cast<__nv_bfloat16 *>(psm);                 // [64][S1]
    __nv_bfloat16 *w2 = w1 + POL_H * S1;                                        // [64][72]
    float *bias = reinterpret_cast<float *>(w2 + POL_H * POL_W2_STRIDE);        // b1[64] b2[64]
    unsigned char *wsm0 = reinterpret_cast<unsigned char *>(bias + 2 * POL_H);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.weights);
        uint4 *dst = reinterpret_cast<uint4 *>(psm);
        const int n16 = (int)((wsm0 - psm) >> 4);
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    uint8_t *stg = wsm0 + warp * CTE_WARP_BYTES;
    const int g = lane >> 2, t = lane & 3;
    const unsigned long long al = (unsigned long long)cells | reinterpret_cast<uintptr_t>(a.obs_grid);
    const int W = (al & 15) == 0 ? 16 : (al & 7) == 0 ? 8 : (al & 3) == 0 ? 4 : 1;
    const int nst = (KP + CTE_KC - 1) / CTE_KC;
    const long long ntiles = ((long long)a.num_envs + 31) >> 5;
    for (long long tile = (long long)blockIdx.x * warps + warp; tile < ntiles; tile += (long long)gridDim.x * warps) {
        const long long e0 = tile << 5;
        const int na = a.num_envs - e0 < 32 ? (int)(a.num_envs - e0) : 32;
        const uint8_t *obs = a.obs_grid + e0 * cells;
#include "mapf_cte_trunk.inc"
        uint32_t *y = reinterpret_cast<uint32_t *>(a.trunk) + e0 * (POL_H / 2);   // 32 bf16x2 words per env
#pragma unroll
        for (int m = 0; m < 2; ++m) {
            const int r0 = 16 * m + g, r1 = r0 + 8;
#pragma unroll
            for (int kk = 0; kk < POL_H / 16; ++kk) {   // cols 16kk + 2t, +1 (word 8kk + t) and 16kk + 8 + 2t, +1
                if (r0 < na) { y[r0 * 32 + 8 * kk + t] = h2[m][kk][0]; y[r0 * 32 + 8 * kk + 4 + t] = h2[m][kk][2]; }
                if (r1 < na) { y[r1 * 32 + 8 * kk + t] = h2[m][kk][1]; y[r1 * 32 + 8 * kk + 4 + t] = h2[m][kk][3]; }
            }
        }
    }
}

// GREEDY = a.greedy: argmax instead of the draw, in the heads only (mapf_cte_heads.inc); the trunk kernel has no mode
template <bool GREEDY>
__global__ void __launch_bounds__(CTEL_THREADS, 1) mapf_cte_lstm_step_kernel(const mapf_cte_lstm_policy_args a) {
    extern __shared__ __align__(16) unsigned char psm[];
    const int N = a.num_agents, NH = ctel_kh(N) / 16, SG = ctel_sg(N), NT = cte_head_tiles(N);
    __nv_bfloat16 *wg = reinterpret_cast<__nv_bfloat16 *>(psm);                 // [256][SG]
    __nv_bfloat16 *w3 = wg + 4 * POL_H * SG;                                    // [8 NT][72]
    float *bg = reinterpret_cast<float *>(w3 + 8 * NT * POL_W2_STRIDE);         // bg[256] wr[256] b3[8 NT]
    const float *wr = bg + 4 * POL_H, *b3 = bg + 8 * POL_H;
    unsigned char *wsm0 = reinterpret_cast<unsigned char *>(bg + 8 * POL_H + 8 * NT);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(static_cast<const unsigned char *>(a.weights) + ctel_trunk_bytes(a.cells));
        uint4 *dst = reinterpret_cast<uint4 *>(psm);
        const int n16 = (int)((wsm0 - psm) >> 4);
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    float *os = reinterpret_cast<float *>(wsm0 + warp * CTEL_WARP_BYTES);      // [32][41] head outputs
    int8_t *pas = reinterpret_cast<int8_t *>(os);                               // [32][N] staged previous actions
    const int g = lane >> 2, t = lane & 3;
    const uint32_t *y = reinterpret_cast<const uint32_t *>(a.trunk);
    const long long ntiles = ((long long)a.num_envs + 31) >> 5;
    constexpr unsigned long long draw_tag = 0x4354454Cull;   // "CTEL"
    for (long long tile = (long long)blockIdx.x * warps + warp; tile < ntiles; tile += (long long)gridDim.x * warps) {
        const long long e0 = tile << 5;
        const int na = a.num_envs - e0 < 32 ? (int)(a.num_envs - e0) : 32;
        for (int i = lane; i < 32 * N; i += 32) pas[i] = i < na * N ? a.prev_action[e0 * N + i] : (int8_t)0;
        __syncwarp();
        uint32_t h2[2][POL_H / 16][4];   // bf16(h'): A fragments of the heads
#pragma unroll
        for (int m = 0; m < 2; ++m) {
            // ------------------------------------------------------------ per-row inputs, episode-start cut
            bool valid[2], live[2];
            long long env[2];
            float pr[2];
            unsigned long long oh[2];   // bit 4 kc + s: one-hot column 16 kc + 2t + (s & 1) + 8 (s >> 1) of the row
            uint32_t yf[POL_H / 16][4], hf[POL_H / 16][4];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int row = 16 * m + g + 8 * r;
                env[r] = e0 + row;
                valid[r] = row < na;
                const bool start = valid[r] && ((a.prev_terminated && a.prev_terminated[env[r]]) ||
                                                (a.prev_truncated && a.prev_truncated[env[r]]));
                live[r] = valid[r] && !start;   // h, c, previous action and reward as stored; otherwise zero
                pr[r] = live[r] ? (float)a.prev_reward[env[r]] : 0.f;
                oh[r] = 0ull;
                if (valid[r]) {   // behind an episode start every agent's previous action counts as 0 (one-hot at 0)
                    for (int kc = 0; kc < NH; ++kc) {
#pragma unroll
                        for (int s = 0; s < 4; ++s) {
                            const int col = 16 * kc + 2 * t + (s & 1) + 8 * (s >> 1), ag = col / 5;
                            if (ag < N && (live[r] ? pas[row * N + ag] : 0) == col - 5 * ag) oh[r] |= 1ull << (4 * kc + s);
                        }
                    }
                }
                const uint32_t *yr = y + env[r] * (POL_H / 2);
                const float *hr = a.h_in + env[r] * POL_H;
#pragma unroll
                for (int kk = 0; kk < POL_H / 16; ++kk) {
                    yf[kk][r] = valid[r] ? yr[8 * kk + t] : 0u;            // a[0] / a[1]: cols 2t, +1 of rows g / g + 8
                    yf[kk][2 + r] = valid[r] ? yr[8 * kk + 4 + t] : 0u;    // a[2] / a[3]: cols 8 + 2t, +1
                    float2 v0 = make_float2(0.f, 0.f), v1 = v0;
                    if (live[r]) {
                        v0 = *reinterpret_cast<const float2 *>(hr + 16 * kk + 2 * t);
                        v1 = *reinterpret_cast<const float2 *>(hr + 16 * kk + 8 + 2 * t);
                    }
                    hf[kk][r] = pack_bf16(v0.x, v0.y);
                    hf[kk][2 + r] = pack_bf16(v1.x, v1.y);
                }
            }
            __syncwarp();   // every h of the m-tile is read (by every lane) before any is written: in place is safe
            // ------------------------------------------------------------ gates + cell update, one 8-column block at a time
#pragma unroll
            for (int j = 0; j < POL_H / 8; ++j) {
                const int col = 8 * j + 2 * t;
                float2 c[2];
#pragma unroll
                for (int r = 0; r < 2; ++r)
                    c[r] = live[r] ? *reinterpret_cast<const float2 *>(a.c_in + env[r] * POL_H + col) : make_float2(0.f, 0.f);
                float d[4][4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {   // bias, then the reward term in f32
                    const float2 bb = *reinterpret_cast<const float2 *>(bg + q * POL_H + col);
                    const float2 ww = *reinterpret_cast<const float2 *>(wr + q * POL_H + col);
                    d[q][0] = fmaf(ww.x, pr[0], bb.x); d[q][1] = fmaf(ww.y, pr[0], bb.y);
                    d[q][2] = fmaf(ww.x, pr[1], bb.x); d[q][3] = fmaf(ww.y, pr[1], bb.y);
                }
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) lstm_gate_chunk(d, yf[kk], wg, j, kk, g, t, SG);
                for (int kc = 0; kc < NH; ++kc) {   // bf16 1.0 = 0x3F80
                    const uint32_t b0 = (uint32_t)(oh[0] >> (4 * kc)), b1 = (uint32_t)(oh[1] >> (4 * kc));
                    const uint32_t af[4] = {((b0 & 1u) ? 0x3F80u : 0u) | ((b0 & 2u) ? 0x3F800000u : 0u),
                                            ((b1 & 1u) ? 0x3F80u : 0u) | ((b1 & 2u) ? 0x3F800000u : 0u),
                                            ((b0 & 4u) ? 0x3F80u : 0u) | ((b0 & 8u) ? 0x3F800000u : 0u),
                                            ((b1 & 4u) ? 0x3F80u : 0u) | ((b1 & 8u) ? 0x3F800000u : 0u)};
                    lstm_gate_chunk(d, af, wg, j, 4 + kc, g, t, SG);
                }
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) lstm_gate_chunk(d, hf[kk], wg, j, 4 + NH + kk, g, t, SG);
                // lane's elements: (row g, col), (row g, col + 1), (row g + 8, col), (row g + 8, col + 1)
                const float cp[4] = {c[0].x, c[0].y, c[1].x, c[1].y};
                float cn[4], hv[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    cn[e] = lstm_sigmoid(d[1][e]) * cp[e] + lstm_sigmoid(d[0][e]) * tanhf(d[2][e]);
                    hv[e] = lstm_sigmoid(d[3][e]) * tanhf(cn[e]);
                }
                if (a.h_out) {   // h_out and c_out are given together
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        if (valid[r]) {
                            *reinterpret_cast<float2 *>(a.c_out + env[r] * POL_H + col) = make_float2(cn[2 * r], cn[2 * r + 1]);
                            *reinterpret_cast<float2 *>(a.h_out + env[r] * POL_H + col) = make_float2(hv[2 * r], hv[2 * r + 1]);
                        }
                    }
                }
                h2[m][j >> 1][(j & 1) * 2 + 0] = pack_bf16(hv[0], hv[1]);
                h2[m][j >> 1][(j & 1) * 2 + 1] = pack_bf16(hv[2], hv[3]);
            }
        }
        __syncwarp();   // every lane is done with the staged actions before the head buffer overwrites them
#include "mapf_cte_heads.inc"
    }
}

}  // namespace mapf
