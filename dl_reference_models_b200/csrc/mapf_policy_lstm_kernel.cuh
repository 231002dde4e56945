// mapf_policy_lstm_kernel.cuh -- the recurrent policy of the reference's PPO configuration (src/agents/ppo.py:67-75:
// fcnet [64, 64] ReLU trunk -> LSTMCell(64 + 5 + 1, 64) fed with the trunk output, the one-hot previous action and the
// previous reward -> logits (masked like the MLP policy) and value from the same cell output, vf_share_layers) evaluated
// straight from the env's output channels, plus the categorical draw, in ONE launch.  recurrent.py's
// RecurrentActionMaskPolicy.step is the specification, RecurrentCollector.collect's reset cut is the episode-start rule.
//
//   * channel loader, trunk, heads and sampler epilogue are mapf_policy_act_kernel's (mapf_policy_kernel.cuh): a warp
//     takes 32 agents, m16n8k16 bf16 mma.sync with f32 accumulation, the accumulator layout of one layer is the
//     A-operand layout of the next;
//   * LSTM input xi = [y (64) | one_hot(prev_action, 5) | prev_reward | 0 x 10]: five k16 chunks, the fifth built in
//     registers (one-hot and the half-integer rewards are exact in bf16); bf16(h_prev) is four more chunks, so the
//     gate GEMM is one K = 144 product against [W_ih | 0 | W_hh] (rows [i; f; g; o] as torch's LSTMCell);
//   * the 256 gate columns never exist as a tile: for each 8-column block j of the cell the four n8 tiles i_j, f_j,
//     g_j, o_j are accumulated side by side, so a lane holds the same (row, column) of all four gates and does the
//     cell update in registers; c (float32 end to end) is read and written there as float2, h' is stored and packed
//     into the A fragments the heads read;
//   * all A fragments of xi and h_prev are loaded before the first column block is stored: in-place state update is
//     safe (every h / c element of the tile is read by this warp before this warp writes it).
#pragma once

#include "mapf_policy_kernel.cuh"

namespace mapf {

constexpr int LSTM_THREADS = 512;   // 16 warps: one block per SM (the ~97 KB weight block), 128 registers per thread
constexpr int LSTM_KX = 80;         // xi columns: 64 trunk + 5 one-hot + 1 reward + 10 zero
constexpr int LSTM_K = LSTM_KX + POL_H;   // 144: gate GEMM depth
constexpr int LSTM_SG = LSTM_K + 8;       // bf16 row stride of the gate weights (152: conflict-free fragment loads)

// packed weight block (bytes), also its shared-memory image: w1 [64][S1] | w2 [64][72] | w3 [8][72] | wg [256][152] |
// f32 b1[64] b2[64] b3[8] bg[256] (bg = b_ih + b_hh)
__host__ __device__ constexpr int lstm_weight_bytes(int kc1) {
    return (POL_H * (16 * kc1 + 8) + POL_H * POL_W2_STRIDE + 8 * POL_W2_STRIDE + 4 * POL_H * LSTM_SG) * 2 +
           (2 * POL_H + 8 + 4 * POL_H) * 4;
}

// sigmoid through the accurate tanhf: no division (and no slow-path call) in the cell update
__device__ __forceinline__ float lstm_sigmoid(float x) { return fmaf(0.5f, tanhf(0.5f * x), 0.5f); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&v);
}

// the four gate tiles i_j, f_j, g_j, o_j of column block j += A chunk kk x [W_ih | 0 | W_hh] rows q * 64 + 8j + g
// (bf16 row stride sg: LSTM_SG here, the recurrent CTE kernel's own in mapf_cte_lstm_policy_kernel.cuh)
__device__ __forceinline__ void lstm_gate_chunk(float (&d)[4][4], const uint32_t (&af)[4], const __nv_bfloat16 *wg, int j,
                                                int kk, int g, int t, int sg = LSTM_SG) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint32_t *wb = reinterpret_cast<const uint32_t *>(wg + (q * POL_H + 8 * j + g) * sg + 16 * kk + 2 * t);
        mma_bf16_16816(d[q], af, wb[0], wb[4]);
    }
}

// GREEDY = a.greedy: argmax instead of the draw, in the epilogue only, where the gate fragments are dead (see
// pol_sample for why it is a template parameter); PER_AGENT: a.weights holds num_agents consecutive blocks and tile
// rows are one agent's (pol_per_agent_tiles)
template <int KC1, bool GREEDY, bool PER_AGENT = false>
__global__ void __launch_bounds__(LSTM_THREADS, 1) mapf_lstm_policy_act_kernel(const mapf_lstm_policy_args a) {
    constexpr int S1 = 16 * KC1 + 8;
    extern __shared__ __align__(16) unsigned char psm[];
    __nv_bfloat16 *w1 = reinterpret_cast<__nv_bfloat16 *>(psm);                 // [64][S1]
    __nv_bfloat16 *w2 = w1 + POL_H * S1;                                        // [64][72]
    __nv_bfloat16 *w3 = w2 + POL_H * POL_W2_STRIDE;                             // [8][72]: 5 logits, value, 2 zero rows
    __nv_bfloat16 *wg = w3 + 8 * POL_W2_STRIDE;                                 // [256][152]
    float *bias = reinterpret_cast<float *>(wg + 4 * POL_H * LSTM_SG);          // b1[64] b2[64] b3[8] bg[256]
    const float *bg = bias + 2 * POL_H + 8;
    unsigned char *wsm0 = psm + lstm_weight_bytes(KC1);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    if constexpr (!PER_AGENT) {   // weights: already bf16 and padded on the host side (mapf_lstm_policy_pack_weights)
        const uint4 *src = reinterpret_cast<const uint4 *>(a.weights);
        uint4 *dst = reinterpret_cast<uint4 *>(psm);
        for (int i = tid; i < lstm_weight_bytes(KC1) / 16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    const int V2 = a.v2, N = a.num_agents;
    unsigned char *wsm = wsm0 + warp * pol_warp_bytes(KC1, V2);
    __nv_bfloat16 *xs = reinterpret_cast<__nv_bfloat16 *>(wsm);                 // [32][S1] bf16 features
    uint32_t *raw = reinterpret_cast<uint32_t *>(wsm + 32 * S1 * 2);
    uint32_t *rawm = reinterpret_cast<uint32_t *>(wsm + 32 * S1 * 2 + pol_raw_bytes(V2));
    float *os = reinterpret_cast<float *>(wsm + 32 * S1 * 2 + pol_raw_bytes(V2) + 160);     // [32][8] head outputs
    const int g = lane >> 2, t = lane & 3;
    auto tile_body = [&](const long long ag0, const int na) {
        if constexpr (PER_AGENT) pol_gather_tile(a.local_obs, a.action_mask, nullptr, V2, ag0, N, na, raw, rawm, lane);
        else pol_load_tile(a.local_obs, a.action_mask, nullptr, V2, ag0, na, raw, rawm, lane);
        __syncwarp();
        pol_feature_row<KC1, PER_AGENT>(xs, raw, a.goal_delta, a.blocking_prev, V2, ag0, na, lane, N);
        __syncwarp();
#pragma unroll 1
        for (int mt = 0; mt < 2; ++mt) {
            const int row0 = 16 * mt + g;   // this lane's rows: row0 and row0 + 8
            uint32_t y[POL_H / 16][4];      // trunk output = xi chunks 0..3
            pol_trunk<KC1>(xs, w1, w2, bias, row0, g, t, y);
            // ------------------------------------------------------------ per-row recurrent inputs, episode-start cut
            bool live[2];
            long long agr[2];
            uint32_t xa[2];   // xi chunk 4 (cols 64 + 2t, +1): rows row0 / row0 + 8; cols 72..79 are zero
            uint32_t hf[POL_H / 16][4];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int row = row0 + 8 * r;
                agr[r] = pol_row<PER_AGENT>(ag0, row, N);
                const bool valid = row < na;
                bool start = false;
                int pa = 0;
                float pr = 0.f;
                if (valid) {
                    const unsigned env = (unsigned)agr[r] / (unsigned)N;   // B * N < 2^32, as in pol_sample
                    start = (a.prev_terminated && a.prev_terminated[env]) || (a.prev_truncated && a.prev_truncated[env]);
                    if (!start) {
                        pa = a.prev_action[agr[r]];
                        pr = a.prev_reward[agr[r]];
                    }
                }
                live[r] = valid && !start;   // h, c as stored; otherwise zero
                // one_hot(pa) at cols 0..4, reward at col 5 of the chunk: lane t holds cols 2t, 2t + 1
                const float lo = t < 3 ? (pa == 2 * t ? 1.f : 0.f) : 0.f;
                const float hi = t < 2 ? (pa == 2 * t + 1 ? 1.f : 0.f) : (t == 2 ? pr : 0.f);
                xa[r] = valid ? pack_bf16(lo, hi) : 0u;
                const float *hr = a.h_in + agr[r] * POL_H;
#pragma unroll
                for (int kk = 0; kk < POL_H / 16; ++kk) {
                    float2 v0 = make_float2(0.f, 0.f), v1 = v0;
                    if (live[r]) {
                        v0 = *reinterpret_cast<const float2 *>(hr + 16 * kk + 2 * t);
                        v1 = *reinterpret_cast<const float2 *>(hr + 16 * kk + 8 + 2 * t);
                    }
                    hf[kk][r] = pack_bf16(v0.x, v0.y);       // a[0] / a[1]: cols 2t, +1 of row0 / row0 + 8
                    hf[kk][2 + r] = pack_bf16(v1.x, v1.y);   // a[2] / a[3]: cols 8 + 2t, +1
                }
            }
            const uint32_t xf[4] = {xa[0], xa[1], 0u, 0u};
            // ------------------------------------------------------------ gates + cell update, one 8-column block at a time
            uint32_t hn[POL_H / 16][4];   // bf16(h'): A fragments of the heads
#pragma unroll
            for (int j = 0; j < POL_H / 8; ++j) {
                const int col = 8 * j + 2 * t;
                float2 c[2];
#pragma unroll
                for (int r = 0; r < 2; ++r)
                    c[r] = live[r] ? *reinterpret_cast<const float2 *>(a.c_in + agr[r] * POL_H + col) : make_float2(0.f, 0.f);
                float d[4][4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float2 bb = *reinterpret_cast<const float2 *>(bg + q * POL_H + col);
                    d[q][0] = bb.x; d[q][1] = bb.y; d[q][2] = bb.x; d[q][3] = bb.y;
                }
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) lstm_gate_chunk(d, y[kk], wg, j, kk, g, t);
                lstm_gate_chunk(d, xf, wg, j, 4, g, t);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) lstm_gate_chunk(d, hf[kk], wg, j, 5 + kk, g, t);
                // lane's elements: (row0, col), (row0, col + 1), (row0 + 8, col), (row0 + 8, col + 1)
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
                        if (PER_AGENT ? row0 + 8 * r < na : agr[r] - ag0 < na) {
                            *reinterpret_cast<float2 *>(a.c_out + agr[r] * POL_H + col) = make_float2(cn[2 * r], cn[2 * r + 1]);
                            *reinterpret_cast<float2 *>(a.h_out + agr[r] * POL_H + col) = make_float2(hv[2 * r], hv[2 * r + 1]);
                        }
                    }
                }
                hn[j >> 1][(j & 1) * 2 + 0] = pack_bf16(hv[0], hv[1]);
                hn[j >> 1][(j & 1) * 2 + 1] = pack_bf16(hv[2], hv[3]);
            }
            pol_heads(hn, w3, bias + 2 * POL_H, os, row0, g, t);
        }
        __syncwarp();
        if (lane < na) pol_sample<GREEDY>(a, os, rawm, lane, pol_row<PER_AGENT>(ag0, lane, N), N, 0x4C53544Dull /* "LSTM" */);
        __syncwarp();
    };
    if constexpr (PER_AGENT) {
        pol_per_agent_tiles(a.num_envs, N, warp, warps, [&](int j) {
            const uint4 *src = reinterpret_cast<const uint4 *>(static_cast<const unsigned char *>(a.weights) +
                                                               (long long)j * lstm_weight_bytes(KC1));
            uint4 *dst = reinterpret_cast<uint4 *>(psm);
            for (int i = tid; i < lstm_weight_bytes(KC1) / 16; i += blockDim.x) dst[i] = src[i];
        }, tile_body);
    } else {
        const long long BN = (long long)a.num_envs * N;
        const long long ntiles = (BN + 31) >> 5;
        for (long long tile = (long long)blockIdx.x * warps + warp; tile < ntiles; tile += (long long)gridDim.x * warps) {
            const long long ag0 = tile << 5;
            const long long left = BN - ag0;
            tile_body(ag0, left < 32 ? (int)left : 32);
        }
    }
}

}  // namespace mapf
