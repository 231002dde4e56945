// mapf_q_kernel.cuh -- DQN's epsilon-greedy action selection over a dueling Q head (the reference's
// src/agents/dqn.py, SURVEY §2 row 6); the C ABI is mapf_q_act / mapf_q_act_per_agent (include/mapf_b200.h).
//
// The network is the fused action-mask MLP of mapf_policy_kernel.cuh, unchanged: the same packed weight block, the
// same tile loads, feature rows, trunk and heads (pol_* helpers, per agent pol_per_agent_tiles).  Only the epilogue is
// new: the 5-wide head is the advantage A and the scalar head the value V, Q = V + (A - mean(A)) in f32, masked Q =
// Q where the action is legal and FLOAT_MIN elsewhere, then an epsilon-greedy choice from one Philox block.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "mapf_policy_kernel.cuh"

namespace mapf {

// one agent per lane (call for lane < na): dueling Q from the head outputs os[lane][0..5], masking, the
// epsilon-greedy action; writes a.actions[ag] and, if requested, the masked Q to a.q_out[ag][0..4]
__device__ __forceinline__ void q_select(const mapf_q_act_args &a, const float *os, const uint32_t *rawm, int lane,
                                         long long ag, int N) {
    const float4 o03 = *reinterpret_cast<const float4 *>(os + lane * 8);
    const float2 o45 = *reinterpret_cast<const float2 *>(os + lane * 8 + 4);
    const float adv[5] = {o03.x, o03.y, o03.z, o03.w, o45.x};
    const float mean = (adv[0] + adv[1] + adv[2] + adv[3] + adv[4]) * 0.2f;
    const uint8_t *mk = reinterpret_cast<const uint8_t *>(rawm) + lane * 5;
    float q[5];
    unsigned legal = 0;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        const bool ok = a.no_masking || mk[k] != 0;
        q[k] = ok ? o45.y + (adv[k] - mean) : -3.4e38f;   // torch.where(mask, Q, FLOAT_MIN)
        legal |= ok ? 1u << k : 0u;
    }
    int act = 0;
    float best = q[0];
#pragma unroll
    for (int k = 1; k < 5; ++k) { if (q[k] > best) { best = q[k]; act = k; } }
    if (a.epsilon > 0.f) {
        const unsigned env = (unsigned)((unsigned long long)ag / (unsigned)N);   // B * N < 2^32 in any batch that fits a GPU
        const int agent = (int)(ag - (long long)env * N);
        Philox ph(a.seed ^ 0x44514E45ull /* "DQNE" */, a.env_id_base + env);
        const uint4 x = ph((uint32_t)a.counter, (uint32_t)(a.counter >> 32), (uint32_t)agent, 0u);
        if ((double)x.x * (1.0 / 4294967296.0) < (double)a.epsilon) {
            const int n_legal = __popc(legal);
            int k = (int)(((unsigned long long)x.y * (unsigned)n_legal) >> 32);   // the k-th legal action
#pragma unroll
            for (int c = 0; c < 5; ++c) {
                if (legal >> c & 1u) {
                    if (k == 0) act = c;
                    --k;
                }
            }
        }
    }
    a.actions[ag] = (int8_t)act;
    if (a.q_out) {
#pragma unroll
        for (int k = 0; k < 5; ++k) a.q_out[ag * 5 + k] = q[k];
    }
}

// KC1 = k16 chunks of the first layer (as mapf_policy_act_kernel); PER_AGENT: a.weights holds num_agents consecutive
// blocks and tile rows are one agent's (pol_per_agent_tiles).  Launched with 256 threads; the register cap replaces
// __launch_bounds__(256), under which ptxas gives the per-agent KC1 = 2 instantiation 64 registers and a spill.
template <int KC1, bool PER_AGENT>
__global__ void __maxnreg__(96) mapf_q_act_kernel(const mapf_q_act_args a) {
    constexpr int S1 = 16 * KC1 + 8;
    extern __shared__ __align__(16) unsigned char psm[];
    __nv_bfloat16 *w1 = reinterpret_cast<__nv_bfloat16 *>(psm);                 // [64][S1]
    __nv_bfloat16 *w2 = w1 + POL_H * S1;                                        // [64][72]
    __nv_bfloat16 *w3 = w2 + POL_H * POL_W2_STRIDE;                             // [8][72]: A[5], V, 2 zero rows
    float *bias = reinterpret_cast<float *>(w3 + 8 * POL_W2_STRIDE);            // b1[64] b2[64] b3[8]
    unsigned char *wsm0 = reinterpret_cast<unsigned char *>(bias + 2 * POL_H + 8);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    const int n16 = (int)((wsm0 - psm) >> 4);   // 16-byte words of one weight block
    if constexpr (!PER_AGENT) {
        const uint4 *src = reinterpret_cast<const uint4 *>(a.weights);
        uint4 *dst = reinterpret_cast<uint4 *>(psm);
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    const int V2 = a.v2, N = a.num_agents;
    unsigned char *wsm = wsm0 + warp * pol_warp_bytes(KC1, V2);
    __nv_bfloat16 *xs = reinterpret_cast<__nv_bfloat16 *>(wsm);
    uint32_t *raw = reinterpret_cast<uint32_t *>(wsm + 32 * S1 * 2);
    uint32_t *rawm = reinterpret_cast<uint32_t *>(wsm + 32 * S1 * 2 + pol_raw_bytes(V2));
    float *os = reinterpret_cast<float *>(wsm + 32 * S1 * 2 + pol_raw_bytes(V2) + 160);
    const int g = lane >> 2, t = lane & 3;
    auto tile_body = [&](const long long ag0, const int na) {
        if constexpr (PER_AGENT) pol_gather_tile(a.local_obs, a.action_mask, nullptr, V2, ag0, N, na, raw, rawm, lane);
        else pol_load_tile(a.local_obs, a.action_mask, nullptr, V2, ag0, na, raw, rawm, lane);
        __syncwarp();
        pol_feature_row<KC1, PER_AGENT>(xs, raw, a.goal_delta, a.blocking_prev, V2, ag0, na, lane, N);
        __syncwarp();
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int row0 = 16 * mt + g;
            uint32_t h2[POL_H / 16][4];
            pol_trunk<KC1>(xs, w1, w2, bias, row0, g, t, h2);
            pol_heads(h2, w3, bias + 2 * POL_H, os, row0, g, t);
        }
        __syncwarp();
        if (lane < na) q_select(a, os, rawm, lane, pol_row<PER_AGENT>(ag0, lane, N), N);
        __syncwarp();
    };
    if constexpr (PER_AGENT) {
        pol_per_agent_tiles(a.num_envs, N, warp, warps, [&](int j) {
            const uint4 *src = reinterpret_cast<const uint4 *>(a.weights) + (long long)j * n16;
            uint4 *dst = reinterpret_cast<uint4 *>(psm);
            for (int i = tid; i < n16; i += blockDim.x) dst[i] = src[i];
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
