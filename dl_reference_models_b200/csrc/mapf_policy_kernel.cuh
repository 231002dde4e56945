// mapf_policy_kernel.cuh -- rollout-loop kernels around the env step (SURVEY 8f N1, BASELINE config 5).
//
// mapf_policy_act_kernel: the reference's action-mask MLP (models/action_mask_model.py:8-67:
// Linear(F,64)-ReLU-Linear(64,64)-ReLU-{Linear(64,5), Linear(64,1)}, logits + log(mask + 1e-6)) evaluated
// straight from the env's output channels, plus the categorical draw, in ONE launch: the float feature block
// the PyTorch loop materialises (112 B per agent and step, written and re-read several times) never exists.
//   * a warp takes 32 agents: raw channels (u8 window, f32 goal delta, u8 pressure) -> bf16 feature tile in
//     shared memory -> three layers of m16n8k16 bf16 mma.sync with f32 accumulation; the accumulator layout of
//     one layer IS the A-operand layout of the next (two n8 tiles = one k16 chunk), so activations stay in
//     registers between layers;
//   * weights live in shared memory as bf16 (padded row strides: conflict-free fragment loads);
//   * the head's 5 logits + value are gathered inside each lane quad; lane 0 of the quad applies the mask,
//     does a stable softmax and draws by inverse CDF from one Philox word (keyed by the global env id).
// The op is tiny-tile GEMM work bounded by its ~50 B of HBM traffic per agent, not by tensor throughput, which
// is why the legacy mma.sync path is enough here (no TMA / TMEM pipeline to amortise at K <= 64).
// With PER_AGENT (mapf_policy_act_per_agent) every agent has its own weight block: a tile is 32 envs of one agent
// (rows N apart, pol_row), and a CTA reloads the block in shared memory when its agent changes (pol_per_agent_tiles).
//
// mapf_gae_kernel: generalised advantage estimation as a backwards scan, one thread per (env, agent) series.
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "mapf_kernels.cuh"

namespace mapf {

constexpr int POL_H = 64;          // hidden width of both trunk layers
constexpr int POL_W2_STRIDE = 72;  // bf16 row stride of W2 / head weights in shared memory (64 + 8: conflict-free)

__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(fmaxf(lo, 0.f), fmaxf(hi, 0.f));
    return *reinterpret_cast<const uint32_t *>(&v);
}

// per-warp shared memory of mapf_policy_act_kernel (bytes)
__host__ __device__ constexpr int pol_raw_bytes(int v2) { return (((32 * v2 + 3) / 4 + 2) * 4 + 15) & ~15; }   // raw window bytes + slack, 16-byte multiple
__host__ __device__ constexpr int pol_warp_bytes(int kc1, int v2) {
    return 32 * (16 * kc1 + 8) * 2 /* bf16 feature tile */ + pol_raw_bytes(v2) + 160 /* masks */ + 32 * 8 * 4 /* head outputs */;
}

// ---------------------------------------------------------------------------------------------------------------
// Pieces shared by mapf_policy_act_kernel and mapf_lstm_policy_act_kernel (mapf_policy_lstm_kernel.cuh).  All of them
// work on one warp's tile of 32 agents; `g` / `t` are the lane's mma.sync group / thread-in-group indices.

// raw channels of the tile, coalesced: window bytes -> raw, mask bytes -> rawm (+ an optional copy of the masks)
__device__ __forceinline__ void pol_load_tile(const uint8_t *local_obs, const int8_t *action_mask, int8_t *action_mask_out,
                                              int V2, long long ag0, int na, uint32_t *raw, uint32_t *rawm, int lane) {
    const uint32_t *ob32 = reinterpret_cast<const uint32_t *>(local_obs + ag0 * V2);   // 32 * V2 bytes: 4-byte aligned
    const int nwords = (na * V2 + 3) >> 2;
    for (int i = lane; i < (32 * V2 + 3) / 4 + 2; i += 32) raw[i] = i < nwords ? ob32[i] : 0u;
    if (action_mask) {
        const uint32_t *mk32 = reinterpret_cast<const uint32_t *>(action_mask + ag0 * 5);
        const int mwords = (na * 5 + 3) >> 2;
        for (int i = lane; i < 40; i += 32) rawm[i] = i < mwords ? mk32[i] : 0u;
        if (action_mask_out) {   // the rollout buffer's copy of the masks (saves a separate copy launch per step)
            uint32_t *mo32 = reinterpret_cast<uint32_t *>(action_mask_out + ag0 * 5);
            // word copies when the destination row is 4-byte aligned (a [T,B,N,5] row may start anywhere)
            const int full_words = (reinterpret_cast<uintptr_t>(action_mask_out) & 3) == 0 ? (na * 5) >> 2 : 0;
            for (int i = lane; i < full_words; i += 32) mo32[i] = mk32[i];
            for (int i = full_words * 4 + lane; i < na * 5; i += 32) action_mask_out[ag0 * 5 + i] = action_mask[ag0 * 5 + i];
        }
    }
}

// Per-agent policies (mapf_policy_act_per_agent, mapf_lstm_policy_act_per_agent): a tile is (agent j, envs e0 ..
// e0 + 31) and its row r is the flat row (e0 + r) N + j, i.e. ag0 + r N with ag0 = e0 N + j; a shared-policy tile is
// 32 consecutive rows ag0 + r.  Every per-row access of the kernels goes through pol_row.
template <bool PER_AGENT>
__device__ __forceinline__ long long pol_row(long long ag0, int r, int N) {
    if constexpr (PER_AGENT) return ag0 + (long long)r * N;
    else return ag0 + r;
}

// pol_load_tile for a per-agent tile: the window rows are N * V2 bytes apart, gathered into the same raw layout (row r
// at r * V2, zero beyond the tile's na rows and in the slack words), the mask rows into rawm (+ the optional copy)
__device__ __forceinline__ void pol_gather_tile(const uint8_t *local_obs, const int8_t *action_mask, int8_t *action_mask_out,
                                                int V2, long long ag0, int N, int na, uint32_t *raw, uint32_t *rawm, int lane) {
    uint8_t *rb = reinterpret_cast<uint8_t *>(raw);
    for (int i = lane; i < ((32 * V2 + 3) / 4 + 2) * 4; i += 32) {
        const int r = i / V2;
        rb[i] = r < na ? local_obs[pol_row<true>(ag0, r, N) * V2 + (i - r * V2)] : 0;
    }
    if (action_mask) {
        uint8_t *mb = reinterpret_cast<uint8_t *>(rawm);
        for (int i = lane; i < 160; i += 32) {
            const int r = i / 5;
            int8_t v = 0;
            if (r < na) {
                const long long m = pol_row<true>(ag0, r, N) * 5 + (i - r * 5);
                v = action_mask[m];
                if (action_mask_out) action_mask_out[m] = v;
            }
            mb[i] = (uint8_t)v;
        }
    }
}

// The tile loop of the per-agent kernels.  Tiles are ordered agent-major (tile k: agent k / tpa, envs 32 (k % tpa) ..,
// tpa = ceil(B / 32)) and each CTA takes one contiguous range of that order (the ranges of the G CTAs differ in length
// by at most one tile), so it meets only a few agent changes.  The range is walked in rounds of at most one tile per warp that never cross an agent boundary; at each
// change of agent the CTA reloads that agent's weight block into shared memory between two barriers (load(j)), so all
// warps use one block between two barriers.  body(ag0, na) runs one tile: rows pol_row<true>(ag0, r, N), r < na.
template <class Load, class Body>
__device__ __forceinline__ void pol_per_agent_tiles(int B, int N, int warp, int warps, Load load, Body body) {
    const int tpa = (B + 31) >> 5, ntiles = tpa * N;   // B * N < 2^31, as in pol_sample
    const int G = gridDim.x, b = blockIdx.x, q = ntiles / G, rm = ntiles % G;
    int k = b * q + (b < rm ? b : rm);
    const int k1 = k + q + (b < rm ? 1 : 0);
    for (int j = k / tpa; k < k1; ++j) {
        __syncthreads();   // every warp is done with the previous agent's block
        load(j);
        __syncthreads();
        const int kend = k1 < (j + 1) * tpa ? k1 : (j + 1) * tpa;
        for (; k < kend; k += warps) {
            if (k + warp < kend) {
                const int e0 = (k + warp - j * tpa) << 5;
                body((long long)e0 * N + j, B - e0 < 32 ? B - e0 : 32);
            }
        }
        k = kend;
    }
}

// bf16 feature row of agent `lane` (ENV:306-328 order: window, goal delta, pressure) into xs[lane][0 .. 16 KC1)
template <int KC1, bool PER_AGENT = false>
__device__ __forceinline__ void pol_feature_row(__nv_bfloat16 *xs, const uint32_t *raw, const float *goal_delta,
                                                const uint8_t *blocking_prev, int V2, long long ag0, int na, int lane,
                                                int N = 1) {
    constexpr int S1 = 16 * KC1 + 8;
    const int NW = (V2 + 3) >> 2;   // words of one agent's window
    uint2 *row = reinterpret_cast<uint2 *>(xs + lane * S1);
    const int off = lane * V2;
    for (int j = 0; j < 4 * KC1; ++j) {   // 4 cells -> 4 bf16 per trip; columns beyond the window are zero
        uint32_t w = 0;
        if (j < NW) {
            const int b = off + 4 * j;
            w = __funnelshift_r(raw[b >> 2], raw[(b >> 2) + 1], (b & 3) * 8);
            if (4 * j + 4 > V2) w &= (1u << (8 * (V2 - 4 * j))) - 1u;
        }
        const __nv_bfloat162 lo = __floats2bfloat162_rn((float)(w & 0xFFu), (float)((w >> 8) & 0xFFu));
        const __nv_bfloat162 hi = __floats2bfloat162_rn((float)((w >> 16) & 0xFFu), (float)(w >> 24));
        row[j] = make_uint2(*reinterpret_cast<const uint32_t *>(&lo), *reinterpret_cast<const uint32_t *>(&hi));
    }
    if (lane < na) {
        const float2 gd = reinterpret_cast<const float2 *>(goal_delta)[pol_row<PER_AGENT>(ag0, lane, N)];
        xs[lane * S1 + V2] = __float2bfloat16(gd.x);
        xs[lane * S1 + V2 + 1] = __float2bfloat16(gd.y);
        if (blocking_prev) xs[lane * S1 + V2 + 2] = __float2bfloat16((float)blocking_prev[pol_row<PER_AGENT>(ag0, lane, N)]);
    }
}

// the second ReLU layer of an m-tile: A fragments h1 (64 wide) -> A fragments h2 of the next GEMM (w2 [64][72], b2[64])
__device__ __forceinline__ void pol_layer2(const uint32_t (&h1)[POL_H / 16][4], const __nv_bfloat16 *w2, const float *b2,
                                           int g, int t, uint32_t (&h2)[POL_H / 16][4]) {
#pragma unroll
    for (int j = 0; j < POL_H / 8; ++j) {
        const float2 bb = *reinterpret_cast<const float2 *>(b2 + 8 * j + 2 * t);
        float d[4] = {bb.x, bb.y, bb.x, bb.y};
#pragma unroll
        for (int kk = 0; kk < POL_H / 16; ++kk) {
            const uint32_t *wb = reinterpret_cast<const uint32_t *>(w2 + (8 * j + g) * POL_W2_STRIDE + 16 * kk + 2 * t);
            mma_bf16_16816(d, h1[kk], wb[0], wb[4]);
        }
        h2[j >> 1][(j & 1) * 2 + 0] = pack_relu_bf16(d[0], d[1]);
        h2[j >> 1][(j & 1) * 2 + 1] = pack_relu_bf16(d[2], d[3]);
    }
}

// the two ReLU layers of the 16-row m-tile whose rows are row0 and row0 + 8: features xs -> A fragments of the next
// GEMM (bias = b1[64] b2[64])
template <int KC1>
__device__ __forceinline__ void pol_trunk(const __nv_bfloat16 *xs, const __nv_bfloat16 *w1, const __nv_bfloat16 *w2,
                                          const float *bias, int row0, int g, int t, uint32_t (&h2)[POL_H / 16][4]) {
    constexpr int S1 = 16 * KC1 + 8;
    // ------------------------------------------------------------ layer 1
    uint32_t af[KC1][4];
#pragma unroll
    for (int kk = 0; kk < KC1; ++kk) {
        const uint32_t *p0 = reinterpret_cast<const uint32_t *>(xs + row0 * S1 + 16 * kk + 2 * t);
        const uint32_t *p1 = reinterpret_cast<const uint32_t *>(xs + (row0 + 8) * S1 + 16 * kk + 2 * t);
        af[kk][0] = p0[0]; af[kk][1] = p1[0]; af[kk][2] = p0[4]; af[kk][3] = p1[4];
    }
    uint32_t h1[POL_H / 16][4];   // A fragments of layer 2
#pragma unroll
    for (int j = 0; j < POL_H / 8; ++j) {
        const float2 bb = *reinterpret_cast<const float2 *>(bias + 8 * j + 2 * t);
        float d[4] = {bb.x, bb.y, bb.x, bb.y};
#pragma unroll
        for (int kk = 0; kk < KC1; ++kk) {
            const uint32_t *wb = reinterpret_cast<const uint32_t *>(w1 + (8 * j + g) * S1 + 16 * kk + 2 * t);
            mma_bf16_16816(d, af[kk], wb[0], wb[4]);
        }
        h1[j >> 1][(j & 1) * 2 + 0] = pack_relu_bf16(d[0], d[1]);   // row g,   cols 8j + 2t, +1
        h1[j >> 1][(j & 1) * 2 + 1] = pack_relu_bf16(d[2], d[3]);   // row g+8
    }
    pol_layer2(h1, w2, bias + POL_H, g, t, h2);
}

// heads: columns 0..4 logits, 5 value (w3 [8][72], b3[8]) of the m-tile -> os[32][8]
__device__ __forceinline__ void pol_heads(const uint32_t (&hf)[POL_H / 16][4], const __nv_bfloat16 *w3, const float *b3,
                                          float *os, int row0, int g, int t) {
    const float2 bb = *reinterpret_cast<const float2 *>(b3 + 2 * t);
    float d[4] = {bb.x, bb.y, bb.x, bb.y};
#pragma unroll
    for (int kk = 0; kk < POL_H / 16; ++kk) {
        const uint32_t *wb = reinterpret_cast<const uint32_t *>(w3 + g * POL_W2_STRIDE + 16 * kk + 2 * t);
        mma_bf16_16816(d, hf[kk], wb[0], wb[4]);
    }
    *reinterpret_cast<float2 *>(os + row0 * 8 + 2 * t) = make_float2(d[0], d[1]);
    *reinterpret_cast<float2 *>(os + (row0 + 8) * 8 + 2 * t) = make_float2(d[2], d[3]);
}

// the policy kernels' draw of one agent from the unnormalised probabilities pr (sum = their sum): inverse CDF of one
// Philox word keyed by (key, env_id), counter (counter, agent)
__device__ __forceinline__ int pol_draw(unsigned long long key, long long env_id, unsigned long long counter, int agent,
                                        const float (&pr)[5], float sum) {
    Philox ph(key, env_id);
    const uint4 x = ph((uint32_t)counter, (uint32_t)(counter >> 32), (uint32_t)agent, 0x53414D50u /* "SAMP" */);
    const float u = ((float)(x.x >> 8) + 0.5f) * (1.0f / 16777216.0f) * sum;   // uniform in (0, sum)
    int act = 0;
    float cum = pr[0];
#pragma unroll
    for (int k = 1; k < 5; ++k) { if (u >= cum) act = k; cum += pr[k]; }
    return act;
}

// one agent per lane (call for lane < na): mask, stable softmax, then the action: with GREEDY the first index of the
// largest masked logit (torch.argmax's tie rule), otherwise an inverse-CDF draw from one Philox word keyed by
// (seed ^ tag, env_id_base + env), counter (counter, agent); writes the outputs of `a` that are not NULL.  GREEDY is a
// template parameter, not a runtime branch: the draw instantiation then compiles to the same code as a draw-only kernel
// (the LSTM kernel has no register to spare).
template <bool GREEDY, class Args>
__device__ __forceinline__ void pol_sample(const Args &a, const float *os, const uint32_t *rawm, int lane, long long ag, int N,
                                           unsigned long long tag) {
    const float4 o03 = *reinterpret_cast<const float4 *>(os + lane * 8);
    const float2 o45 = *reinterpret_cast<const float2 *>(os + lane * 8 + 4);
    float l[5] = {o03.x, o03.y, o03.z, o03.w, o45.x};
    if (!a.no_masking && a.action_mask) {   // logits + clamp(log(mask + 1e-6), FLOAT_MIN), action_mask_model.py:57-61
        const uint8_t *mk = reinterpret_cast<const uint8_t *>(rawm) + lane * 5;
#pragma unroll
        for (int k = 0; k < 5; ++k) l[k] += mk[k] ? 9.99999e-07f : -13.815511f;
    }
    float mx = l[0];
#pragma unroll
    for (int k = 1; k < 5; ++k) mx = fmaxf(mx, l[k]);
    float pr[5], sum = 0.f;
#pragma unroll
    for (int k = 0; k < 5; ++k) { pr[k] = __expf(l[k] - mx); sum += pr[k]; }
    int act = 0;
    if constexpr (GREEDY) {
        float best = l[0];
#pragma unroll
        for (int k = 1; k < 5; ++k) { if (l[k] > best) { best = l[k]; act = k; } }
    } else {
        const unsigned env = (unsigned)((unsigned long long)ag / (unsigned)N);   // B * N < 2^32 in any batch that fits a GPU
        const int agent = (int)(ag - (long long)env * N);
        act = pol_draw(a.seed ^ tag, a.env_id_base + env, a.counter, agent, pr, sum);
    }
    if (a.actions) a.actions[ag] = (int8_t)act;
    if (a.actions64) a.actions64[ag] = (long long)act;
    if (a.logp) a.logp[ag] = l[act] - mx - __logf(sum);
    if (a.value) a.value[ag] = o45.y;
    if (a.logits_out) {
#pragma unroll
        for (int k = 0; k < 5; ++k) a.logits_out[ag * 5 + k] = l[k];
    }
}

// KC1 = k16 chunks of the first layer (F <= 16 * KC1), W1 row stride = 16 * KC1 + 8; GREEDY = a.greedy (argmax, no draw);
// PER_AGENT: a.weights holds num_agents consecutive blocks and tile rows are one agent's (pol_per_agent_tiles)
template <int KC1, bool GREEDY, bool PER_AGENT = false>
__global__ void __launch_bounds__(256) mapf_policy_act_kernel(const mapf_policy_args a) {
    constexpr int S1 = 16 * KC1 + 8;   // bf16 row stride of the feature tile and of W1
    extern __shared__ __align__(16) unsigned char psm[];
    __nv_bfloat16 *w1 = reinterpret_cast<__nv_bfloat16 *>(psm);                 // [64][S1]
    __nv_bfloat16 *w2 = w1 + POL_H * S1;                                        // [64][72]
    __nv_bfloat16 *w3 = w2 + POL_H * POL_W2_STRIDE;                             // [8][72]: 5 logits, value, 2 zero rows
    float *bias = reinterpret_cast<float *>(w3 + 8 * POL_W2_STRIDE);            // b1[64] b2[64] b3[8]
    unsigned char *wsm0 = reinterpret_cast<unsigned char *>(bias + 2 * POL_H + 8);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = blockDim.x >> 5;
    if constexpr (!PER_AGENT) {   // weights: already bf16 and padded on the host side (mapf_policy_pack_weights)
        const uint4 *src = reinterpret_cast<const uint4 *>(a.weights);
        uint4 *dst = reinterpret_cast<uint4 *>(psm);
        const int n16 = (int)((wsm0 - psm) >> 4);
        for (int i = tid; i < n16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
    }
    const int V2 = a.v2, F = a.feature_dim, N = a.num_agents;
    unsigned char *wsm = wsm0 + warp * pol_warp_bytes(KC1, V2);
    __nv_bfloat16 *xs = reinterpret_cast<__nv_bfloat16 *>(wsm);                 // [32][S1] bf16 features
    uint32_t *raw = reinterpret_cast<uint32_t *>(wsm + 32 * S1 * 2);            // the tile's window bytes, as loaded
    uint32_t *rawm = reinterpret_cast<uint32_t *>(wsm + 32 * S1 * 2 + pol_raw_bytes(V2));   // 32 x 5 mask bytes
    float *os = reinterpret_cast<float *>(wsm + 32 * S1 * 2 + pol_raw_bytes(V2) + 160);     // [32][8] head outputs
    const int g = lane >> 2, t = lane & 3;
    auto tile_body = [&](const long long ag0, const int na) {
        if constexpr (PER_AGENT) pol_gather_tile(a.local_obs, a.action_mask, a.action_mask_out, V2, ag0, N, na, raw, rawm, lane);
        else pol_load_tile(a.local_obs, a.action_mask, a.action_mask_out, V2, ag0, na, raw, rawm, lane);
        __syncwarp();
        pol_feature_row<KC1, PER_AGENT>(xs, raw, a.goal_delta, a.blocking_prev, V2, ag0, na, lane, N);
        if (a.features_out) {   // float32 feature block for the learner (optional)
            float *fo = a.features_out + ag0 * F;
            const uint8_t *rb = reinterpret_cast<const uint8_t *>(raw);
            for (int i = lane; i < na * F; i += 32) {
                const int r = i / F, c = i - r * F;
                float v;
                if (c < V2) v = (float)rb[r * V2 + c];
                else if (c < V2 + 2) v = a.goal_delta[pol_row<PER_AGENT>(ag0, r, N) * 2 + (c - V2)];
                else v = (float)a.blocking_prev[pol_row<PER_AGENT>(ag0, r, N)];
                if constexpr (PER_AGENT) a.features_out[pol_row<true>(ag0, r, N) * F + c] = v;
                else fo[i] = v;
            }
        }
        __syncwarp();
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int row0 = 16 * mt + g;   // this lane's rows: row0 and row0 + 8
            uint32_t h2[POL_H / 16][4];
            pol_trunk<KC1>(xs, w1, w2, bias, row0, g, t, h2);
            pol_heads(h2, w3, bias + 2 * POL_H, os, row0, g, t);
        }
        __syncwarp();
        if (lane < na) pol_sample<GREEDY>(a, os, rawm, lane, pol_row<PER_AGENT>(ag0, lane, N), N, 0x504F4C49ull /* "POLI" */);
        __syncwarp();
    };
    if constexpr (PER_AGENT) {
        const int n16 = (int)((wsm0 - psm) >> 4);   // 16-byte words of one agent's block
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

// Generalised advantage estimation (ppo.py:104-117 hyper-parameters are arguments): adv[t] = delta_t + gamma * lam *
// nd_t * adv[t+1], delta_t = r_t + gamma * V_{t+1} * nd_t - V_t, nd_t = 1 - done_t; one thread per (env, agent).
__global__ void mapf_gae_kernel(const float *rewards, const float *values, const uint8_t *dones, const float *last_value,
                                float *adv, float *ret, int T, long long BN, int N, float gamma, float lam) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= BN) return;
    const long long env = i / N, B = BN / N;
    float running = 0.f, next_value = last_value[i];
    for (int t = T - 1; t >= 0; --t) {
        const float nd = dones[(long long)t * B + env] ? 0.f : 1.f;
        const float v = values[(long long)t * BN + i];
        const float delta = rewards[(long long)t * BN + i] + gamma * next_value * nd - v;
        running = delta + gamma * lam * nd * running;
        adv[(long long)t * BN + i] = running;
        ret[(long long)t * BN + i] = running + v;
        next_value = v;
    }
}

}  // namespace mapf
