// mapf_replay_kernel.cuh -- DQN's prioritized replay (RLlib's PrioritizedReplayBuffer, the reference's
// src/agents/dqn.py default, SURVEY §2 row 6) as a sum tree on the device; the C ABI is mapf_replay_advance /
// mapf_replay_sample / mapf_replay_update (include/mapf_b200.h).
//
// The tree is an implicit binary heap over L = N' K' B' leaves ordered (agent, slot, env), each of N, K, B padded to a
// power of two: node i has children 2i, 2i + 1, node L + l is leaf l.  One (agent, slot) pair is the subtree of B'
// leaves under node (L + (j K' + k) B') / B', one agent the subtree under node N' + j.  Leaves are float32 p^alpha,
// internal sums float64 (descending 2^26 leaves never lands on a zero leaf through rounding), internal minimums
// float32 over the nonzero leaves (+inf when there are none).  Every node is recomputed as a function of its two
// children only, so the tree's contents do not depend on thread order.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/mapf_b200.h"
#include "mapf_kernels.cuh"

namespace mapf {

constexpr int REPLAY_CHUNK = 1024;     // leaves (and threads) of one block of the advance kernel
constexpr int REPLAY_THREADS = 1024;   // threads of the one-block kernels

__host__ __device__ inline int replay_log2_ceil(long long x) {
    int l = 0;
    while ((1ll << l) < x) ++l;
    return l;
}

struct ReplayLayout {
    int lb, lk, ln;   // log2 of B', K', N'
    long long L;      // leaves = N' K' B'
    __host__ __device__ explicit ReplayLayout(const mapf_replay_tree &t)
        : lb(replay_log2_ceil(t.num_envs)), lk(replay_log2_ceil(t.capacity)), ln(replay_log2_ceil(t.num_agents)),
          L(1ll << (lb + lk + ln)) {}
    __device__ long long leaf(int j, int k, long long b) const { return ((long long)j << (lk + lb)) + ((long long)k << lb) + b; }
};

// p^alpha; alpha 1 (proportional) and 0 (uniform) exactly, as torch's pow takes them
__device__ __forceinline__ float replay_pow(float p, float alpha) {
    return alpha == 1.f ? p : alpha == 0.f ? 1.f : powf(p, alpha);
}

// the sum / minimum of heap node c (an internal node or a leaf)
__device__ __forceinline__ double replay_sum(const mapf_replay_tree &t, long long L, long long c) {
    return c < L ? t.sums[c] : (double)t.leaves[c - L];
}
__device__ __forceinline__ float replay_min(const mapf_replay_tree &t, long long L, long long c) {
    if (c < L) return t.mins[c];
    const float v = t.leaves[c - L];
    return v > 0.f ? v : CUDART_INF_F;
}
__device__ __forceinline__ void replay_refresh_node(const mapf_replay_tree &t, long long L, long long n) {
    t.sums[n] = replay_sum(t, L, 2 * n) + replay_sum(t, L, 2 * n + 1);
    t.mins[n] = fminf(replay_min(t, L, 2 * n), replay_min(t, L, 2 * n + 1));
}

// Advance, part 1: block (which, j, chunk) writes REPLAY_CHUNK (or B') leaves of agent j in slot `complete`
// (which = 0: max_priority^alpha for env < B) or `clear` (which = 1: 0), then the nodes of its chunk's subtree, level
// by level in shared memory.
__global__ void __launch_bounds__(REPLAY_CHUNK) mapf_replay_advance_kernel(const mapf_replay_advance_args a) {
    __shared__ double s_sum[REPLAY_CHUNK];
    __shared__ float s_min[REPLAY_CHUNK];
    const ReplayLayout lay(a.tree);
    const long long Bp = 1ll << lay.lb;
    const int CH = (int)(Bp < REPLAY_CHUNK ? Bp : REPLAY_CHUNK);
    const int chunks = (int)(Bp / CH), N = a.tree.num_agents;
    const int which = blockIdx.x / (N * chunks), rest = blockIdx.x - which * N * chunks;
    const int j = rest / chunks, c = rest - j * chunks;
    const int i = threadIdx.x;
    const long long leaf0 = lay.leaf(j, which ? a.clear : a.complete, (long long)c * CH);
    if (i < CH) {
        const long long b = (long long)c * CH + i;
        const float v = (which == 0 && b < a.tree.num_envs) ? replay_pow(*a.tree.max_priority, a.alpha) : 0.f;
        a.tree.leaves[leaf0 + i] = v;
        s_sum[i] = (double)v;
        s_min[i] = v > 0.f ? v : CUDART_INF_F;
    }
    for (int h = CH >> 1, lev = 1; h >= 1; h >>= 1, ++lev) {
        double sv = 0.0;
        float mv = 0.f;
        __syncthreads();
        if (i < h) {
            sv = s_sum[2 * i] + s_sum[2 * i + 1];
            mv = fminf(s_min[2 * i], s_min[2 * i + 1]);
        }
        __syncthreads();
        if (i < h) {
            s_sum[i] = sv;
            s_min[i] = mv;
            const long long n = ((lay.L + leaf0) >> lev) + i;
            a.tree.sums[n] = sv;
            a.tree.mins[n] = mv;
        }
    }
}

// Advance, part 2 (one block): the nodes above the chunks' subtrees, level by level up to the root: per level, for
// each of the 2N (slot, agent) ranges, the nodes above that range.
__global__ void __launch_bounds__(REPLAY_THREADS) mapf_replay_advance_top_kernel(const mapf_replay_advance_args a) {
    const ReplayLayout lay(a.tree);
    const int D = lay.lb + lay.lk + lay.ln, N = a.tree.num_agents;
    const int lev0 = (lay.lb < 10 ? lay.lb : 10) + 1;   // the levels part 1 wrote: log2(min(B', REPLAY_CHUNK))
    for (int lev = lev0; lev <= D; ++lev) {
        const long long per = lev < lay.lb ? (1ll << (lay.lb - lev)) : 1;   // nodes above one range at this level
        for (long long w = threadIdx.x; w < 2ll * N * per; w += blockDim.x) {
            const int r = (int)(w / per), j = r % N;
            const long long first = (lay.L + lay.leaf(j, r < N ? a.complete : a.clear, 0)) >> lev;
            replay_refresh_node(a.tree, lay.L, first + (w - r * per));
        }
        __syncthreads();
    }
}

// One thread per draw: a uniform u in [0, 1) (53 bits of one Philox block), target u * total, descent to the first
// leaf whose prefix sum exceeds the target (a running prefix `base`, so with integer-valued priorities every
// comparison is exact and equals a search of the f64 cumulative sum); a right subtree with a zero sum is never
// entered, so a draw always ends on a nonzero leaf.
__global__ void __launch_bounds__(256) mapf_replay_sample_kernel(const mapf_replay_sample_args a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.M) return;
    const ReplayLayout lay(a.tree);
    const mapf_replay_tree &t = a.tree;
    const long long root = a.per_agent ? (1ll << lay.ln) + i % t.num_agents : 1;
    const double total = replay_sum(t, lay.L, root);
    Philox ph(a.seed ^ 0x50525053ull /* "PRPS" */, i);
    const uint4 x = ph((uint32_t)a.counter, (uint32_t)(a.counter >> 32), 0u, 0u);
    const double u = (double)(((unsigned long long)x.x << 21) | (x.y >> 11)) * (1.0 / 9007199254740992.0);
    if (a.uniforms) a.uniforms[i] = u;
    if (!(total > 0.0)) {
        a.indices[i] = -1;
        a.weights[i] = 0.f;
        return;
    }
    const double target = u * total;
    double base = 0.0;
    long long n = root;
    while (n < lay.L) {
        const double lv = replay_sum(t, lay.L, 2 * n);
        if (target < base + lv || !(replay_sum(t, lay.L, 2 * n + 1) > 0.0)) {
            n = 2 * n;
        } else {
            base += lv;
            n = 2 * n + 1;
        }
    }
    const long long leaf = n - lay.L;
    const int j = (int)(leaf >> (lay.lk + lay.lb));
    const long long k = (leaf >> lay.lb) & ((1ll << lay.lk) - 1), b = leaf & ((1ll << lay.lb) - 1);
    a.indices[i] = (k * t.num_envs + b) * t.num_agents + j;
    const double p_min = (double)replay_min(t, lay.L, root);
    a.weights[i] = (float)pow((double)t.leaves[leaf] / p_min, -(double)a.beta);
}

// the leaf of flat transition index idx = (k B + b) N + j
__device__ __forceinline__ long long replay_leaf_of(const ReplayLayout &lay, long long idx, long long BN, int N) {
    const long long k = idx / BN, r = idx - k * BN, b = r / N;
    return lay.leaf((int)(r - b * N), (int)k, b);
}

// One block: (A) mark the in-range targeted leaves that hold a transition (nonzero) with the smallest positive float;
// (B) atomicMax of the new value (|delta| + 1e-6)^alpha into each marked leaf (positive floats order as their bits),
// so among duplicates the largest value is kept whatever the thread order, and of |delta| + 1e-6 into max_priority;
// (C) the ancestors, level by level.
__global__ void __launch_bounds__(REPLAY_THREADS, 1) mapf_replay_update_kernel(const mapf_replay_update_args a) {
    const ReplayLayout lay(a.tree);
    const mapf_replay_tree &t = a.tree;
    const long long BN = (long long)t.num_envs * t.num_agents, total = BN * t.capacity;
    const int D = lay.lb + lay.lk + lay.ln;
    for (long long i = threadIdx.x; i < a.M; i += blockDim.x) {
        const long long idx = a.indices[i];
        if (idx < 0 || idx >= total) continue;
        const long long l = replay_leaf_of(lay, idx, BN, t.num_agents);
        if (t.leaves[l] > 0.f) t.leaves[l] = __int_as_float(1);
    }
    __syncthreads();
    for (long long i = threadIdx.x; i < a.M; i += blockDim.x) {
        const long long idx = a.indices[i];
        if (idx < 0 || idx >= total) continue;
        const long long l = replay_leaf_of(lay, idx, BN, t.num_agents);
        if (!(t.leaves[l] > 0.f)) continue;
        const float p = a.td_abs[i] + 1e-6f;
        atomicMax(reinterpret_cast<int *>(t.leaves + l), __float_as_int(replay_pow(p, a.alpha)));
        atomicMax(reinterpret_cast<int *>(t.max_priority), __float_as_int(p));
    }
    __syncthreads();
    for (int lev = 1; lev <= D; ++lev) {
        for (long long i = threadIdx.x; i < a.M; i += blockDim.x) {
            const long long idx = a.indices[i];
            if (idx < 0 || idx >= total) continue;
            const long long l = replay_leaf_of(lay, idx, BN, t.num_agents);
            if (!(t.leaves[l] > 0.f)) continue;
            replay_refresh_node(t, lay.L, (lay.L + l) >> lev);
        }
        __syncthreads();
    }
}

}  // namespace mapf
