// mapf_eval_kernel.cuh -- per-step bookkeeping of the batched evaluator (evaluate.py, main.py:test_trained_model with
// one episode per env) in one launch, leaving the host one 4-byte count to read per step.
//   * one lane group per env, one lane per agent: a group is P lanes, P = N rounded up to a power of two, and a warp
//     takes 32 / P envs at a time (two at N = 16), so a warp walks fewer envs one after the other; the agent returns
//     are one coalesced f64 row per env, the episode return is a reduction of the same values inside the group
//     (rewards are whole numbers of halves, so the f64 sums are exact in any order and equal to the sequential ones);
//   * an inactive env costs one byte read;
//   * the envs still active after the step are counted per warp, reduced per block and added with one atomic per block
//     into active_count[step & 1]; block 0 zeroes the other word, the one the next step counts into.
// mapf_cte_eval_accumulate_kernel does the same for the single-agent (CTE) view, one thread per env.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "mapf_kernels.cuh"

namespace mapf {

constexpr int EVAL_THREADS = 256;

__global__ void __launch_bounds__(EVAL_THREADS, 8) mapf_eval_accumulate_kernel(const mapf_eval_args a, int P) {
    __shared__ unsigned warp_still[EVAL_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5, N = a.num_agents;
    const int G = 32 / P, grp = lane / P, sub = lane - grp * P;   // envs per warp, this lane's env and agent
    const int slot = (int)(a.step & 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) a.active_count[slot ^ 1] = 0u;
    unsigned still = 0;
#pragma unroll 1
    for (long long b0 = ((long long)blockIdx.x * warps + warp) * G; b0 < a.num_envs; b0 += (long long)gridDim.x * warps * G) {
        const long long b = b0 + grp;
        const bool act = b < a.num_envs && a.active[b];
        double r = 0.0;
        if (act && sub < N) {
            const long long i = b * N + sub;
            r = (double)a.reward[i];
            a.agent_reward[i] += r;                                   // main.py:262
        }
        for (int o = P >> 1; o; o >>= 1) r += __shfl_xor_sync(0xFFFFFFFFu, r, o, P);
        if (!act) continue;
        for (int w = sub; w < MAPF_INFO_WORDS; w += P) a.last_info[b * MAPF_INFO_WORDS + w] = a.info[b * MAPF_INFO_WORDS + w];
        if (sub == 0) {
            a.episode_reward[b] += r;                                 // main.py:251
            a.timesteps[b] += 1;
            const bool term = a.terminated[b] != 0, trunc = a.truncated[b] != 0;
            if (term || trunc) {
                a.success[b] = (uint8_t)(term && !trunc);             // main.py:294
                a.active[b] = 0;
            } else {
                ++still;
            }
        }
    }
    still = __reduce_add_sync(0xFFFFFFFFu, still);
    if (lane == 0) warp_still[warp] = still;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned s = 0;
        for (int w = 0; w < warps; ++w) s += warp_still[w];
        if (s) atomicAdd(a.active_count + slot, s);
    }
}

// The CTE view's bookkeeping (mapf_cte_eval_accumulate), one thread per env: the view has one f64 reward per env, so
// there is nothing to reduce.  Each env adds its rewards in step order, the same sequence of f64 additions as a Python
// `total += reward` loop.  The heat-map is counted before this launch by mapf_occupancy_kernel.  The block-count tail
// is mapf_eval_accumulate_kernel's, written out again: shared as a device function it changed that kernel's code.
__global__ void __launch_bounds__(EVAL_THREADS) mapf_cte_eval_accumulate_kernel(const mapf_cte_eval_args a) {
    __shared__ unsigned warp_still[EVAL_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int slot = (int)(a.step & 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) a.active_count[slot ^ 1] = 0u;
    unsigned still = 0;
#pragma unroll 1
    for (long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x; b < a.num_envs; b += (long long)gridDim.x * blockDim.x) {
        if (!a.active[b]) continue;
        a.episode_reward[b] += a.reward[b];
        a.timesteps[b] += 1;
#pragma unroll
        for (int w = 0; w < MAPF_CTE_INFO_WORDS; ++w) a.last_info[b * MAPF_CTE_INFO_WORDS + w] = a.info[b * MAPF_CTE_INFO_WORDS + w];
        const bool term = a.terminated[b] != 0, trunc = a.truncated[b] != 0;
        if (term || trunc) {
            a.success[b] = (uint8_t)(term && !trunc);
            a.active[b] = 0;
        } else {
            ++still;
        }
    }
    still = __reduce_add_sync(0xFFFFFFFFu, still);
    if (lane == 0) warp_still[warp] = still;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned s = 0;
        for (int w = 0; w < warps; ++w) s += warp_still[w];
        if (s) atomicAdd(a.active_count + slot, s);
    }
}

}  // namespace mapf
