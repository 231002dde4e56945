// mapf_vtrace_kernel.cuh -- V-trace targets (IMPALA's off-policy correction) as a backwards scan, one thread per
// processed column; the C ABI is mapf_vtrace (include/mapf_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mapf_b200.h"

namespace mapf {

// Steps whose loads are issued together ahead of the recurrence: none of a step's inputs depends on the running
// value, so a column pays T dependent FMAs and about T / VTRACE_UNROLL memory round trips instead of T.
constexpr int VTRACE_UNROLL = 8;
constexpr int VTRACE_THREADS = 256;

// Processed column m is batch column col = columns[m] (or m): env col / num_agents, agent col % num_agents.  The
// batch-layout inputs (rewards, behaviour log-probabilities, dones, bootstrap value) are read at that column, the
// minibatch-layout ones (target log-probabilities, values) and the outputs at m.  With d_t the episode end of step t
// and V_T the bootstrap value:
//   rho_t = exp(pi_t - mu_t), rho_bar_t = min(clip_rho, rho_t), c_t = min(1, rho_t), rho_pg_t = min(clip_pg_rho, rho_t)
//   disc_t = gamma * (1 - d_t), delta_t = rho_bar_t * (r_t + disc_t * V_{t+1} - V_t)
//   acc_T = 0, acc_t = delta_t + disc_t * c_t * acc_{t+1}, vs_t = V_t + acc_t
//   pg_adv_t = rho_pg_t * (r_t + disc_t * vs_{t+1} - V_t), vs_T = V_T
// A column id outside [0, num_columns) writes NaN to the column's outputs and reads no input.
__global__ void __launch_bounds__(VTRACE_THREADS) mapf_vtrace_kernel(const mapf_vtrace_args a) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= a.M) return;
    const long long NC = a.num_columns, M = a.M;
    const long long col = a.columns ? a.columns[m] : m;
    const int T = a.T;
    if (col < 0 || col >= NC) {
        for (int t = 0; t < T; ++t) {
            a.vs[(long long)t * M + m] = __int_as_float(0x7fc00000);
            a.pg_advantages[(long long)t * M + m] = __int_as_float(0x7fc00000);
        }
        return;
    }
    const long long B = NC / a.num_agents, env = col / a.num_agents;
    const float gamma = a.gamma, clip_rho = a.clip_rho, clip_pg_rho = a.clip_pg_rho;
    float v_next = a.bootstrap_value[col], vs_next = v_next, acc = 0.f;
    for (int t0 = T - 1; t0 >= 0; t0 -= VTRACE_UNROLL) {
        float r[VTRACE_UNROLL], mu[VTRACE_UNROLL], pi[VTRACE_UNROLL], v[VTRACE_UNROLL];
        uint8_t d[VTRACE_UNROLL];
#pragma unroll
        for (int k = 0; k < VTRACE_UNROLL; ++k) {
            const long long t = t0 - k;
            if (t >= 0) {
                r[k] = a.rewards[t * NC + col];
                mu[k] = a.behaviour_logp[t * NC + col];
                d[k] = a.dones[t * B + env];
                pi[k] = a.target_logp[t * M + m];
                v[k] = a.values[t * M + m];
            }
        }
#pragma unroll
        for (int k = 0; k < VTRACE_UNROLL; ++k) {
            const long long t = t0 - k;
            if (t >= 0) {
                const float rho = expf(pi[k] - mu[k]);
                const float rho_bar = fminf(clip_rho, rho), c = fminf(1.f, rho), rho_pg = fminf(clip_pg_rho, rho);
                const float disc = gamma * (1.f - (d[k] ? 1.f : 0.f));
                const float delta = rho_bar * (r[k] + disc * v_next - v[k]);
                acc = delta + disc * c * acc;
                const float vs = v[k] + acc;
                a.vs[t * M + m] = vs;
                a.pg_advantages[t * M + m] = rho_pg * (r[k] + disc * vs_next - v[k]);
                v_next = v[k];
                vs_next = vs;
            }
        }
    }
}

}  // namespace mapf
