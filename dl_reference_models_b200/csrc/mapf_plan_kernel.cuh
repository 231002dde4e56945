// Prioritized space-time planner (DESIGN.md §7 N4b): agents plan in index order 0..N-1 under the env's own move rule,
// each by a bit-parallel wavefront over (cell, t) and a backtrack, then reserve their path for the agents after them.
//
// The env moves agents in index order (ENV:502-526): agent i's move into cell c fails when c holds a lower-index agent
// at its new position or a higher-index agent at its old position.  With R_t = the cells the agents planned so far
// hold at time t (R_{H+1} = R_H), agent i may stand on cell c at time t >= 1 iff
//   c in W_t = free & ~R_t & ~R_{t+1} & (t == 1 ? ~(starts of the agents after i) : all)
// (~R_t: vertex; ~R_{t+1}: a lower index cannot enter a cell a higher one still holds, which also rules out swaps; the
// unplanned agents stand on their starts at t = 0).  Agents stay on their goal once there, so agent i arrives at the
// first t of its wavefront with its goal outside R_t' for every t' >= t; from then on it reserves its goal up to H.
// An agent with no arrival by H (or an unreachable goal) gets arrival -1 and reserves its start for every t; the env's
// status is then 0 and the plan carries no validity guarantee.
//
// One warp per env, one lane per map row (R, C <= 32): lane r's word is row r's column mask.  Forward:
//   F_0 = {start};  F_t = (F | F<<1 | F>>1 | shfl_up(F) | shfl_down(F)) & W_t
// F_t is stored for the backtrack, which walks from (goal, t_a) back to t = 0 taking at every step the first
// predecessor in the action order NO_OP, UP, RIGHT, DOWN, LEFT (actions.py), so plans are deterministic.
//
// Windowed mode (WINDOWED = true, mapf_plan_windowed; DESIGN.md §7 N4c): the same rule with H read as the window W,
// for rolling-horizon replanning from mid-episode states, where arrival within W is not required.  The target is the
// goal if the distance table reaches it from the start (!= 255), else the start itself.  An agent whose target is its
// goal arrives as above (first t <= W with the goal in F_t and t >= max(d, last[goal] + 1)) and holds it to W.  An
// agent with no arrival searches on to t = W and ends on the cell of F_W with the smallest (d(target, cell), cell
// index), each lane scanning its row word against the target's distance-table row and one warp min-reduce picking
// the key; it backtracks from (end cell, W), reserves that path, last[end] = W, and gets arrival -1.  Only a wavefront
// that empties by W (or a start / goal off the map) fails as above.  status = 1 iff every agent got a path.
//
// Per-env workspace (mapf_plan_workspace_bytes): R[(H+1) * rows] and F[(H+1) * rows] uint32 row words, then
// last[R*C] int16 = the last t at which a planned agent holds the cell (-1 = never), which gives the arrival bound
// last[goal] + 1 with one load.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "mapf_kernels.cuh"

namespace mapf {

constexpr int PLAN_THREADS = 128;

__host__ __device__ inline int64_t plan_env_words(int rows, int cols, int horizon) {
    // two [(H+1) x rows] word planes + the int16 last-use table, padded to a whole number of 16-byte units
    const int64_t words = 2LL * (horizon + 1) * rows + (rows * cols + 1) / 2;
    return (words + 3) & ~3LL;
}

template <bool WINDOWED>
__global__ void __launch_bounds__(PLAN_THREADS) mapf_plan_kernel(
    const uint32_t *__restrict__ free_bits, int R, int C, long long B, int N, int H,
    const uint32_t *__restrict__ starts, const uint32_t *__restrict__ goals, const uint8_t *__restrict__ dist,
    uint32_t *__restrict__ ws, long long env_words, int8_t *__restrict__ actions, int16_t *__restrict__ arrival,
    uint8_t *__restrict__ status) {
    const unsigned full = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int cells = R * C;
    uint32_t freerow = 0;
    if (lane < R) {
        const int b0 = lane * C;
        const uint64_t w = (uint64_t)free_bits[b0 >> 5] |
                           ((uint64_t)(((b0 >> 5) + 1) * 32 < cells + 32 ? free_bits[(b0 >> 5) + 1] : 0u) << 32);
        freerow = (uint32_t)(w >> (b0 & 31)) & (C >= 32 ? full : ((1u << C) - 1u));
    }
    const long long warps = (long long)gridDim.x * (PLAN_THREADS / 32);
    for (long long b = (long long)blockIdx.x * (PLAN_THREADS / 32) + (threadIdx.x >> 5); b < B; b += warps) {
        uint32_t *Rw = ws + b * env_words;
        uint32_t *Fw = Rw + (long long)(H + 1) * R;
        int16_t *last = reinterpret_cast<int16_t *>(Fw + (long long)(H + 1) * R);
        for (int i = lane; i < (H + 1) * R; i += 32) Rw[i] = 0u;
        for (int i = lane; i < cells; i += 32) last[i] = -1;
        // lane a holds agent a's start and goal; an agent whose cell lies off the map neither plans nor reserves
        const uint32_t my_s = lane < N ? starts[b * N + lane] : 0u, my_g = lane < N ? goals[b * N + lane] : 0u;
        const bool my_ok = lane < N && prow(my_s) >= 0 && prow(my_s) < R && pcol(my_s) >= 0 && pcol(my_s) < C &&
                           prow(my_g) >= 0 && prow(my_g) < R && pcol(my_g) >= 0 && pcol(my_g) < C;
        const unsigned okmask = __ballot_sync(full, my_ok);
        // my row's starts of the agents not planned yet (the t = 1 term of W)
        uint32_t hi = 0u;
        for (int a = 0; a < N; ++a) {
            const uint32_t s = __shfl_sync(full, my_s, a);
            if ((okmask >> a & 1u) && prow(s) == lane) hi |= 1u << pcol(s);
        }
        __syncwarp();
        bool all_ok = true;
        for (int i = 0; i < N; ++i) {
            const uint32_t s = __shfl_sync(full, my_s, i), g = __shfl_sync(full, my_g, i);
            int8_t *act = actions + b * N + i;              // act[t * B * N]
            const long long tstride = B * N;
            if (!(okmask >> i & 1u)) {
                for (int t = lane; t < H; t += 32) act[t * tstride] = 0;
                if (lane == 0) arrival[b * N + i] = -1;
                all_ok = false;
                continue;
            }
            const int sr = prow(s), sc = pcol(s);
            int gr = prow(g), gc = pcol(g);
            if (lane == sr) hi &= ~(1u << sc);
            const int d = dist[(long long)(gr * C + gc) * cells + sr * C + sc];
            const int lo = last[gr * C + gc] + 1;
            // windowed: an unreachable goal makes the start the target, which is never arrived at
            const int tmin = WINDOWED && d == 255 ? H + 1 : (d > lo ? d : lo);
            int ta = -1;
            bool end_cell = false;   // windowed: the path ends at (end cell, W) without an arrival
            if (WINDOWED || (d != 255 && tmin <= H)) {
                uint32_t F = lane == sr ? 1u << sc : 0u;
                if (lane < R) Fw[lane] = F;
                if (tmin == 0) {
                    ta = 0;
                } else {
                    // R_t and R_{t+1} of step t, the load of R_{t+2} issued one step ahead
                    uint32_t rt = lane < R ? Rw[R + lane] : 0u;
                    uint32_t rn = lane < R ? Rw[(H >= 2 ? 2 : 1) * R + lane] : 0u;
                    for (int t = 1; t <= H; ++t) {
                        const int tn2 = t + 2 <= H ? t + 2 : H;
                        const uint32_t rnn = lane < R ? Rw[tn2 * R + lane] : 0u;
                        const uint32_t up = __shfl_up_sync(full, F, 1), dn = __shfl_down_sync(full, F, 1);
                        uint32_t nf = F | (F << 1) | (F >> 1) | (lane > 0 ? up : 0u) | (lane < 31 ? dn : 0u);
                        uint32_t w = freerow & ~rt & ~rn;
                        if (t == 1) w &= ~hi;
                        F = nf & w;
                        if (lane < R) Fw[t * R + lane] = F;
                        const uint32_t at_goal = __shfl_sync(full, F, gr) >> gc & 1u;
                        if (t >= tmin && at_goal) { ta = t; break; }
                        if (!__any_sync(full, F != 0u)) break;
                        rt = rn;
                        rn = rnn;
                    }
                }
                if (WINDOWED && ta < 0 && __any_sync(full, F != 0u)) {
                    // F = F_W: the end cell is its cell of least (d(target, cell), cell index)
                    const uint8_t *drow = dist + (long long)(d == 255 ? sr * C + sc : gr * C + gc) * cells;
                    unsigned key = 0xFFFFFFFFu;
                    for (uint32_t f = F; f; f &= f - 1) {
                        const unsigned cell = (unsigned)(lane * C + __ffs(f) - 1);
                        const unsigned k = (unsigned)drow[cell] << 10 | cell;
                        key = k < key ? k : key;
                    }
                    key = __reduce_min_sync(full, key) & 1023u;
                    gr = (int)key / C;
                    gc = (int)key % C;
                    ta = H;
                    end_cell = true;
                }
            }
            if (lane == 0) arrival[b * N + i] = (int16_t)(end_cell ? -1 : ta);
            __syncwarp();
            if (ta < 0) {
                all_ok = false;
                for (int t = lane; t <= H; t += 32) Rw[t * R + sr] |= 1u << sc;
                for (int t = lane; t < H; t += 32) act[t * tstride] = 0;
                if (lane == 0) last[sr * C + sc] = (int16_t)H;
            } else {
                for (int t = ta + 1 + lane; t <= H; t += 32) Rw[t * R + gr] |= 1u << gc;
                for (int t = ta + lane; t < H; t += 32) act[t * tstride] = 0;
                // backtrack: F_{t-1}'s row words are loaded by every lane (one coalesced load), the three rows
                // around the current cell taken by shuffles; the next step's load is issued one step ahead
                int r = gr, c = gc;
                uint32_t f = (ta >= 1 && lane < R) ? Fw[(ta - 1) * R + lane] : 0u;
                for (int t = ta; t >= 1; --t) {
                    const uint32_t fnext = (t >= 2 && lane < R) ? Fw[(t - 2) * R + lane] : 0u;
                    const uint32_t fm = __shfl_sync(full, f, r > 0 ? r - 1 : 0);
                    const uint32_t f0 = __shfl_sync(full, f, r);
                    const uint32_t fp = __shfl_sync(full, f, r + 1 < 32 ? r + 1 : 31);
                    int a, pr = r, pc = c;
                    if (f0 >> c & 1u) { a = 0; }                                             // NO_OP from (r, c)
                    else if (r + 1 < R && (fp >> c & 1u)) { a = 1; pr = r + 1; }              // UP from (r+1, c)
                    else if (c > 0 && (f0 >> (c - 1) & 1u)) { a = 2; pc = c - 1; }            // RIGHT from (r, c-1)
                    else if (r > 0 && (fm >> c & 1u)) { a = 3; pr = r - 1; }                  // DOWN from (r-1, c)
                    else { a = 4; pc = c + 1; }                                               // LEFT from (r, c+1)
                    if (lane == 0) {
                        Rw[t * R + r] |= 1u << c;
                        if (last[r * C + c] < t) last[r * C + c] = (int16_t)t;
                        act[(long long)(t - 1) * tstride] = (int8_t)a;
                    }
                    r = pr;
                    c = pc;
                    f = fnext;
                }
                if (lane == 0) {
                    Rw[r] |= 1u << c;   // the start at t = 0
                    if (last[r * C + c] < 0) last[r * C + c] = 0;
                    last[gr * C + gc] = (int16_t)H;
                }
            }
            __syncwarp();
        }
        if (lane == 0) status[b] = all_ok ? 1 : 0;
    }
}

}  // namespace mapf
