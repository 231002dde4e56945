// Conflict-based search (CBS, Sharon et al. 2015) under the env's own move rule (DESIGN.md §7 N4d): plans with the least
// sum of arrivals (SOC) within H, for small agent counts, one warp per env.
//
// A joint plan p_i(t), t = 0..H, every agent on its goal from its arrival on, replays through mapf_step without a
// failed move iff for every t < H and every pair a != b: p_a(t+1) != p_b(t+1) (vertex), and if a moves and b > a then
// p_a(t+1) != p_b(t) (following: agents move in index order, so a lower index cannot enter a cell a higher index still
// holds; this also rules out swaps).  A vertex conflict at (c, t+1) splits into the constraints (a, c, t+1) / (b, c,
// t+1), a following conflict into (a, c, t+1) / (b, c, t).
//
// Low level (one agent under its constraints): F_0 = {start} (none if (start, 0) is constrained), F_t = step(F_{t-1})
// & free & ~Cons_t; arrival = the first t <= H with the goal in F_t and t >= L = 1 + the last constrained t of the goal
// (0 if none), t = 0 iff start = goal and L = 0; none when F empties or t passes H.  Backtrack with mapf_plan_kernel's
// tie rule (first predecessor in the order NO_OP, UP, RIGHT, DOWN, LEFT).  Cost = arrival.
// First conflict of a node: t = 0, 1, ..., within a t vertex conflicts first (lowest a, then lowest b), then following
// conflicts (lowest a).  High level: pop the open node of least (SOC, id); a conflict-free node is the answer
// (outcome 1); otherwise create the child constraining a, then the one constraining b, each replanning only its agent
// (a child without a path is not created and takes no id).  An empty open list gives outcome 0, max_nodes pops without
// an answer outcome 2.  The root (every agent unconstrained) gives outcome 0 with no search when an agent has no path
// or a start / goal lies off the map, on an obstacle, or repeats.
//
// Mapping: one warp per env, envs taken from a global atomic counter (expansion counts are heavy-tailed, so a static
// split would leave the launch waiting on its unluckiest warp; each env's result does not depend on its warp).  Lane r
// holds map row r's word in the wavefront, lane i agent i in the conflict scan: each lane steps its path through t,
// vertex conflicts by __match_any_sync on the next cell, following conflicts by a per-warp shared owner table (agent on
// each cell at t), the order above by ballots and the lowest lane.  The open list is a warp-wide min scan over the
// created nodes' keys (SOC << 32 | id, closed = ~0).
//
// Workspace: a 16-byte header (the env counter, zeroed by the launcher on the caller's stream), then per env
// (cbs_env_bytes): nodes int4 [1 + 2K] = {parent, SOC, agent | cell << 16, t | arrival << 16} (cell = row << 5 | col;
// the constrained agent's constraint and its replanned arrival), keys uint64 [1 + 2K], the root's arrivals int16 [32],
// the constraint plane Cons and the wavefront plane F, uint32 [(H+1) x rows] each, and the path slots int8
// [N + 2K][ceil16(H)] (root agent i in slot i, node j >= 1 in slot N + j - 1): the actions up to the arrival.
// Cons is zero between nodes: a child sets its agent's constraints, found by one walk up the parent chain, plans, and
// clears the same words.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "mapf_kernels.cuh"

namespace mapf {

constexpr int CBS_THREADS = 128;

__host__ __device__ inline int64_t cbs_slot_bytes(int horizon) { return ((int64_t)horizon + 15) & ~15LL; }

__host__ __device__ inline int64_t cbs_env_bytes(int rows, int num_agents, int horizon, int max_nodes) {
    const int64_t nodes = 2LL * max_nodes + 1;
    const int64_t bytes = 24 * nodes + 64 + 8LL * (horizon + 1) * rows +
                          (num_agents + 2LL * max_nodes) * cbs_slot_bytes(horizon);
    return (bytes + 15) & ~15LL;
}

// The wavefront step and the backtrack step of mapf_plan_kernel, written out here: the same code as helpers shared
// with that kernel changes its instruction schedule, and the prioritized and windowed planners keep their SASS.
__device__ __forceinline__ uint32_t cbs_wave_step(uint32_t F, int lane) {
    const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, F, 1), dn = __shfl_down_sync(0xFFFFFFFFu, F, 1);
    return F | (F << 1) | (F >> 1) | (lane > 0 ? up : 0u) | (lane < 31 ? dn : 0u);
}

// One backtrack step from (r, c) at t: the first predecessor in F_{t-1} (row words f, one per lane) in the action order
// NO_OP, UP, RIGHT, DOWN, LEFT; returns the action and sets (pr, pc).
__device__ __forceinline__ int cbs_back_step(uint32_t f, int R, int r, int c, int &pr, int &pc) {
    const unsigned full = 0xFFFFFFFFu;
    const uint32_t fm = __shfl_sync(full, f, r > 0 ? r - 1 : 0);
    const uint32_t f0 = __shfl_sync(full, f, r);
    const uint32_t fp = __shfl_sync(full, f, r + 1 < 32 ? r + 1 : 31);
    int a;
    pr = r;
    pc = c;
    if (f0 >> c & 1u) { a = 0; }                                             // NO_OP from (r, c)
    else if (r + 1 < R && (fp >> c & 1u)) { a = 1; pr = r + 1; }              // UP from (r+1, c)
    else if (c > 0 && (f0 >> (c - 1) & 1u)) { a = 2; pc = c - 1; }            // RIGHT from (r, c-1)
    else if (r > 0 && (fm >> c & 1u)) { a = 3; pr = r - 1; }                  // DOWN from (r-1, c)
    else { a = 4; pc = c + 1; }                                               // LEFT from (r, c+1)
    return a;
}

// The low level of one agent under the constraints set in Cons (goal bound L): writes its actions to act[0..ta-1] and
// returns the arrival ta, or -1.  Every lane of the warp calls it with the same arguments.
__device__ __forceinline__ int cbs_low_level(uint32_t freerow, int lane, int R, int H, int sr, int sc, int gr, int gc,
                                             int L, const uint32_t *Cons, uint32_t *Fw, int8_t *act) {
    const unsigned full = 0xFFFFFFFFu;
    if (Cons[sr] >> sc & 1u) return -1;
    uint32_t F = lane == sr ? 1u << sc : 0u;
    if (lane < R) Fw[lane] = F;
    int ta = -1;
    if (sr == gr && sc == gc && L == 0) {
        ta = 0;
    } else {
        uint32_t cn = lane < R ? Cons[R + lane] : 0u;   // Cons_t, the load of Cons_{t+1} issued one step ahead
        for (int t = 1; t <= H; ++t) {
            const uint32_t cnn = (t < H && lane < R) ? Cons[(t + 1) * R + lane] : 0u;
            F = cbs_wave_step(F, lane) & freerow & ~cn;
            if (lane < R) Fw[t * R + lane] = F;
            const uint32_t at_goal = __shfl_sync(full, F, gr) >> gc & 1u;
            if (t >= L && at_goal) { ta = t; break; }
            if (!__any_sync(full, F != 0u)) break;
            cn = cnn;
        }
    }
    __syncwarp();
    int r = gr, c = gc;
    uint32_t f = (ta >= 1 && lane < R) ? Fw[(ta - 1) * R + lane] : 0u;
    for (int t = ta; t >= 1; --t) {
        const uint32_t fnext = (t >= 2 && lane < R) ? Fw[(t - 2) * R + lane] : 0u;
        int pr, pc;
        const int a = cbs_back_step(f, R, r, c, pr, pc);
        if (lane == 0) act[t - 1] = (int8_t)a;
        r = pr;
        c = pc;
        f = fnext;
    }
    __syncwarp();
    return ta;
}

// Sets (set = true) or clears the Cons words of agent x's constraints on the chain from node j up to the root, and
// returns L over them and `base` (the goal bound of the new constraint).  Lane 0 writes; every lane walks.
__device__ __forceinline__ int cbs_walk_constraints(const int4 *nodes, int j, int x, int gcell, int base, bool set,
                                                    uint32_t *Cons, int R, int lane) {
    int L = base;
    while (j != 0) {
        const int4 n = nodes[j];
        if ((n.z & 0xFF) == x) {
            const int cell = n.z >> 16, t = n.w & 0xFFFF;
            if (lane == 0) {
                uint32_t &w = Cons[t * R + (cell >> 5)];
                w = set ? (w | 1u << (cell & 31)) : 0u;
            }
            if (cell == gcell && t + 1 > L) L = t + 1;
        }
        j = n.x;
    }
    __syncwarp();
    return L;
}

__global__ void __launch_bounds__(CBS_THREADS) mapf_cbs_kernel(
    const uint32_t *__restrict__ free_bits, int R, int C, long long B, int N, int H, int K,
    const uint32_t *__restrict__ starts, const uint32_t *__restrict__ goals, const uint8_t *__restrict__ dist,
    unsigned char *__restrict__ ws, long long env_bytes, int8_t *__restrict__ actions, int16_t *__restrict__ arrival,
    uint8_t *__restrict__ status, int32_t *__restrict__ expanded_out) {
    const unsigned full = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31;
    const int cells = R * C;
    __shared__ int8_t owner_all[CBS_THREADS / 32][1024];   // agent on each cell (row << 5 | col) at t, -1 = none
    int8_t *owner = owner_all[threadIdx.x >> 5];
    for (int i = lane; i < 1024; i += 32) owner[i] = -1;
    __syncwarp();
    uint32_t freerow = 0;
    if (lane < R) {
        const int b0 = lane * C;
        const uint64_t w = (uint64_t)free_bits[b0 >> 5] |
                           ((uint64_t)(((b0 >> 5) + 1) * 32 < cells + 32 ? free_bits[(b0 >> 5) + 1] : 0u) << 32);
        freerow = (uint32_t)(w >> (b0 & 31)) & (C >= 32 ? full : ((1u << C) - 1u));
    }
    unsigned long long *counter = reinterpret_cast<unsigned long long *>(ws);
    const long long nodes_n = 2LL * K + 1;
    const int64_t slot = cbs_slot_bytes(H);
    const long long tstride = B * N;
    for (;;) {
        long long b = 0;
        if (lane == 0) b = (long long)atomicAdd(counter, 1ull);
        b = __shfl_sync(full, b, 0);
        if (b >= B) break;
        unsigned char *e = ws + 16 + b * env_bytes;
        int4 *nodes = reinterpret_cast<int4 *>(e);
        unsigned long long *keys = reinterpret_cast<unsigned long long *>(e + 16 * nodes_n);
        int16_t *arr0 = reinterpret_cast<int16_t *>(e + 24 * nodes_n);
        uint32_t *Cons = reinterpret_cast<uint32_t *>(e + 24 * nodes_n + 64);
        uint32_t *Fw = Cons + (long long)(H + 1) * R;
        int8_t *paths = reinterpret_cast<int8_t *>(Fw + (long long)(H + 1) * R);
        for (int i = lane; i < (H + 1) * R; i += 32) Cons[i] = 0u;
        __syncwarp();
        // lane i: agent i's start and goal; off the map, on an obstacle or repeated -> outcome 0 without a search
        const uint32_t my_s = lane < N ? starts[b * N + lane] : 0u, my_g = lane < N ? goals[b * N + lane] : 0u;
        const int sr = prow(my_s), sc = pcol(my_s), gr = prow(my_g), gc = pcol(my_g);
        const bool inside = sr >= 0 && sr < R && sc >= 0 && sc < C && gr >= 0 && gr < R && gc >= 0 && gc < C;
        const uint32_t fs = __shfl_sync(full, freerow, inside ? sr : 0), fg = __shfl_sync(full, freerow, inside ? gr : 0);
        const bool ok = lane >= N || (inside && (fs >> sc & 1u) && (fg >> gc & 1u));
        const int scell = lane < N && inside ? sr << 5 | sc : 4096 + lane, gcell = lane < N && inside ? gr << 5 | gc : 4096 + lane;
        // both collectives on every lane (no short-circuit: a full-mask __match_any_sync needs the whole warp)
        const unsigned sm = __match_any_sync(full, scell), gm = __match_any_sync(full, gcell);
        const bool unique = __popc(sm) == 1 && __popc(gm) == 1;
        int outcome = __all_sync(full, ok && unique) ? 1 : 0;
        int expanded = 0;
        // root: every agent unconstrained; the distance table settles an unreachable goal (255 = none within 254)
        int soc = 0;
        for (int i = 0; i < N && outcome; ++i) {
            const int isr = __shfl_sync(full, sr, i), isc = __shfl_sync(full, sc, i);
            const int igr = __shfl_sync(full, gr, i), igc = __shfl_sync(full, gc, i);
            const int d = dist[(long long)(igr * C + igc) * cells + isr * C + isc];
            int ta = -1;
            if (d == 255 ? H > 254 : d <= H)
                ta = cbs_low_level(freerow, lane, R, H, isr, isc, igr, igc, 0, Cons, Fw, paths + i * slot);
            if (ta < 0) outcome = 0;
            if (lane == 0) arr0[i] = (int16_t)ta;
            soc += ta;
        }
        int my_slot = lane, my_arr = 0;
        if (outcome) {
            if (lane == 0) {
                nodes[0] = make_int4(-1, soc, 0xFF, 0);
                keys[0] = (unsigned long long)soc << 32;
            }
            __syncwarp();
            int next_id = 1;
            for (;;) {
                // pop the open node of least (SOC, id)
                unsigned long long best = ~0ull;
                for (int j = lane; j < next_id; j += 32) {
                    const unsigned long long k = keys[j];
                    best = k < best ? k : best;
                }
                for (int o = 16; o; o >>= 1) {
                    const unsigned long long k = __shfl_xor_sync(full, best, o);
                    best = k < best ? k : best;
                }
                if (best == ~0ull) { outcome = 0; break; }
                if (expanded == K) { outcome = 2; break; }
                const int P = (int)(best & 0xFFFFFFFFu), psoc = (int)(best >> 32);
                ++expanded;
                if (lane == 0) keys[P] = ~0ull;
                // lane i: agent i's latest path on P's chain (its slot and arrival)
                int found = -1;
                for (int j = P; j != 0;) {
                    const int4 n = nodes[j];
                    if (found < 0 && (n.z & 0xFF) == lane) found = j;
                    j = n.x;
                }
                my_slot = found < 0 ? lane : N + found - 1;
                my_arr = lane >= N ? 0 : found < 0 ? arr0[lane] : nodes[found].w >> 16;
                const int8_t *my_path = paths + (long long)my_slot * slot;
                // first conflict: step every agent through t, vertex conflicts before following ones
                const int T = __reduce_max_sync(full, (unsigned)my_arr);
                int r = sr, c = sc;
                if (lane < N) owner[r << 5 | c] = (int8_t)lane;
                __syncwarp();
                int ca = -1, cb = -1, cell = 0, ta_ = 0, tb_ = 0;
                uint32_t aw = 0;
                for (int t = 0; t < T; ++t) {
                    if ((t & 3) == 0) aw = t < my_arr ? *reinterpret_cast<const uint32_t *>(my_path + t) : 0u;
                    const int a = t < my_arr ? (int)(aw >> (8 * (t & 3)) & 0xFFu) : 0;
                    const int nr = r + (a == 3) - (a == 1), nc = c + (a == 2) - (a == 4);
                    const int next = lane < N ? nr << 5 | nc : 4096 + lane;
                    const unsigned m = __match_any_sync(full, next);
                    const unsigned vb = __ballot_sync(full, (m & ~(1u << lane)) != 0u);
                    if (vb) {
                        ca = __ffs(vb) - 1;
                        const unsigned ma = __shfl_sync(full, m, ca);
                        cb = __ffs(ma & ~(1u << ca)) - 1;
                        cell = __shfl_sync(full, next, ca);
                        ta_ = tb_ = t + 1;
                        break;
                    }
                    const int o = (lane < N && a != 0) ? owner[next] : -1;
                    const unsigned fb = __ballot_sync(full, o > lane);
                    if (fb) {
                        ca = __ffs(fb) - 1;
                        cb = __shfl_sync(full, o, ca);
                        cell = __shfl_sync(full, next, ca);
                        ta_ = t + 1;
                        tb_ = t;
                        break;
                    }
                    if (lane < N) owner[r << 5 | c] = -1;
                    __syncwarp();
                    if (lane < N) owner[next] = (int8_t)lane;
                    __syncwarp();
                    r = nr;
                    c = nc;
                }
                if (lane < N) owner[r << 5 | c] = -1;
                __syncwarp();
                if (ca < 0) { outcome = 1; break; }
                // the two children: agent a constrained at (cell, ta_), then agent b at (cell, tb_)
                for (int side = 0; side < 2; ++side) {
                    const int x = side ? cb : ca, xt = side ? tb_ : ta_;
                    const int xsr = __shfl_sync(full, sr, x), xsc = __shfl_sync(full, sc, x);
                    const int xgr = __shfl_sync(full, gr, x), xgc = __shfl_sync(full, gc, x);
                    const int xg = xgr << 5 | xgc;
                    const int xarr = __shfl_sync(full, my_arr, x);
                    if (lane == 0) Cons[xt * R + (cell >> 5)] |= 1u << (cell & 31);
                    const int L = cbs_walk_constraints(nodes, P, x, xg, cell == xg ? xt + 1 : 0, true, Cons, R, lane);
                    int8_t *dst = paths + (long long)(N + next_id - 1) * slot;
                    const int ta = cbs_low_level(freerow, lane, R, H, xsr, xsc, xgr, xgc, L, Cons, Fw, dst);
                    if (lane == 0) Cons[xt * R + (cell >> 5)] = 0u;
                    cbs_walk_constraints(nodes, P, x, xg, 0, false, Cons, R, lane);
                    if (ta >= 0) {
                        const int csoc = psoc - xarr + ta;
                        if (lane == 0) {
                            nodes[next_id] = make_int4(P, csoc, x | cell << 16, xt | ta << 16);
                            keys[next_id] = (unsigned long long)csoc << 32 | (unsigned)next_id;
                        }
                        __syncwarp();
                        ++next_id;
                    }
                }
            }
        }
        // outputs: the answer's actions up to each arrival, NO_OPs after; NO_OPs and arrival -1 for outcomes 0 and 2
        if (lane < N) arrival[b * N + lane] = (int16_t)(outcome == 1 ? my_arr : -1);
        for (int i = 0; i < N; ++i) {
            const int is = __shfl_sync(full, my_slot, i), ia = outcome == 1 ? __shfl_sync(full, my_arr, i) : 0;
            const int8_t *src = paths + (long long)is * slot;
            for (int t = lane; t < H; t += 32) actions[t * tstride + b * N + i] = t < ia ? src[t] : (int8_t)0;
        }
        if (lane == 0) {
            status[b] = (uint8_t)outcome;
            expanded_out[b] = expanded;
        }
    }
}

}  // namespace mapf
