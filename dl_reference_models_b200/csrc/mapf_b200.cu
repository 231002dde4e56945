// mapf_b200.cu -- the C ABI of libmapf_b200.so (see include/mapf_b200.h) over the sm_100a kernels
// of mapf_kernels.cuh.  Host side only: argument validation, map bit-packing, launch geometry,
// state/IO buffer management.  There is no CPU implementation of the transition in here: every
// entry point that computes launches a kernel, and fails with MAPF_ERR_CUDA if it cannot.
#include "mapf_env_kernel.cuh"
#include "mapf_pair_kernel.cuh"
#include "mapf_cte_kernel.cuh"
#include "mapf_cte_policy_kernel.cuh"
#include "mapf_cte_lstm_policy_kernel.cuh"
#include "mapf_policy_kernel.cuh"
#include "mapf_policy_lstm_kernel.cuh"
#include "mapf_eval_kernel.cuh"
#include "mapf_vtrace_kernel.cuh"
#include "mapf_q_kernel.cuh"
#include "mapf_replay_kernel.cuh"
#include "mapf_pack_kernel.cuh"
#include "mapf_host_unpack.h"

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sched.h>
#include <new>
#include <string>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return fail(MAPF_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                   \
    } while (0)

using KernelFn = void (*)(const mapf::KParams);

// MAPF_DEV_MINIMAL (kernel A/B experiments only, tools/build_variant.sh): instantiate sensor range 2 alone, so that
// a variant library builds in a fraction of the time; every other shape then fails loudly in mapf_create.
template <int G>
KernelFn step_for_sr(int sr) {
    switch (sr) {
#ifndef MAPF_DEV_MINIMAL
        case 1: return mapf::mapf_step_kernel<G, 1>;
        case 3: return mapf::mapf_step_kernel<G, 3>;
#endif
        case 2: return mapf::mapf_step_kernel<G, 2>;
    }
    return nullptr;
}
template <int G>
KernelFn reset_for_sr(int sr) {
    switch (sr) {
#ifndef MAPF_DEV_MINIMAL
        case 1: return mapf::mapf_reset_kernel<G, 1>;
        case 3: return mapf::mapf_reset_kernel<G, 3>;
#endif
        case 2: return mapf::mapf_reset_kernel<G, 2>;
    }
    return nullptr;
}
// the default sensor range also comes with the lifelong / episodic switches compiled in (mode 1 / 2, lock metrics on)
template <int G>
KernelFn step_for_mode(int mode) {
    if (mode == 1) return mapf::mapf_step_kernel<G, 2, 1>;
    if (mode == 2) return mapf::mapf_step_kernel<G, 2, 2>;
    return nullptr;
}
KernelFn pick_step(int G, int sr, int mode = 0) {
    if (sr == 2 && mode != 0) {
        switch (G) {
#ifndef MAPF_DEV_MINIMAL
            case 4: return step_for_mode<4>(mode);
            case 8: return step_for_mode<8>(mode);
#endif
            case 16: return step_for_mode<16>(mode);
            case 32: return step_for_mode<32>(mode);
        }
    }
    switch (G) {
#ifndef MAPF_DEV_MINIMAL
        case 4: return step_for_sr<4>(sr);
        case 8: return step_for_sr<8>(sr);
#endif
        case 16: return step_for_sr<16>(sr);
        case 32: return step_for_sr<32>(sr);
    }
    return nullptr;
}
KernelFn pick_reset(int G, int sr) {
    switch (G) {
#ifndef MAPF_DEV_MINIMAL
        case 4: return reset_for_sr<4>(sr);
        case 8: return reset_for_sr<8>(sr);
#endif
        case 16: return reset_for_sr<16>(sr);
        case 32: return reset_for_sr<32>(sr);
    }
    return nullptr;
}

constexpr size_t kMaxSmem = 200 * 1024;
constexpr size_t kMaxSmemEnv = 227 * 1024;  // opt-in limit of one sm_100 CTA

using EnvKernelFn = void (*)(const mapf::KParams, const mapf::EnvLayout);
template <bool VEC, bool FAST, bool MANY>
EnvKernelFn env_step_for_sr(int sr) {
    switch (sr) {
#ifndef MAPF_DEV_MINIMAL
        case 1: return mapf::mapf_step_env_kernel<1, VEC, FAST, MANY>;
        case 3: return mapf::mapf_step_env_kernel<3, VEC, FAST, MANY>;
#endif
        case 2: return mapf::mapf_step_env_kernel<2, VEC, FAST, MANY>;
    }
    return nullptr;
}
template <bool FAST>
EnvKernelFn pair_step_for_sr(int sr) {
    switch (sr) {
#ifndef MAPF_DEV_MINIMAL
        case 1: return mapf::mapf_step_pair_kernel<1, FAST>;
        case 3: return mapf::mapf_step_pair_kernel<3, FAST>;
#endif
        case 2: return mapf::mapf_step_pair_kernel<2, FAST>;
    }
    return nullptr;
}
EnvKernelFn pick_pair_step(int sr, bool fast) {
#ifndef MAPF_DEV_MINIMAL
    return fast ? pair_step_for_sr<true>(sr) : pair_step_for_sr<false>(sr);
#else
    return fast ? pair_step_for_sr<true>(sr) : nullptr;
#endif
}
template <bool MANY>
EnvKernelFn pick_env_step_m(int sr, bool vec, bool fast) {
    if (fast && vec) return env_step_for_sr<true, true, MANY>(sr);   // lifelong + lock metrics as compile-time constants
#ifndef MAPF_DEV_MINIMAL
    return vec ? env_step_for_sr<true, false, MANY>(sr) : env_step_for_sr<false, false, MANY>(sr);
#else
    return vec ? env_step_for_sr<true, false, MANY>(sr) : nullptr;
#endif
}
// many: the mapf_step_many instantiation (K env steps per launch)
EnvKernelFn pick_env_step(int sr, bool vec, bool fast, bool many = false) {
    return many ? pick_env_step_m<true>(sr, vec, fast) : pick_env_step_m<false>(sr, vec, fast);
}

}  // namespace

constexpr int kMaxHostSlices = 16;

struct mapf_handle {
    mapf_config cfg;
    int G, SR, V2, LW;
    int wpr, map_words, fw;
    int threads;
    size_t smem_bytes;
    mapf::SmemLayout layout;
    int step_grid_cap;
    int8_t *fused_actions;
    int fused_mode;
    uint64_t fused_counter;
    KernelFn step_fn, reset_fn;
    // env-per-thread step kernel (maps up to 32 columns wide, shared map); 0 threads = not available
    EnvKernelFn env_fn, env_fn_many;   // env_fn_many: K steps per launch (mapf_step_many), null when not available
    mapf::EnvLayout env_layout;
    int env_threads, env_grid;
    bool use_env_kernel, env_pdl;
    bool env_prefetch;  // MAPF_ENV_PREFETCH (default on): L2 prefetch of a warp's first tile ahead of griddepcontrol.wait
    bool pair_kernel;   // the env kernel in use is the two-lanes-per-env one (mapf_pair_kernel.cuh)
    uint32_t *d_map_rows, *d_free_bits;
    uint32_t *d_env_tables;
    int32_t *d_num_free;
    bool map_set;
    uint32_t *d_err;
    mapf_state st;
    bool bound, owns_state;
    int64_t launches;
    // device mirrors of the *_host entry points' arguments (allocated on first use)
    cudaStream_t hstream, hstream2;
    bool io_alloc;
    int8_t *io_actions;
    uint32_t *io_goal_override, *io_starts_override, *io_goals_override;
    int32_t *io_goal_rank;
    uint8_t *io_reset_mask;
    mapf_outputs io_out;
    // packed device->host transfer of mapf_step_host (mapf_pack_kernel.cuh / mapf_host_unpack.cpp)
    bool pack_alloc;
    uint8_t *d_packed, *h_packed;
    mapf::HostPool *pool;
    uint32_t *h_tickets;   // pinned: slot c = number of the last step whose slice c has arrived on the host
    uint32_t ticket_seq;
    float gdt_row[256], gdt_col[256];
    int64_t last_h2d_bytes, last_d2h_bytes;
    // tuning knobs of the host-buffer path, read from the environment ONCE (mapf_create), not per call
    int knob_host_threads;      // MAPF_HOST_THREADS (0 = derive from the affinity mask)
    int knob_host_pack;         // MAPF_HOST_PACK: -1 unset, 0 off, 1 on
    int knob_host_slices;       // MAPF_HOST_SLICES (0 = default)
    int knob_plan_n, knob_plan[kMaxHostSlices];   // MAPF_HOST_PLAN=w0,w1,...
    int knob_raw32;             // MAPF_HOST_RAW_32NDS
    bool knob_trace;            // MAPF_HOST_TRACE
    int local_world;            // LOCAL_WORLD_SIZE (ranks sharing this node's cores), >= 1
    int local_rank;             // LOCAL_RANK, 0 when unset
    int knob_host_pin;          // MAPF_HOST_PIN: -1 unset (pin when the node is shared), 0 off, 1 on
    // packed-or-plain, decided by measurement: calls 0-2 go packed, 3-5 plain (the first of each untimed), then the
    // faster one stays -- on THIS host, with whatever else (the other ranks of the node) is running beside it
    int auto_calls, auto_choice;          // auto_choice: -1 undecided, 0 plain, 1 packed, 2 packed + non-temporal expansion
    int64_t auto_ns[3];                   // best call time of the timed calls: [plain, packed, packed + NT]
    int knob_host_nt;                     // MAPF_HOST_NT: -1 unset (measured with the rest), 0 off, 1 on
    // ordering of the *_host entry points (private streams) against work the caller queued on ITS stream
    cudaEvent_t ev_user;
    cudaStream_t last_user_stream;
    bool user_dirty;
};

namespace {

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() {
        if (ok && prev >= 0) cudaSetDevice(prev);
    }
};

void state_sizes(const mapf_handle *h, int64_t n[10]) {
    const int64_t B = h->cfg.num_envs, N = h->cfg.num_agents;
    n[0] = B * N * 4;                      // positions  int16[B,N,2]
    n[1] = B * N * 4;                      // goals
    n[2] = B * N * 4;                      // starts
    n[3] = B * N;                          // agent_flags
    n[4] = B * N * 4;                      // lock_goal_progress
    n[5] = B * N * 4;                      // lock_moved
    n[6] = B * N * 4;                      // lock_failed_move
    n[7] = B * (int64_t)h->LW * N * 2;     // lock_distance int16[B,LW,N]
    n[8] = B * MAPF_ENV_WORDS * 4;         // env_words
    n[9] = B * MAPF_METRIC_COUNT * 8;      // env_metrics
}

void **state_member(mapf_state *s, int i) {
    switch (i) {
        case 0: return reinterpret_cast<void **>(&s->positions);
        case 1: return reinterpret_cast<void **>(&s->goals);
        case 2: return reinterpret_cast<void **>(&s->starts);
        case 3: return reinterpret_cast<void **>(&s->agent_flags);
        case 4: return reinterpret_cast<void **>(&s->lock_goal_progress);
        case 5: return reinterpret_cast<void **>(&s->lock_moved);
        case 6: return reinterpret_cast<void **>(&s->lock_failed_move);
        case 7: return reinterpret_cast<void **>(&s->lock_distance);
        case 8: return reinterpret_cast<void **>(&s->env_words);
        case 9: return reinterpret_cast<void **>(&s->env_metrics);
    }
    return nullptr;
}

void output_sizes(const mapf_handle *h, int64_t n[10]) {
    const int64_t B = h->cfg.num_envs, N = h->cfg.num_agents;
    n[0] = B * N * h->V2;           // local_obs
    n[1] = B * N * 5;               // action_mask
    n[2] = B * N * 8;               // goal_delta
    n[3] = B * N;                   // blocking_prev
    n[4] = B * N * 4;               // reward
    n[5] = B;                       // terminated
    n[6] = B;                       // truncated
    n[7] = B;                       // step_flags
    n[8] = B * N;                   // agent_step_flags
    n[9] = B * MAPF_INFO_WORDS * 4; // info
}

void **output_member(mapf_outputs *o, int i) {
    switch (i) {
        case 0: return reinterpret_cast<void **>(&o->local_obs);
        case 1: return reinterpret_cast<void **>(&o->action_mask);
        case 2: return reinterpret_cast<void **>(&o->goal_delta);
        case 3: return reinterpret_cast<void **>(&o->blocking_prev);
        case 4: return reinterpret_cast<void **>(&o->reward);
        case 5: return reinterpret_cast<void **>(&o->terminated);
        case 6: return reinterpret_cast<void **>(&o->truncated);
        case 7: return reinterpret_cast<void **>(&o->step_flags);
        case 8: return reinterpret_cast<void **>(&o->agent_step_flags);
        case 9: return reinterpret_cast<void **>(&o->info);
    }
    return nullptr;
}

int check_ready(const mapf_handle *h) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    if (!h->map_set) return fail(MAPF_ERR_STATE, "mapf_set_map has not been called");
    if (!h->bound) return fail(MAPF_ERR_STATE, "no state bound (mapf_bind_state / mapf_alloc_state)");
    return MAPF_OK;
}

void fill_params(const mapf_handle *h, mapf::KParams &p) {
    const mapf_config &c = h->cfg;
    memset(&p, 0, sizeof(p));
    p.B = c.num_envs; p.N = c.num_agents; p.R = c.rows; p.C = c.cols;
    p.steps_per_episode = c.steps_per_episode;
    p.lifelong = c.lifelong_mapf != 0;
    p.lock_enabled = c.enable_lock_metrics != 0;
    p.dw = c.deadlock_window_steps; p.lw = c.livelock_window_steps;
    p.nearby = c.lock_nearby_manhattan; p.min_nb = c.lock_min_neighbors;
    p.eps_floor = c.lock_progress_epsilon_floor;
    p.normalize = c.normalize_goal_delta != 0;
    p.deterministic = c.deterministic != 0;
    p.per_env_maps = c.per_env_maps != 0;
    p.env_id_base = c.env_id_base;
    p.seed = c.seed;
    p.den0 = (float)(c.rows - 1 > 1 ? c.rows - 1 : 1);  // ENV:152-155
    p.den1 = (float)(c.cols - 1 > 1 ? c.cols - 1 : 1);
    p.map_rows = h->d_map_rows; p.free_bits = h->d_free_bits; p.num_free = h->d_num_free;
    p.env_tables = h->d_env_tables;
    p.wpr = h->wpr; p.map_words = h->map_words; p.fw = h->fw;
    p.positions = reinterpret_cast<uint32_t *>(h->st.positions);
    p.goals = reinterpret_cast<uint32_t *>(h->st.goals);
    p.starts = reinterpret_cast<uint32_t *>(h->st.starts);
    p.agent_flags = h->st.agent_flags;
    p.lock_gp = h->st.lock_goal_progress; p.lock_mv = h->st.lock_moved; p.lock_fm = h->st.lock_failed_move;
    p.lock_dist = h->st.lock_distance;
    p.env_words = reinterpret_cast<int4 *>(h->st.env_words);
    p.env_metrics = h->st.env_metrics;
    p.err_bits = h->d_err;
    p.L = h->layout;
    p.inner_steps = 1;
    p.out_step_stride = 0;
    p.env_prefetch = h->env_prefetch ? 1 : 0;
}

void fill_outputs(mapf::KParams &p, const mapf_outputs *o) {
    if (!o) return;
    p.o_local_obs = o->local_obs; p.o_action_mask = o->action_mask;
    p.o_goal_delta = reinterpret_cast<float2 *>(o->goal_delta);
    p.o_blocking_prev = o->blocking_prev; p.o_reward = o->reward;
    p.o_terminated = o->terminated; p.o_truncated = o->truncated;
    p.o_step_flags = o->step_flags; p.o_agent_step_flags = o->agent_step_flags;
    p.o_info = reinterpret_cast<int4 *>(o->info);
}

void note_user_stream(mapf_handle *h, cudaStream_t s);

int launch_env_step(mapf_handle *h, const mapf::KParams &p, cudaStream_t s, EnvKernelFn fn = nullptr) {
    // launched with programmatic stream serialization: back-to-back steps overlap the next launch's ramp-up and
    // table copy with this launch's tail (the kernel waits with griddepcontrol.wait before it touches env state)
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)h->env_grid);
    cfg.blockDim = dim3((unsigned)h->env_threads);
    cfg.dynamicSmemBytes = (size_t)h->env_layout.total_bytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = h->env_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, fn ? fn : h->env_fn, p, h->env_layout));
    h->launches++;
    return MAPF_OK;
}

// The step kernels contain griddepcontrol.wait and are launched with programmatic stream serialization (see
// launch_env_step); every other kernel is launched the plain way (full stream order).
int launch_lane_step(mapf_handle *h, const mapf::KParams &p, unsigned grid, cudaStream_t s) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3((unsigned)h->threads);
    cfg.dynamicSmemBytes = h->smem_bytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = h->env_pdl ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, h->step_fn, p));
    h->launches++;
    return MAPF_OK;
}

int launch(mapf_handle *h, KernelFn fn, const mapf::KParams &p, cudaStream_t s) {
    note_user_stream(h, s);
    if (fn == h->step_fn && h->use_env_kernel) return launch_env_step(h, p, s);
    const int groups = h->threads / h->G;
    unsigned grid = (unsigned)((h->cfg.num_envs + groups - 1) / groups);
    // the step kernel is persistent: one wave of resident CTAs walks over the env tiles
    if (fn == h->step_fn && h->step_grid_cap > 0 && grid > (unsigned)h->step_grid_cap) grid = (unsigned)h->step_grid_cap;
    if (fn == h->step_fn) return launch_lane_step(h, p, grid, s);
    fn<<<grid, h->threads, h->smem_bytes, s>>>(p);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

// The step over envs [e0, e0 + n) only: every per-env pointer advanced, Philox keys kept (global env ids).
// Sub-batches always take the lane-per-agent kernel (the env-per-thread kernel needs a GPU-filling batch).
int launch_step_range(mapf_handle *h, mapf::KParams p, int64_t e0, int n, cudaStream_t s) {
    const int64_t N = h->cfg.num_agents, LW = h->LW;
    auto adv = [&](auto *&ptr, int64_t elems) { if (ptr) ptr += e0 * elems; };
    adv(p.positions, N); adv(p.goals, N); adv(p.starts, N); adv(p.agent_flags, N);
    adv(p.lock_gp, N); adv(p.lock_mv, N); adv(p.lock_fm, N); adv(p.lock_dist, LW * N);
    adv(p.env_words, 4); adv(p.env_metrics, MAPF_METRIC_COUNT);
    adv(p.actions, N); adv(p.goal_override, N); adv(p.goal_rank, N); adv(p.reset_mask, 1);
    adv(p.starts_override, N); adv(p.goals_override, N);
    adv(p.o_local_obs, N * h->V2); adv(p.o_action_mask, N * 5); adv(p.o_goal_delta, N); adv(p.o_blocking_prev, N);
    adv(p.o_reward, N); adv(p.o_terminated, 1); adv(p.o_truncated, 1); adv(p.o_step_flags, 1);
    adv(p.o_agent_step_flags, N); adv(p.o_info, 4); adv(p.o_next_actions, N);
    if (p.per_env_maps) { adv(p.map_rows, h->map_words); adv(p.free_bits, h->fw); adv(p.num_free, 1); }
    p.B = n;
    p.env_id_base += e0;
    const int groups = h->threads / h->G;
    unsigned grid = (unsigned)((n + groups - 1) / groups);
    if (h->step_grid_cap > 0 && grid > (unsigned)h->step_grid_cap) grid = (unsigned)h->step_grid_cap;
    return launch_lane_step(h, p, grid, s);
}

int ensure_io(mapf_handle *h) {
    if (h->io_alloc) return MAPF_OK;
    const int64_t B = h->cfg.num_envs, N = h->cfg.num_agents;
    if (!h->hstream) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    if (!h->hstream2) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream2, cudaStreamNonBlocking));
    CUDA_TRY(cudaMalloc(&h->io_actions, B * N));
    CUDA_TRY(cudaMalloc(&h->io_goal_override, B * N * 4));
    CUDA_TRY(cudaMalloc(&h->io_starts_override, B * N * 4));
    CUDA_TRY(cudaMalloc(&h->io_goals_override, B * N * 4));
    CUDA_TRY(cudaMalloc(&h->io_goal_rank, B * N * 4));
    CUDA_TRY(cudaMalloc(&h->io_reset_mask, B));
    int64_t n[10];
    output_sizes(h, n);
    for (int i = 0; i < 10; ++i) CUDA_TRY(cudaMalloc(output_member(&h->io_out, i), (size_t)n[i]));
    h->io_alloc = true;
    return MAPF_OK;
}

// device copies of the requested host outputs: only channels the caller asked for are computed
void select_outputs(mapf_handle *h, const mapf_outputs *host, mapf_outputs *dev) {
    memset(dev, 0, sizeof(*dev));
    if (!host) return;
    mapf_outputs tmp = *host;
    for (int i = 0; i < 10; ++i)
        if (*output_member(&tmp, i)) *output_member(dev, i) = *output_member(&h->io_out, i);
}

int copy_outputs_back(mapf_handle *h, const mapf_outputs *host) {
    if (!host) return MAPF_OK;
    int64_t n[10];
    output_sizes(h, n);
    mapf_outputs tmp = *host;
    for (int i = 0; i < 10; ++i) {
        void *dst = *output_member(&tmp, i);
        if (dst)
            CUDA_TRY(cudaMemcpyAsync(dst, *output_member(&h->io_out, i), (size_t)n[i],
                                     cudaMemcpyDeviceToHost, h->hstream));
    }
    return MAPF_OK;
}

void read_knobs(mapf_handle *h) {
    h->knob_host_threads = 0; h->knob_host_pack = -1; h->knob_host_slices = 0; h->knob_plan_n = 0; h->knob_raw32 = 0;
    h->knob_trace = getenv("MAPF_HOST_TRACE") != nullptr;
    h->local_world = 1;
    if (const char *ov = getenv("MAPF_HOST_THREADS")) { const int v = atoi(ov); if (v >= 1) h->knob_host_threads = v > 64 ? 64 : v; }
    if (const char *ov = getenv("MAPF_HOST_PACK")) h->knob_host_pack = atoi(ov) != 0 ? 1 : 0;
    if (const char *ov = getenv("MAPF_HOST_SLICES")) { const int v = atoi(ov); if (v >= 1) h->knob_host_slices = v > kMaxHostSlices ? kMaxHostSlices : v; }
    if (const char *ov = getenv("MAPF_HOST_PLAN")) {
        int k = 0;
        for (const char *q = ov; *q && k < kMaxHostSlices;) {
            const int v = atoi(q);
            if (v >= 1) h->knob_plan[k++] = v;
            while (*q && *q != ',') ++q;
            if (*q == ',') ++q;
        }
        h->knob_plan_n = k;
    }
    if (const char *ov = getenv("MAPF_HOST_RAW_32NDS")) { const int v = atoi(ov); if (v >= 0 && v <= 16) h->knob_raw32 = v; }
    // one process per GPU: the ranks of a node share its cores (torchrun exports LOCAL_WORLD_SIZE)
    if (const char *lw = getenv("LOCAL_WORLD_SIZE")) { const int w = atoi(lw); if (w > 1) h->local_world = w; }
    h->local_rank = 0;
    if (const char *lr = getenv("LOCAL_RANK")) { const int r = atoi(lr); if (r >= 0 && r < h->local_world) h->local_rank = r; }
    h->knob_host_pin = -1;
    if (const char *ov = getenv("MAPF_HOST_PIN")) h->knob_host_pin = atoi(ov) != 0 ? 1 : 0;
    h->auto_calls = 0; h->auto_choice = -1; h->auto_ns[0] = h->auto_ns[1] = h->auto_ns[2] = 0;
    h->knob_host_nt = -1;
    if (const char *ov = getenv("MAPF_HOST_NT")) h->knob_host_nt = atoi(ov) != 0 ? 1 : 0;
}

// This rank's share of the cores the process may run on: a contiguous chunk of the affinity mask per local rank.
int rank_cores(const mapf_handle *h, int *cpus, int cap) {
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) != 0) return 0;
    int all[CPU_SETSIZE], n = 0;
    for (int c = 0; c < CPU_SETSIZE; ++c) if (CPU_ISSET(c, &set)) all[n++] = c;
    const int per = n / h->local_world;
    if (per < 1) return 0;
    int k = 0;
    for (int i = h->local_rank * per; i < (h->local_rank + 1) * per && k < cap; ++i) cpus[k++] = all[i];
    return k;
}

int host_threads_default(const mapf_handle *h) {
    if (h->knob_host_threads >= 1) return h->knob_host_threads;
    int n = 0;
    cpu_set_t set;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
    n /= h->local_world;
    if (n < 1) n = 1;
    return n > 16 ? 16 : n;
}

// The *_host entry points run on the handle's private streams.  Whatever the caller queued before -- through the
// stream-taking entry points (remembered in last_user_stream) or on a stream it names with mapf_host_wait_stream --
// must be ordered in front of them: one event, two waits, only when something is pending.
int order_after_user_work(mapf_handle *h) {
    if (!h->user_dirty) return MAPF_OK;
    if (!h->ev_user) CUDA_TRY(cudaEventCreateWithFlags(&h->ev_user, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(h->ev_user, h->last_user_stream));
    if (h->hstream) CUDA_TRY(cudaStreamWaitEvent(h->hstream, h->ev_user, 0));
    if (h->hstream2) CUDA_TRY(cudaStreamWaitEvent(h->hstream2, h->ev_user, 0));
    h->user_dirty = false;
    return MAPF_OK;
}
void note_user_stream(mapf_handle *h, cudaStream_t s) {
    if (s == h->hstream || s == h->hstream2) return;   // our own launches
    h->last_user_stream = s;
    h->user_dirty = true;
}

// The bit-packed transfer applies when the four big per-agent channels are all requested, the integer goal
// differences fit an int8, the batch is big enough for the PCIe time to matter, and this process has at least 12
// host cores to itself: the expansion trades PCIe bytes for host memory traffic, and on a node whose cores and
// DRAM are shared by many ranks plain copies win (measured on an 8-GPU / 32-core host: plain 2.24e9, packed
// 1.76e9 agent-steps/s aggregate; on 1 GPU / 16 cores: plain 1.13e9, packed 2.36e9; 2 GPUs / 24 cores: packed
// 2.72e9).  MAPF_HOST_PACK=0 / 1 forces it off / on.
bool host_pack_eligible(const mapf_handle *h, const mapf_outputs *host) {
    if (!host || !host->local_obs || !host->action_mask || !host->goal_delta || !host->reward) return false;
    if (h->cfg.rows > 128 || h->cfg.cols > 128 || h->cfg.num_envs < 8192) return false;
    return true;
}

int ensure_pack(mapf_handle *h) {
    if (h->pack_alloc) return MAPF_OK;
    const size_t BN = (size_t)h->cfg.num_envs * h->cfg.num_agents;
    const size_t bytes = BN * (mapf::pack_record_bytes(h->V2) + 1) + (size_t)h->cfg.num_envs * 3 + 64;
    CUDA_TRY(cudaMalloc(&h->d_packed, bytes));
    CUDA_TRY(cudaMallocHost(&h->h_packed, bytes));
    CUDA_TRY(cudaMallocHost(&h->h_tickets, (kMaxHostSlices + 1) * sizeof(uint32_t)));
    memset(h->h_tickets, 0, (kMaxHostSlices + 1) * sizeof(uint32_t));
    const float den0 = (float)(h->cfg.rows - 1 > 1 ? h->cfg.rows - 1 : 1);
    const float den1 = (float)(h->cfg.cols - 1 > 1 ? h->cfg.cols - 1 : 1);
    for (int d = -128; d < 128; ++d) {  // the kernels' goal-delta table (mapf_kernels.cuh fill_goal_delta_table)
        h->gdt_row[d + 128] = h->cfg.normalize_goal_delta ? (float)d / den0 : (float)d;  // d / 1 == d
        h->gdt_col[d + 128] = h->cfg.normalize_goal_delta ? (float)d / den1 : (float)d;
    }
    {
        // On a node shared by several ranks every rank keeps to its own cores: the workers are pinned one per core to
        // this rank's chunk of the affinity mask (its first core is left to the calling thread).  Alone on the node
        // the scheduler is left to it.  MAPF_HOST_PIN=0 / 1 forces it off / on.
        int cpus[64];
        int n = 0;
        const bool pin = h->knob_host_pin >= 0 ? h->knob_host_pin != 0 : h->local_world > 1;
        if (pin) n = rank_cores(h, cpus, 64);
        if (n >= 2) h->pool = mapf::host_pool_create(host_threads_default(h), cpus + 1, n - 1);
        else h->pool = mapf::host_pool_create(host_threads_default(h));
    }
    h->pack_alloc = true;
    return MAPF_OK;
}

}  // namespace

extern "C" {

const char *mapf_version(void) { return "mapf_b200 0.1.0 (sm_100a)"; }
const char *mapf_last_error(void) { return g_err.c_str(); }

int mapf_create(const mapf_config *cfg, mapf_handle **out) {
    if (!cfg || !out) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    *out = nullptr;
    const mapf_config &c = *cfg;
    if (c.num_envs < 1) return fail(MAPF_ERR_INVALID_ARG, "num_envs must be >= 1");
    if (c.num_agents < 1 || c.num_agents > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "num_agents=%d outside 1..%d", c.num_agents, MAPF_MAX_AGENTS);
    if (c.rows < 1 || c.cols < 1 || c.rows > MAPF_MAX_DIM || c.cols > MAPF_MAX_DIM)
        return fail(MAPF_ERR_UNSUPPORTED, "map %dx%d outside 1..%d", c.rows, c.cols, MAPF_MAX_DIM);
    if (c.sensor_range < 1 || c.sensor_range > MAPF_MAX_SENSOR_RANGE)
        return fail(MAPF_ERR_UNSUPPORTED, "sensor_range=%d outside 1..%d", c.sensor_range, MAPF_MAX_SENSOR_RANGE);
    if (c.deadlock_window_steps < 1 || c.deadlock_window_steps > MAPF_MAX_LOCK_WINDOW ||
        c.livelock_window_steps < 1 || c.livelock_window_steps > MAPF_MAX_LOCK_WINDOW)
        return fail(MAPF_ERR_UNSUPPORTED, "lock windows must be in 1..%d", MAPF_MAX_LOCK_WINDOW);
    if (c.lock_nearby_manhattan < 1 || c.lock_nearby_manhattan > 255 || c.lock_min_neighbors < 1)
        return fail(MAPF_ERR_INVALID_ARG, "lock_nearby_manhattan / lock_min_neighbors must be >= 1");
    if (c.steps_per_episode < 1) return fail(MAPF_ERR_INVALID_ARG, "steps_per_episode must be >= 1");
    if (c.step_kernel < 0 || c.step_kernel > 3) return fail(MAPF_ERR_INVALID_ARG, "step_kernel must be 0 (auto), 1 (lane), 2 (env) or 3 (pair)");

    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device: %s (libmapf_b200 has no CPU fallback)",
                    ce != cudaSuccess ? cudaGetErrorString(ce) : "device count is 0");
    if (c.device < 0 || c.device >= ndev) return fail(MAPF_ERR_INVALID_ARG, "device %d of %d", c.device, ndev);
    DeviceGuard guard(c.device);
    if (!guard.ok) return fail(MAPF_ERR_CUDA, "cudaSetDevice(%d) failed", c.device);

    mapf_handle *h = new (std::nothrow) mapf_handle();
    if (!h) return fail(MAPF_ERR_STATE, "out of host memory");
    memset(h, 0, sizeof(*h));
    h->cfg = c;
    read_knobs(h);
    h->G = c.num_agents <= 4 ? 4 : c.num_agents <= 8 ? 8 : c.num_agents <= 16 ? 16 : 32;
    h->SR = c.sensor_range;
    h->V2 = (2 * c.sensor_range + 1) * (2 * c.sensor_range + 1);
    h->LW = c.livelock_window_steps;
    // +1 word: the window extractor reads a 64-bit funnel (word, word + 1) of every padded row
    h->wpr = (c.cols + 2 * mapf::PAD + 31) / 32 + 1;
    h->map_words = (c.rows + 2 * mapf::PAD) * h->wpr;
    h->fw = (c.rows * c.cols + 31) / 32;
    {
        // compile-time modes: lock metrics on, lifelong (1) or episodic (2), map up to 32 x 32 (fixed mask layout)
        int mode = (c.enable_lock_metrics && c.rows <= 32 && c.cols <= 32) ? (c.lifelong_mapf ? 1 : 2) : 0;
        if (const char *ov = getenv("MAPF_LANE_FAST")) mode = atoi(ov) != 0 ? mode : 0;
        h->step_fn = pick_step(h->G, h->SR, mode);
    }
    h->reset_fn = pick_reset(h->G, h->SR);
    h->threads = 0;
    for (int t = 256; t >= 32; t >>= 1) {
        mapf::SmemLayout L = mapf::make_layout(h->G, h->V2, c.num_agents, h->wpr, c.rows, c.cols, h->SR, h->fw,
                                               c.per_env_maps != 0, t);
        if ((size_t)L.total_words * 4 <= kMaxSmem) {
            h->threads = t;
            h->smem_bytes = (size_t)L.total_words * 4;
            h->layout = L;
            break;
        }
    }
    if (!h->threads) {
        delete h;
        return fail(MAPF_ERR_UNSUPPORTED, "map %dx%d needs more shared memory than one SM has", c.rows, c.cols);
    }
    if (h->threads != 256) h->step_fn = pick_step(h->G, h->SR, 0);   // the compile-time modes assume 256-thread CTAs
    if (!h->step_fn || !h->reset_fn) {
        delete h;
        return fail(MAPF_ERR_UNSUPPORTED, "no kernel instantiation for %d agents at sensor range %d in this build",
                    c.num_agents, c.sensor_range);
    }
    cudaError_t e1 = cudaFuncSetAttribute(reinterpret_cast<const void *>(h->step_fn),
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
    cudaError_t e2 = cudaFuncSetAttribute(reinterpret_cast<const void *>(h->reset_fn),
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem);
    int nsm = 0, per_sm = 0;
    if (e1 == cudaSuccess) e1 = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, c.device);
    if (e1 == cudaSuccess)
        e1 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void *>(h->step_fn),
                                                           h->threads, h->smem_bytes);
    h->step_grid_cap = nsm * (per_sm > 0 ? per_sm : 1);
    if (const char *ov = getenv("MAPF_STEP_CTAS_PER_SM")) {  // tuning knob: 0 = one CTA per tile (not persistent)
        const int v = atoi(ov);
        h->step_grid_cap = v > 0 ? nsm * v : 0;
    }
    // Step-kernel choice (cfg.step_kernel: 0 auto, 1 lane-per-agent, 2 env-per-thread; the environment
    // variable MAPF_STEP_KERNEL=lane|env overrides "auto").  Both are sm_100a kernels with identical results.
    h->env_threads = 0;
    h->use_env_kernel = false;
    h->env_pdl = true;
    if (const char *ov = getenv("MAPF_ENV_PDL")) h->env_pdl = atoi(ov) != 0;
    h->env_prefetch = true;
    if (const char *ov = getenv("MAPF_ENV_PREFETCH")) h->env_prefetch = atoi(ov) != 0;
    if (e1 == cudaSuccess && c.cols <= 32 && c.rows <= mapf::ENV_MAX_ROWS && !c.per_env_maps) {
        const int max_warps = 14;   // __launch_bounds__ of mapf_step_env_kernel
        const int ntiles = (c.num_envs + 31) / 32;
        int want = (ntiles + (nsm > 0 ? nsm : 1) - 1) / (nsm > 0 ? nsm : 1);  // warps per CTA for one resident wave
        if (want > max_warps) want = max_warps;
        if (want < 1) want = 1;
        if (const char *ov = getenv("MAPF_ENV_WARPS")) { const int v = atoi(ov); if (v >= 1 && v <= max_warps) want = v; }
        for (int w = want; w >= 1; --w) {
            mapf::EnvLayout E = mapf::make_env_layout(c.num_agents, c.rows, c.cols, h->SR, h->fw, w);
            if ((size_t)E.total_bytes <= kMaxSmemEnv) {
                h->env_threads = 32 * w;
                h->env_layout = E;
                break;
            }
        }
        if (h->env_threads) {
            // FAST: lifelong + lock metrics as compile-time constants, and at most 16 agents (its epilogue keeps the row and
            // the column owner masks in the two halves of one word)
            bool fast = c.lifelong_mapf != 0 && c.enable_lock_metrics != 0 && c.num_agents <= 16;
            if (const char *ov = getenv("MAPF_ENV_FAST")) fast = fast && atoi(ov) != 0;
            h->env_fn = pick_env_step(h->SR, c.num_agents % 4 == 0, fast);
            h->env_fn_many = pick_env_step(h->SR, c.num_agents % 4 == 0, fast, true);
            if (!h->env_fn) h->env_threads = 0;
        }
        if (h->env_threads) {
            e1 = cudaFuncSetAttribute(reinterpret_cast<const void *>(h->env_fn),
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmemEnv);
            if (h->env_fn_many && cudaFuncSetAttribute(reinterpret_cast<const void *>(h->env_fn_many),
                                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmemEnv) != cudaSuccess) {
                cudaGetLastError();
                h->env_fn_many = nullptr;
            }
            const int w = h->env_threads / 32;
            int grid = (ntiles + w - 1) / w;
            if (nsm > 0 && grid > nsm) grid = nsm;  // persistent: every warp walks over env tiles
            h->env_grid = grid;
        }
    }
    {
        int want_kernel = c.step_kernel;
        if (want_kernel == 0) {
            if (const char *ov = getenv("MAPF_STEP_KERNEL"))
                want_kernel = (ov[0] == 'l') ? 1 : (ov[0] == 'e') ? 2 : (ov[0] == 'p') ? 3 : 0;
        }
        // Two lanes per env (mapf_pair_kernel.cuh): same limits as the env-per-thread kernel, N a multiple of 4.  It takes
        // the env kernel's place in the handle (function, layout, CTA shape); everything downstream is shared.
        h->pair_kernel = false;
        if (want_kernel == 3 && h->env_threads && c.num_agents % 4 == 0) {
            const int max_warps = 28;   // __launch_bounds__ of mapf_step_pair_kernel
            const int ntiles16 = (c.num_envs + mapf::PAIR_EPW - 1) / mapf::PAIR_EPW;
            int want = (ntiles16 + (nsm > 0 ? nsm : 1) - 1) / (nsm > 0 ? nsm : 1);
            if (want > max_warps) want = max_warps;
            if (want < 1) want = 1;
            if (const char *ov = getenv("MAPF_PAIR_WARPS")) { const int v = atoi(ov); if (v >= 1 && v <= max_warps) want = v; }
            bool fast = c.lifelong_mapf != 0 && c.enable_lock_metrics != 0;
            if (const char *ov = getenv("MAPF_ENV_FAST")) fast = fast && atoi(ov) != 0;
            EnvKernelFn fn = pick_pair_step(h->SR, fast);
            for (int w = want; fn && w >= 1; --w) {
                mapf::EnvLayout E = mapf::make_pair_layout(c.num_agents, c.rows, c.cols, h->SR, h->fw, w);
                if ((size_t)E.total_bytes > kMaxSmemEnv) continue;
                if (cudaFuncSetAttribute(reinterpret_cast<const void *>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kMaxSmemEnv) != cudaSuccess) { cudaGetLastError(); break; }
                h->env_fn = fn;
                h->env_fn_many = nullptr;
                h->env_layout = E;
                h->env_threads = 32 * w;
                int grid = (ntiles16 + w - 1) / w;
                if (nsm > 0 && grid > nsm) grid = nsm;
                h->env_grid = grid;
                h->pair_kernel = true;
                break;
            }
        }
        if (want_kernel == 3) {
            if (!h->pair_kernel && c.step_kernel == 3) {
                delete h;
                return fail(MAPF_ERR_UNSUPPORTED,
                            "pair step kernel needs cols <= 32, rows <= 64, a shared map and num_agents %% 4 == 0 (got %dx%d, %d agents)",
                            c.rows, c.cols, c.num_agents);
            }
            want_kernel = h->pair_kernel ? 2 : 0;
        }
        if (c.step_kernel == 2 && !h->env_threads) {   // explicit request only; the environment variable is a preference
            delete h;
            return fail(MAPF_ERR_UNSUPPORTED,
                        "env-per-thread step kernel needs cols <= 32, rows <= 64 and a shared map (got %dx%d, per_env_maps=%d)",
                        c.rows, c.cols, c.per_env_maps);
        }
        // auto: the env-per-thread kernel is one latency chain per warp (~50 us on B200, whatever the batch), so it only
        // pays once the batch fills the GPU several times over (measured at 16 agents on 148 SMs, us per step env / lane:
        // 32 768 envs 49.4 / 35.0, 49 152 envs 46.7 / 51.0, 65 536 envs 59.9 / 66.2 => from 10 tiles of 32 envs per SM);
        // below that the lane-per-agent kernel has 16x more warps in flight and wins.
        const long long ntiles = (c.num_envs + 31) / 32;
        // ... and only up to 16 agents: its chain grows with N and its shared-memory footprint per warp too (fewer
        // resident warps, a second wave).  Measured at 65 536 envs, us per launch env-per-thread / lane-per-agent:
        // N=4 24.9 / 36.0, N=8 35.3 / 47.4, N=16 64.9 / 84.3, N=24 157 / 147, N=32 237 / 154.
        h->use_env_kernel = h->env_threads && (want_kernel == 2 || (want_kernel == 0 && c.num_agents <= 16 &&
                                                                    ntiles >= 10LL * (nsm > 0 ? nsm : 1)));
        (void)ntiles;
    }
    cudaError_t e3 = cudaMalloc(&h->d_err, 4);
    if (e3 == cudaSuccess) e3 = cudaMemset(h->d_err, 0, 4);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
        cudaError_t e = e1 != cudaSuccess ? e1 : e2 != cudaSuccess ? e2 : e3;
        if (h->d_err) cudaFree(h->d_err);
        delete h;
        return fail(MAPF_ERR_CUDA, "kernel setup failed: %s (built for sm_100a only)", cudaGetErrorString(e));
    }
    *out = h;
    return MAPF_OK;
}

int mapf_destroy(mapf_handle *h) {
    if (!h) return MAPF_OK;
    DeviceGuard guard(h->cfg.device);
    cudaDeviceSynchronize();
    if (h->owns_state)
        for (int i = 0; i < 10; ++i) cudaFree(*state_member(&h->st, i));
    if (h->io_alloc) {
        cudaFree(h->io_actions); cudaFree(h->io_goal_override); cudaFree(h->io_starts_override);
        cudaFree(h->io_goals_override); cudaFree(h->io_goal_rank); cudaFree(h->io_reset_mask);
        for (int i = 0; i < 10; ++i) cudaFree(*output_member(&h->io_out, i));
    }
    if (h->pack_alloc) {
        mapf::host_pool_destroy(h->pool);
        cudaFree(h->d_packed); cudaFreeHost(h->h_packed);
        cudaFreeHost(h->h_tickets);
    }
    if (h->hstream) cudaStreamDestroy(h->hstream);
    if (h->hstream2) cudaStreamDestroy(h->hstream2);
    if (h->ev_user) cudaEventDestroy(h->ev_user);
    cudaFree(h->d_map_rows); cudaFree(h->d_free_bits); cudaFree(h->d_num_free); cudaFree(h->d_err);
    cudaFree(h->d_env_tables);
    delete h;
    return MAPF_OK;
}

int mapf_set_map(mapf_handle *h, const uint8_t *grid) {
    if (!h || !grid) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    DeviceGuard guard(h->cfg.device);
    const int R = h->cfg.rows, C = h->cfg.cols, N = h->cfg.num_agents;
    const int64_t copies = h->cfg.per_env_maps ? h->cfg.num_envs : 1;
    std::vector<uint32_t> rows((size_t)copies * h->map_words, 0xFFFFFFFFu);  // padding = obstacle (OOB -> 1, ENV:718)
    std::vector<uint32_t> freeb((size_t)copies * h->fw, 0u);
    std::vector<int32_t> nfree((size_t)copies, 0);
    for (int64_t m = 0; m < copies; ++m) {
        const uint8_t *g = grid + (size_t)m * R * C;
        uint32_t *mr = rows.data() + (size_t)m * h->map_words;
        uint32_t *fb = freeb.data() + (size_t)m * h->fw;
        int F = 0;
        for (int r = 0; r < R; ++r)
            for (int c = 0; c < C; ++c) {
                const uint8_t v = g[r * C + c];
                if (v > 1) return fail(MAPF_ERR_INVALID_ARG, "grid cell (%d,%d) = %d, expected 0 or 1", r, c, v);
                if (v == 0) {  // ENV:82 free cell
                    const int bit = c + mapf::PAD;
                    mr[(r + mapf::PAD) * h->wpr + (bit >> 5)] &= ~(1u << (bit & 31));
                    const int cell = r * C + c;
                    fb[cell >> 5] |= 1u << (cell & 31);
                    ++F;
                }
            }
        nfree[m] = F;
        if (!h->cfg.deterministic && F < 2 * N)  // ENV:270-275
            return fail(MAPF_ERR_INVALID_ARG, "Not enough free cells (%d) for %d agents (need %d)", F, N, 2 * N);
    }
    cudaFree(h->d_map_rows); cudaFree(h->d_free_bits); cudaFree(h->d_num_free);
    h->d_map_rows = nullptr; h->d_free_bits = nullptr; h->d_num_free = nullptr;
    h->map_set = false;
    CUDA_TRY(cudaMalloc(&h->d_map_rows, rows.size() * 4));
    CUDA_TRY(cudaMalloc(&h->d_free_bits, freeb.size() * 4));
    CUDA_TRY(cudaMalloc(&h->d_num_free, nfree.size() * 4));
    CUDA_TRY(cudaMemcpy(h->d_map_rows, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->d_free_bits, freeb.data(), freeb.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->d_num_free, nfree.data(), nfree.size() * 4, cudaMemcpyHostToDevice));
    cudaFree(h->d_env_tables);
    h->d_env_tables = nullptr;
    if (h->env_threads) {   // table image of the env-per-thread kernel (obstacle windows, free rows, quotient tables)
        const mapf::EnvLayout &E = h->env_layout;
        std::vector<unsigned char> img((size_t)E.tables_bytes, 0);
        mapf::build_env_tables(h->SR, R, C, h->wpr, h->fw, rows.data(), freeb.data(), h->cfg.normalize_goal_delta != 0,
                               (float)(R - 1 > 1 ? R - 1 : 1), (float)(C - 1 > 1 ? C - 1 : 1), img.data(), E.pre_off);
        CUDA_TRY(cudaMalloc(&h->d_env_tables, img.size()));
        CUDA_TRY(cudaMemcpy(h->d_env_tables, img.data(), img.size(), cudaMemcpyHostToDevice));
    }
    h->map_set = true;
    return MAPF_OK;
}

int mapf_state_nbytes(const mapf_handle *h, int64_t out_nbytes[10]) {
    if (!h || !out_nbytes) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    state_sizes(h, out_nbytes);
    return MAPF_OK;
}

int mapf_bind_state(mapf_handle *h, const mapf_state *state) {
    if (!h || !state) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    mapf_state s = *state;
    for (int i = 0; i < 10; ++i)
        if (!*state_member(&s, i)) return fail(MAPF_ERR_INVALID_ARG, "mapf_state member %d is NULL", i);
    if (h->owns_state) {
        DeviceGuard guard(h->cfg.device);
        for (int i = 0; i < 10; ++i) cudaFree(*state_member(&h->st, i));
        h->owns_state = false;
    }
    h->st = s;
    h->bound = true;
    return MAPF_OK;
}

int mapf_alloc_state(mapf_handle *h) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    if (h->owns_state) return MAPF_OK;
    DeviceGuard guard(h->cfg.device);
    int64_t n[10];
    state_sizes(h, n);
    mapf_state s;
    memset(&s, 0, sizeof(s));
    for (int i = 0; i < 10; ++i) {
        CUDA_TRY(cudaMalloc(state_member(&s, i), (size_t)n[i]));
        CUDA_TRY(cudaMemset(*state_member(&s, i), 0, (size_t)n[i]));
    }
    h->st = s;
    h->bound = true;
    h->owns_state = true;
    return MAPF_OK;
}

int mapf_get_state_host(mapf_handle *h, const mapf_state *host) {
    if (!h || !host) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (!h->bound) return fail(MAPF_ERR_STATE, "no state bound");
    DeviceGuard guard(h->cfg.device);
    int64_t n[10];
    state_sizes(h, n);
    mapf_state hs = *host;
    CUDA_TRY(cudaDeviceSynchronize());
    if (!h->hstream) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    for (int i = 0; i < 10; ++i)
        if (*state_member(&hs, i))
            CUDA_TRY(cudaMemcpyAsync(*state_member(&hs, i), *state_member(&h->st, i), (size_t)n[i], cudaMemcpyDeviceToHost,
                                     h->hstream));
    CUDA_TRY(cudaStreamSynchronize(h->hstream));
    return MAPF_OK;
}

int mapf_set_state_host(mapf_handle *h, const mapf_state *host) {
    if (!h || !host) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (!h->bound) return fail(MAPF_ERR_STATE, "no state bound");
    DeviceGuard guard(h->cfg.device);
    int64_t n[10];
    state_sizes(h, n);
    mapf_state hs = *host;
    CUDA_TRY(cudaDeviceSynchronize());
    // Pageable sources: a blocking cudaMemcpy may return once the data is staged, before the DMA has landed, and the
    // next *_host call launches on a non-blocking stream that the legacy stream does not order.  Copy on the stream
    // those calls use and wait for it: when this returns the state IS on the device.
    if (!h->hstream) CUDA_TRY(cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking));
    for (int i = 0; i < 10; ++i)
        if (*state_member(&hs, i))
            CUDA_TRY(cudaMemcpyAsync(*state_member(&h->st, i), *state_member(&hs, i), (size_t)n[i], cudaMemcpyHostToDevice,
                                     h->hstream));
    CUDA_TRY(cudaStreamSynchronize(h->hstream));
    return MAPF_OK;
}

int mapf_reset(mapf_handle *h, const uint8_t *reset_mask, const int16_t *starts_override,
               const int16_t *goals_override, const mapf_outputs *out, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if ((starts_override == nullptr) != (goals_override == nullptr))
        return fail(MAPF_ERR_INVALID_ARG, "starts_override and goals_override must be given together");
    DeviceGuard guard(h->cfg.device);
    mapf::KParams p;
    fill_params(h, p);
    fill_outputs(p, out);
    p.reset_mask = reset_mask;
    p.starts_override = reinterpret_cast<const uint32_t *>(starts_override);
    p.goals_override = reinterpret_cast<const uint32_t *>(goals_override);
    return launch(h, h->reset_fn, p, static_cast<cudaStream_t>(stream));
}

int mapf_observe(mapf_handle *h, const mapf_outputs *out, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!out) return fail(MAPF_ERR_INVALID_ARG, "null outputs");
    DeviceGuard guard(h->cfg.device);
    mapf::KParams p;
    fill_params(h, p);
    fill_outputs(p, out);
    p.o_reward = nullptr; p.o_terminated = nullptr; p.o_truncated = nullptr;
    p.o_step_flags = nullptr; p.o_agent_step_flags = nullptr; p.o_info = nullptr;
    p.observe_only = 1;
    return launch(h, h->reset_fn, p, static_cast<cudaStream_t>(stream));
}

int mapf_observe_host(mapf_handle *h, const mapf_outputs *out_host) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!out_host) return fail(MAPF_ERR_INVALID_ARG, "null outputs");
    DeviceGuard guard(h->cfg.device);
    rc = ensure_io(h);
    if (rc) return rc;
    rc = order_after_user_work(h);
    if (rc) return rc;
    mapf_outputs want;
    memset(&want, 0, sizeof(want));
    want.local_obs = out_host->local_obs; want.action_mask = out_host->action_mask;
    want.goal_delta = out_host->goal_delta; want.blocking_prev = out_host->blocking_prev;
    mapf_outputs dev;
    select_outputs(h, &want, &dev);
    rc = mapf_observe(h, &dev, h->hstream);
    if (rc) return rc;
    rc = copy_outputs_back(h, &want);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->hstream));
    return MAPF_OK;
}

int mapf_step(mapf_handle *h, const int8_t *actions, const int16_t *goal_override,
              const int32_t *goal_rank, const mapf_outputs *out, int32_t auto_reset, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    mapf::KParams p;
    fill_params(h, p);
    fill_outputs(p, out);
    p.actions = actions;
    p.goal_override = reinterpret_cast<const uint32_t *>(goal_override);
    p.goal_rank = goal_rank;
    p.auto_reset = auto_reset != 0;
    if (h->fused_mode && h->fused_actions) {
        p.o_next_actions = h->fused_actions;
        p.sample_mode = h->fused_mode;
        p.sample_counter = h->fused_counter++;
    }
    return launch(h, h->step_fn, p, static_cast<cudaStream_t>(stream));
}

int mapf_step_many(mapf_handle *h, const int8_t *actions, const mapf_outputs *out, int32_t steps,
                   int64_t out_step_stride_envs, int32_t auto_reset, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (steps < 1) return fail(MAPF_ERR_INVALID_ARG, "steps must be >= 1");
    if (out_step_stride_envs != 0 && out_step_stride_envs < h->cfg.num_envs)
        return fail(MAPF_ERR_INVALID_ARG, "out_step_stride_envs must be 0 (overwrite) or >= num_envs");
    if (steps > 1 && !(h->fused_mode && h->fused_actions))
        return fail(MAPF_ERR_STATE, "mapf_step_many needs the fused sampler (mapf_set_fused_sampler): the actions of "
                                    "steps 2..K are drawn inside the launch");
    DeviceGuard guard(h->cfg.device);
    mapf::KParams p;
    fill_params(h, p);
    fill_outputs(p, out);
    p.actions = actions;
    p.auto_reset = auto_reset != 0;
    if (h->fused_mode && h->fused_actions) {
        p.o_next_actions = h->fused_actions;
        p.sample_mode = h->fused_mode;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!h->use_env_kernel) {   // lane-per-agent kernel: the K steps run inside one launch
        p.sample_counter = h->fused_counter;
        h->fused_counter += (uint64_t)steps;
        p.inner_steps = steps;
        p.out_step_stride = out_step_stride_envs;
        return launch(h, h->step_fn, p, s);
    }
    if (h->env_fn_many && steps > 1) {   // env-per-thread kernel: every warp takes its tile through the K steps in one launch
        p.sample_counter = h->fused_counter;
        h->fused_counter += (uint64_t)steps;
        p.inner_steps = steps;
        p.out_step_stride = out_step_stride_envs;
        note_user_stream(h, s);
        return launch_env_step(h, p, s, h->env_fn_many);
    }
    // two-lanes-per-env kernel: K launches, same results
    const int64_t N = h->cfg.num_agents;
    for (int t = 0; t < steps; ++t) {
        mapf::KParams q = p;
        q.actions = t == 0 ? actions : h->fused_actions;
        q.sample_counter = h->fused_counter++;
        const int64_t so = (int64_t)t * out_step_stride_envs;
        auto adv = [&](auto *&ptr, int64_t elems) { if (ptr) ptr += so * elems; };
        adv(q.o_local_obs, N * h->V2); adv(q.o_action_mask, N * 5); adv(q.o_goal_delta, N); adv(q.o_blocking_prev, N);
        adv(q.o_reward, N); adv(q.o_terminated, 1); adv(q.o_truncated, 1); adv(q.o_step_flags, 1);
        adv(q.o_agent_step_flags, N); adv(q.o_info, 4);
        rc = launch(h, h->step_fn, q, s);
        if (rc) return rc;
    }
    return MAPF_OK;
}

int mapf_reset_host(mapf_handle *h, const uint8_t *reset_mask, const int16_t *starts_override,
                    const int16_t *goals_override, const mapf_outputs *out_host) {
    int rc = check_ready(h);
    if (rc) return rc;
    if ((starts_override == nullptr) != (goals_override == nullptr))
        return fail(MAPF_ERR_INVALID_ARG, "starts_override and goals_override must be given together");
    DeviceGuard guard(h->cfg.device);
    rc = ensure_io(h);
    if (rc) return rc;
    rc = order_after_user_work(h);
    if (rc) return rc;
    const size_t B = h->cfg.num_envs, BN = B * h->cfg.num_agents;
    if (reset_mask) CUDA_TRY(cudaMemcpyAsync(h->io_reset_mask, reset_mask, B, cudaMemcpyHostToDevice, h->hstream));
    if (starts_override) {
        CUDA_TRY(cudaMemcpyAsync(h->io_starts_override, starts_override, BN * 4, cudaMemcpyHostToDevice, h->hstream));
        CUDA_TRY(cudaMemcpyAsync(h->io_goals_override, goals_override, BN * 4, cudaMemcpyHostToDevice, h->hstream));
    }
    mapf_outputs dev;
    select_outputs(h, out_host, &dev);
    rc = mapf_reset(h, reset_mask ? h->io_reset_mask : nullptr,
                    starts_override ? reinterpret_cast<const int16_t *>(h->io_starts_override) : nullptr,
                    starts_override ? reinterpret_cast<const int16_t *>(h->io_goals_override) : nullptr, &dev,
                    h->hstream);
    if (rc) return rc;
    rc = copy_outputs_back(h, out_host);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(h->hstream));
    return MAPF_OK;
}

static int step_host_impl(mapf_handle *h, const int8_t *actions, const int16_t *goal_override,
                          const int32_t *goal_rank, const mapf_outputs *out_host, int32_t auto_reset, uint8_t *records_host) {
    int rc = check_ready(h);
    if (rc) return rc;
    DeviceGuard guard(h->cfg.device);
    rc = ensure_io(h);
    if (rc) return rc;
    rc = order_after_user_work(h);
    if (rc) return rc;
    const int64_t B = h->cfg.num_envs, N = h->cfg.num_agents;
    mapf_outputs dev;
    select_outputs(h, out_host, &dev);
    if (records_host) {   // the four big channels are computed on the device and leave as records only
        dev.local_obs = h->io_out.local_obs; dev.action_mask = h->io_out.action_mask;
        dev.goal_delta = h->io_out.goal_delta; dev.reward = h->io_out.reward;
    }
    mapf::KParams p;
    fill_params(h, p);
    fill_outputs(p, &dev);
    p.actions = actions ? h->io_actions : nullptr;
    p.goal_override = goal_override ? h->io_goal_override : nullptr;
    p.goal_rank = goal_rank ? h->io_goal_rank : nullptr;
    p.auto_reset = auto_reset != 0;
    // Big batches go through in slices on two streams: the device-to-host copies of slice c (the PCIe-bound part)
    // overlap the host-to-device copy and the kernel of slice c + 1.  Envs are independent and Philox is keyed by
    // the global env id, so slicing does not change any result.  When the four big per-agent channels are all
    // requested they cross PCIe bit-packed (42 -> 13 B per agent at sensor range 2) and host threads expand slice c
    // into the caller's arrays while slice c + 1 is in flight (and while this thread is still enqueueing).
    // MAPF_HOST_RAW_32NDS=k sends the last k/32 of the batch as plain copies behind the packed slices (for hosts
    // with too few cores to keep up with PCIe; measured no gain on the 16-core B200 hosts, so 0 by default).
    // packed or plain: forced by MAPF_HOST_PACK, else measured on the first sixteen eligible calls (see mapf_handle)
    // ... three candidates: packed, packed with the expansion going through non-temporal stores (hosts whose memory
    // system is the bound: no read-for-ownership of the 45 MB it writes), plain; three calls each, the first untimed.
    // Ranks that share a node should make these calls in step (they do when they step their envs in step): a rank
    // that calibrates while the others idle sees a host that is not the one it will run on.
    bool packed = false, nt = h->knob_host_nt > 0;
    int auto_phase = -1;   // >= 0: this call is a timed calibration call for mode auto_phase
    const bool records = records_host != nullptr;
    if (records) packed = true;   // same kernels and slicing as the packed path; nothing is expanded on the host
    else if (host_pack_eligible(h, out_host)) {
        if (h->knob_host_pack >= 0) packed = h->knob_host_pack != 0;
        else if (h->auto_choice >= 0) { packed = h->auto_choice != 0; nt = h->auto_choice == 2; }
        else {
            // candidate modes in calibration order; a forced MAPF_HOST_NT leaves two of them
            int modes[3], nm = 0;
            if (h->knob_host_nt != 1) modes[nm++] = 1;
            if (h->knob_host_nt != 0) modes[nm++] = 2;
            modes[nm++] = 0;
            // four calls per candidate in a row: the first untimed (it follows a call of another mode: the expansion
            // threads may be asleep behind a plain call, the staging cold), the best of the other three counts -- one
            // hiccup (a page fault, a late worker) must not decide
            // (and four untimed calls in front of it all: kernels loaded, expansion threads created, staging touched,
            // clocks up -- none of that may count against the candidate that happens to go first)
            const int c = h->auto_calls++ - 4;
            const int mode = c < 0 ? modes[0] : modes[(c / 4) < nm ? c / 4 : nm - 1];
            packed = mode != 0; nt = mode == 2;
            if (c >= 0 && c % 4 != 0) auto_phase = mode;
            if (c + 1 >= 4 * nm) auto_phase |= 0x100;   // last calibration call: decide behind it
        }
    }

    if (packed) {
        rc = ensure_pack(h);
        if (rc) return rc;
        if (!records) mapf::host_pool_set_nt(h->pool, nt);
    }
    // slice sizes as weights: uniform by default; the packed path tapers them (small first slice: its records are
    // on the wire early; small last slice: the expansion nobody overlaps is short).  MAPF_HOST_SLICES=n -> n
    // uniform slices, MAPF_HOST_PLAN=w0,w1,... -> explicit weights.
    int weights[kMaxHostSlices];
    int nslices = B >= 8192 ? 2 : 1;
    for (int i = 0; i < kMaxHostSlices; ++i) weights[i] = 1;
    if (records && B < 8192) nslices = 1;
    if (packed && B >= 32768) {
        // measured on B200 / PCIe Gen5 / 16 host cores at 65 536 x 16 (e9 agent-steps/s): 1,1 1.88 | 1,1,1,1 2.19 |
        // 1,3,4,4,3,1 2.26 | 2,4,4,4,2 2.36 | 1,2,3,4,3,2,1 2.16
        static const int taper[5] = {2, 4, 4, 4, 2};
        nslices = 5;
        for (int i = 0; i < 5; ++i) weights[i] = taper[i];
    }
    if (h->knob_host_slices >= 1) {
        nslices = h->knob_host_slices;
        for (int i = 0; i < kMaxHostSlices; ++i) weights[i] = 1;
    }
    if (h->knob_plan_n >= 1) {
        nslices = h->knob_plan_n;
        for (int i = 0; i < nslices; ++i) weights[i] = h->knob_plan[i];
    }
    const int raw32 = (packed && !records) ? h->knob_raw32 : 0;
    struct HostSlice { int64_t e0, n; bool packed; };
    HostSlice plan[kMaxHostSlices + 1];
    int S = 0;
    const int64_t Bp = B - (B * raw32 / 32) / 32 * 32;  // envs [0, Bp): sliced (packed if applicable); [Bp, B): plain tail
    {
        int wsum = 0, wacc = 0;
        for (int i = 0; i < nslices; ++i) wsum += weights[i];
        int64_t e0 = 0;
        for (int i = 0; i < nslices && e0 < Bp; ++i) {
            wacc += weights[i];
            int64_t e1 = (i == nslices - 1) ? Bp : (Bp * wacc / wsum + 31) / 32 * 32;
            if (e1 > Bp) e1 = Bp;
            if (e1 > e0) plan[S++] = HostSlice{e0, e1 - e0, packed};
            e0 = e1;
        }
    }
    if (Bp < B) plan[S++] = HostSlice{Bp, B - Bp, false};
    int64_t n_out[10];
    output_sizes(h, n_out);
    mapf_outputs host_tmp;
    memset(&host_tmp, 0, sizeof(host_tmp));
    if (out_host) host_tmp = *out_host;
    const int RS = mapf::pack_record_bytes(h->V2);
    const float inv0 = h->cfg.normalize_goal_delta ? (float)(h->cfg.rows - 1 > 1 ? h->cfg.rows - 1 : 1) : 1.f;
    const float inv1 = h->cfg.normalize_goal_delta ? (float)(h->cfg.cols - 1 > 1 ? h->cfg.cols - 1 : 1) : 1.f;
    int64_t h2d = 0, d2h = 0;
    const uint32_t ticket = ++h->ticket_seq;
    const bool trace = packed && !records && h->knob_trace;
    const int64_t t_begin = std::chrono::steady_clock::now().time_since_epoch().count();
    // closes the step for the host threads on every exit path (an early error return must not leave them polling)
    struct PoolStep {
        mapf::HostPool *pool = nullptr;
        ~PoolStep() { if (pool) mapf::host_pool_finish(pool); }
    } pool_step;
    if (packed && !records) {
        mapf::host_pool_begin(h->pool);
        pool_step.pool = h->pool;
    }
    const int PBr = mapf::pack_obs_bytes(h->V2);   // batch-wide record streams: [BN x PBr bits][BN x 2 diffs][BN x 1 reward]
    for (int c = 0; c < S; ++c) {
        const int64_t e0 = plan[c].e0, n = plan[c].n;
        cudaStream_t st = (c & 1) ? h->hstream2 : h->hstream;
        if (actions) {
            CUDA_TRY(cudaMemcpyAsync(h->io_actions + e0 * N, actions + e0 * N, (size_t)(n * N), cudaMemcpyHostToDevice, st));
            h2d += n * N;
        }
        if (goal_override) {
            CUDA_TRY(cudaMemcpyAsync(h->io_goal_override + e0 * N, goal_override + e0 * N * 2, (size_t)(n * N * 4),
                                     cudaMemcpyHostToDevice, st));
            h2d += n * N * 4;
        }
        if (goal_rank) {
            CUDA_TRY(cudaMemcpyAsync(h->io_goal_rank + e0 * N, goal_rank + e0 * N, (size_t)(n * N * 4), cudaMemcpyHostToDevice, st));
            h2d += n * N * 4;
        }
        if (S == 1) {
            rc = launch(h, h->step_fn, p, st);
        } else {
            rc = launch_step_range(h, p, e0, (int)n, st);
        }
        if (rc) return rc;
        if (plan[c].packed && records) {
            // records delivery: the slice's share of the three batch-wide streams, straight into the caller's buffer
            const int64_t a0 = e0 * N, na = n * N, BN = B * N;
            uint8_t *d_bits = h->d_packed + a0 * PBr, *d_diff = h->d_packed + BN * PBr + a0 * 2, *d_rew = h->d_packed + BN * (PBr + 2) + a0;
            const int threads = 256;
            mapf::mapf_pack_host_kernel<<<(unsigned)((na + threads - 1) / threads), threads, threads * RS + 4, st>>>(
                h->io_out.local_obs + a0 * h->V2, h->io_out.action_mask + a0 * 5,
                reinterpret_cast<const float2 *>(h->io_out.goal_delta) + a0, h->io_out.reward + a0, d_bits, na, h->V2,
                inv0, inv1, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, d_diff, d_rew);
            CUDA_TRY(cudaGetLastError());
            h->launches++;
            CUDA_TRY(cudaMemcpyAsync(records_host + a0 * PBr, d_bits, (size_t)(na * PBr), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(records_host + BN * PBr + a0 * 2, d_diff, (size_t)(na * 2), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(records_host + BN * (PBr + 2) + a0, d_rew, (size_t)na, cudaMemcpyDeviceToHost, st));
            d2h += na * RS;
        } else if (plan[c].packed) {
            // one block, one DMA per slice: the three packed streams, then the requested byte channels as they are
            const int64_t a0 = e0 * N, na = n * N;
            uint8_t *blk = h->d_packed + a0 * (RS + 1) + e0 * 3;
            int64_t off = na * RS;
            uint8_t *b_bp = nullptr, *b_env[3] = {nullptr, nullptr, nullptr};
            if (host_tmp.blocking_prev) { b_bp = blk + off; off += na; }
            for (int i = 5; i <= 7; ++i)
                if (*output_member(&host_tmp, i)) { b_env[i - 5] = blk + off; off += n; }
            const int threads = 256;
            mapf::mapf_pack_host_kernel<<<(unsigned)((na + threads - 1) / threads), threads, threads * RS + 4, st>>>(
                h->io_out.local_obs + a0 * h->V2, h->io_out.action_mask + a0 * 5,
                reinterpret_cast<const float2 *>(h->io_out.goal_delta) + a0, h->io_out.reward + a0, blk, na, h->V2,
                inv0, inv1, h->io_out.blocking_prev + a0, b_bp, h->io_out.terminated + e0, b_env[0],
                h->io_out.truncated + e0, b_env[1], h->io_out.step_flags + e0, b_env[2], n);
            CUDA_TRY(cudaGetLastError());
            h->launches++;
            CUDA_TRY(cudaMemcpyAsync(h->h_packed + (blk - h->d_packed), blk, (size_t)off, cudaMemcpyDeviceToHost, st));
            d2h += off;
        }
        for (int i = 0; i < 10; ++i) {
            char *dst = static_cast<char *>(*output_member(&host_tmp, i));
            if (!dst || (plan[c].packed && !records && i <= 7)) continue;  // everything but agent_step_flags / info rides in the block
            const int64_t per_env = n_out[i] / B;
            CUDA_TRY(cudaMemcpyAsync(dst + e0 * per_env, static_cast<char *>(*output_member(&h->io_out, i)) + e0 * per_env,
                                     (size_t)(n * per_env), cudaMemcpyDeviceToHost, st));
            d2h += n * per_env;
        }
        if (plan[c].packed && !records) {
            // the slice's ticket: written into pinned host memory behind the block's copy; the host threads start on
            // the job when they see it (no CUDA call, no event wait on their side)
            mapf::mapf_ticket_kernel<<<1, 1, 0, st>>>(h->h_tickets + c, ticket);
            CUDA_TRY(cudaGetLastError());
            h->launches++;
            const int64_t a0 = e0 * N, na = n * N;
            const uint8_t *blk = h->h_packed + a0 * (RS + 1) + e0 * 3;
            mapf::UnpackJob job;
            job.packed = blk;
            job.a0 = a0; job.a1 = a0 + na;
            job.V2 = h->V2;
            job.obs = host_tmp.local_obs; job.mask = host_tmp.action_mask; job.goal_delta = host_tmp.goal_delta;
            job.reward = host_tmp.reward;
            job.gdt_row = h->gdt_row; job.gdt_col = h->gdt_col;
            job.den_row = inv0; job.den_col = inv1;
            job.bytes_src = host_tmp.blocking_prev ? blk + na * RS : nullptr;
            job.bytes_dst = host_tmp.blocking_prev;
            if (!mapf::host_pool_submit(h->pool, job, h->h_tickets + c, ticket))
                return fail(MAPF_ERR_STATE, "host expansion queue overflow");
        }
    }
    const int64_t t_enq = std::chrono::steady_clock::now().time_since_epoch().count();
    if (packed && !records) {
        pool_step.pool = nullptr;
        if (!mapf::host_pool_finish(h->pool)) {  // this thread joins in; returns when every slice is expanded
            const cudaError_t e = cudaDeviceSynchronize();
            return fail(MAPF_ERR_CUDA, "mapf_step_host: a slice never arrived on the host (%s)", cudaGetErrorString(e));
        }
        for (int c = 0; c < S; ++c) {     // per-env byte channels: a few KB, copied here
            if (!plan[c].packed) continue;
            const int64_t e0 = plan[c].e0, n = plan[c].n, na = n * N;
            const uint8_t *blk = h->h_packed + e0 * N * (RS + 1) + e0 * 3;
            int64_t off = na * RS + (host_tmp.blocking_prev ? na : 0);
            for (int i = 5; i <= 7; ++i)
                if (void *dst = *output_member(&host_tmp, i)) {
                    memcpy(static_cast<char *>(dst) + e0, blk + off, (size_t)n);
                    off += n;
                }
        }
    }
    CUDA_TRY(cudaStreamSynchronize(h->hstream));
    if (S > 1) CUDA_TRY(cudaStreamSynchronize(h->hstream2));
    if (trace) {  // where the time of one call went (microseconds since entry)
        const int64_t t_end = std::chrono::steady_clock::now().time_since_epoch().count();
        fprintf(stderr, "mapf_step_host: enqueued %.0f", (t_enq - t_begin) * 1e-3);
        int q = 0;
        for (int c = 0; c < S; ++c) {
            if (!plan[c].packed) continue;
            int64_t f = 0, l = 0;
            mapf::host_pool_job_times(h->pool, q++, &f, &l);
            fprintf(stderr, " | slice %d (%lld envs) %.0f-%.0f", c, (long long)plan[c].n, (f - t_begin) * 1e-3, (l - t_begin) * 1e-3);
        }
        fprintf(stderr, " | done %.0f us\n", (t_end - t_begin) * 1e-3);
    }
    h->last_h2d_bytes = h2d;
    h->last_d2h_bytes = d2h;
    if (auto_phase >= 0) {
        {   // the best of a mode's timed calls: one hiccup (a page fault, a late worker) must not decide
            const int64_t dt = std::chrono::steady_clock::now().time_since_epoch().count() - t_begin;
            int64_t &slot = h->auto_ns[auto_phase & 0xFF];
            if (slot == 0 || dt < slot) slot = dt;
        }
        if (auto_phase & 0x100) {
            // every candidate has its best of three timed calls.  In order of preference -- packed, packed + NT, plain:
            // fewest PCIe bytes, least host memory traffic per byte -- a later one has to win by 10 % (single calls
            // are not timed better than that; where the host decides the margin is 30 % and more)
            int best = -1;
            const int order[3] = {1, 2, 0};
            for (int i = 0; i < 3; ++i) {
                const int m = order[i];
                if (h->auto_ns[m] <= 0) continue;
                if (best < 0 || h->auto_ns[m] * 10 < h->auto_ns[best] * 9) best = m;
            }
            h->auto_choice = best < 0 ? 1 : best;
        }
    }
    return MAPF_OK;
}

int mapf_host_wait_stream(mapf_handle *h, void *stream) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    h->last_user_stream = static_cast<cudaStream_t>(stream);
    h->user_dirty = true;
    return MAPF_OK;
}

int mapf_step_host(mapf_handle *h, const int8_t *actions, const int16_t *goal_override,
                   const int32_t *goal_rank, const mapf_outputs *out_host, int32_t auto_reset) {
    return step_host_impl(h, actions, goal_override, goal_rank, out_host, auto_reset, nullptr);
}

int mapf_step_host_records(mapf_handle *h, const int8_t *actions, uint8_t *records_host, const mapf_outputs *out_host_small,
                           int32_t auto_reset) {
    if (!records_host) return fail(MAPF_ERR_INVALID_ARG, "null records buffer");
    if (h && (h->cfg.rows > 128 || h->cfg.cols > 128))
        return fail(MAPF_ERR_UNSUPPORTED, "records carry the goal difference as int8: maps up to 128 x 128");
    if (out_host_small && (out_host_small->local_obs || out_host_small->action_mask || out_host_small->goal_delta ||
                           out_host_small->reward))
        return fail(MAPF_ERR_INVALID_ARG, "local_obs / action_mask / goal_delta / reward arrive as records: leave them NULL");
    return step_host_impl(h, actions, nullptr, nullptr, out_host_small, auto_reset, records_host);
}

int mapf_host_memory_probe(const mapf_handle *h, int64_t bytes, int32_t *threads_out, double *fill_gbs, double *copy_gbs) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    if (bytes < (1 << 20)) return fail(MAPF_ERR_INVALID_ARG, "probe at least 1 MiB");
    int cpus[64];
    int n = 0;
    const bool pin = h->knob_host_pin >= 0 ? h->knob_host_pin != 0 : h->local_world > 1;
    if (pin) n = rank_cores(h, cpus, 64);
    const int threads = host_threads_default(h);
    mapf::host_memory_probe(threads, bytes, n > 0 ? cpus : nullptr, n, fill_gbs, copy_gbs);
    if (threads_out) *threads_out = threads;
    return MAPF_OK;
}

int mapf_host_transfer_bytes(const mapf_handle *h, int64_t *h2d_bytes, int64_t *d2h_bytes) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    if (h2d_bytes) *h2d_bytes = h->last_h2d_bytes;
    if (d2h_bytes) *d2h_bytes = h->last_d2h_bytes;
    return MAPF_OK;
}

int mapf_host_transfer_mode(const mapf_handle *h) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    if (h->knob_host_pack == 0) return 0;
    if (h->knob_host_pack > 0) return h->knob_host_nt > 0 ? 2 : 1;
    return h->auto_choice;
}

int mapf_packed_record_bytes(int32_t v2) { return v2 >= 1 ? mapf::pack_record_bytes(v2) : 0; }

int mapf_unpack_records(const uint8_t *packed, int64_t n_agents, int32_t v2, int32_t threads, uint8_t *local_obs,
                        int8_t *action_mask, float *goal_delta, float *reward, float den_row, float den_col) {
    if (!packed || !local_obs || !action_mask || !goal_delta || !reward) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (n_agents < 0 || (v2 != 9 && v2 != 25 && v2 != 49) || threads < 1 || !(den_row > 0.f) || !(den_col > 0.f))
        return fail(MAPF_ERR_INVALID_ARG, "bad argument (v2 must be 9, 25 or 49; denominators > 0)");
    float gdt_row[256], gdt_col[256];
    for (int d = -128; d < 128; ++d) {
        gdt_row[d + 128] = (float)d / den_row;
        gdt_col[d + 128] = (float)d / den_col;
    }
    mapf::HostPool *pool = mapf::host_pool_create(threads);
    mapf::UnpackJob job;
    job.packed = packed; job.a0 = 0; job.a1 = n_agents; job.V2 = v2;
    job.obs = local_obs; job.mask = action_mask; job.goal_delta = goal_delta; job.reward = reward;
    job.gdt_row = gdt_row; job.gdt_col = gdt_col; job.den_row = den_row; job.den_col = den_col;
    job.bytes_src = nullptr; job.bytes_dst = nullptr;
    mapf::host_pool_unpack(pool, job);
    mapf::host_pool_destroy(pool);
    return MAPF_OK;
}

int mapf_flat_obs_dim(const mapf_handle *h, int32_t include_goal_distance, int32_t include_blocking_pressure,
                      int32_t include_action_mask) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    return h->V2 + 2 + (include_goal_distance ? 1 : 0) + (include_blocking_pressure ? 1 : 0) +
           (include_action_mask ? 5 : 0);
}

int mapf_pack_flat_obs(mapf_handle *h, const mapf_outputs *ch, int32_t include_goal_distance,
                       int32_t include_blocking_pressure, int32_t include_action_mask, float *flat,
                       void *stream) {
    if (!h || !ch || !flat) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (!ch->local_obs || !ch->goal_delta) return fail(MAPF_ERR_INVALID_ARG, "local_obs and goal_delta are required");
    if (include_blocking_pressure && !ch->blocking_prev) return fail(MAPF_ERR_INVALID_ARG, "blocking_prev is required");
    if (include_action_mask && !ch->action_mask) return fail(MAPF_ERR_INVALID_ARG, "action_mask is required");
    DeviceGuard guard(h->cfg.device);
    const int D = mapf_flat_obs_dim(h, include_goal_distance, include_blocking_pressure, include_action_mask);
    const long long BN = (long long)h->cfg.num_envs * h->cfg.num_agents;
    const long long total = BN * D;
    const int threads = 256;
    const unsigned grid = (unsigned)((total + threads - 1) / threads);
    note_user_stream(h, static_cast<cudaStream_t>(stream));
    mapf::mapf_pack_flat_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(
        ch->local_obs, reinterpret_cast<const float2 *>(ch->goal_delta), ch->blocking_prev, ch->action_mask, flat,
        BN, h->V2, include_goal_distance ? 1 : 0, include_blocking_pressure ? 1 : 0, include_action_mask ? 1 : 0, D);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

static int sample_actions(mapf_handle *h, const int8_t *mask, int8_t *actions, uint64_t counter, void *stream) {
    if (!h || !actions) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    DeviceGuard guard(h->cfg.device);
    const long long BN = (long long)h->cfg.num_envs * h->cfg.num_agents;
    const int threads = 256;
    const unsigned grid = (unsigned)((BN + threads - 1) / threads);
    note_user_stream(h, static_cast<cudaStream_t>(stream));
    mapf::mapf_sample_actions_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(
        mask, actions, BN, h->cfg.num_agents, h->cfg.seed, h->cfg.env_id_base, counter);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

int mapf_sample_masked_actions(mapf_handle *h, const int8_t *action_mask, int8_t *actions, uint64_t counter,
                               void *stream) {
    if (!action_mask) return fail(MAPF_ERR_INVALID_ARG, "null action_mask");
    return sample_actions(h, action_mask, actions, counter, stream);
}

int mapf_sample_random_actions(mapf_handle *h, int8_t *actions, uint64_t counter, void *stream) {
    return sample_actions(h, nullptr, actions, counter, stream);
}

int mapf_set_fused_sampler(mapf_handle *h, int8_t *next_actions, int32_t mode, uint64_t first_counter) {
    if (!h) return fail(MAPF_ERR_INVALID_ARG, "null handle");
    if (mode < 0 || mode > 2) return fail(MAPF_ERR_INVALID_ARG, "sampler mode %d outside 0..2", mode);
    if (mode != 0 && !next_actions) return fail(MAPF_ERR_INVALID_ARG, "null next_actions");
    h->fused_actions = next_actions;
    h->fused_mode = mode;
    h->fused_counter = first_counter;
    return MAPF_OK;
}

int mapf_metrics_reduce(mapf_handle *h, double *out_device, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!out_device) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    DeviceGuard guard(h->cfg.device);
    mapf::mapf_metrics_reduce_kernel<<<MAPF_METRIC_COUNT, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        h->st.env_metrics, h->cfg.num_envs, out_device);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

// the heat-map launch of mapf_occupancy_accumulate and mapf_cte_eval_accumulate: positions are packed uint32 words
// (row in the low 16 bits, column in the high 16 bits, both signed), one per agent
static void occupancy_launch(const uint32_t *positions, const uint8_t *active, int num_envs, int num_agents, int rows,
                             int cols, uint64_t *counts, void *stream) {
    const long long BN = (long long)num_envs * num_agents;
    const int cells = rows * cols;
    const int use_smem = cells * 4 <= 48 * 1024;
    const int threads = 256;
    long long blocks = (BN + threads * 8 - 1) / (threads * 8);
    if (blocks > 1184) blocks = 1184;
    if (blocks < 1) blocks = 1;
    mapf::mapf_occupancy_kernel<<<(unsigned)blocks, threads, use_smem ? cells * 4 : 0, static_cast<cudaStream_t>(stream)>>>(
        positions, active, BN, num_agents, rows, cols, reinterpret_cast<unsigned long long *>(counts), use_smem);
}

int mapf_occupancy_accumulate(mapf_handle *h, const uint8_t *active, uint64_t *counts, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!counts) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    DeviceGuard guard(h->cfg.device);
    occupancy_launch(reinterpret_cast<const uint32_t *>(h->st.positions), active, h->cfg.num_envs, h->cfg.num_agents,
                     h->cfg.rows, h->cfg.cols, counts, stream);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

int mapf_distance_table(mapf_handle *h, uint8_t *table, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!table) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (h->cfg.per_env_maps || h->cfg.rows > 32 || h->cfg.cols > 32)
        return fail(MAPF_ERR_UNSUPPORTED, "distance table needs one shared map of at most 32x32 cells (got %dx%d, per_env_maps=%d)",
                    h->cfg.rows, h->cfg.cols, h->cfg.per_env_maps);
    DeviceGuard guard(h->cfg.device);
    const int cells = h->cfg.rows * h->cfg.cols, warps = 8;
    mapf::mapf_distance_table_kernel<<<(cells + warps - 1) / warps, warps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        h->d_free_bits, h->cfg.rows, h->cfg.cols, table);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

int mapf_goal_path_lengths(mapf_handle *h, const uint8_t *table, int16_t *out, void *stream) {
    int rc = check_ready(h);
    if (rc) return rc;
    if (!table || !out) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    DeviceGuard guard(h->cfg.device);
    const long long BN = (long long)h->cfg.num_envs * h->cfg.num_agents;
    mapf::mapf_goal_path_lengths_kernel<<<(unsigned)((BN + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const uint32_t *>(h->st.positions), reinterpret_cast<const uint32_t *>(h->st.goals), table, BN,
        h->cfg.rows, h->cfg.cols, out);
    CUDA_TRY(cudaGetLastError());
    h->launches++;
    return MAPF_OK;
}

int mapf_poll_errors(mapf_handle *h, uint32_t *bits, void *stream) {
    if (!h || !bits) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    DeviceGuard guard(h->cfg.device);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemcpyAsync(bits, h->d_err, 4, cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemsetAsync(h->d_err, 0, 4, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    if (h->hstream && s != h->hstream) {
        // the *_host entry points run on the handle's own stream and are synchronous, nothing pending
    }
    return MAPF_OK;
}

static int cte_launch(const mapf_cte_args *a, int mode, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (a->num_envs < 1 || a->num_agents < 1 || a->num_agents > MAPF_MAX_AGENTS || a->rows < 1 || a->cols < 1 ||
        a->rows > MAPF_MAX_DIM || a->cols > MAPF_MAX_DIM)
        return fail(MAPF_ERR_UNSUPPORTED, "cte: num_envs=%d num_agents=%d map %dx%d outside the supported range",
                    a->num_envs, a->num_agents, a->rows, a->cols);
    if (!a->grid || !a->positions || !a->goals || !a->reached_once || !a->step_count || !a->blocking_total || !a->err_bits)
        return fail(MAPF_ERR_INVALID_ARG, "cte: grid / state / err_bits pointers are required");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    const int threads = 128;
    const unsigned grid = (unsigned)((a->num_envs + threads - 1) / threads);
    mapf::mapf_cte_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(*a, mode);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_cte_step(const mapf_cte_args *a, void *stream) { return cte_launch(a, 0, stream); }
int mapf_cte_reset(const mapf_cte_args *a, void *stream) { return cte_launch(a, 1, stream); }

static int policy_kc1(int F) { return F < 1 ? 0 : F <= 32 ? 2 : F <= 64 ? 4 : 0; }

int64_t mapf_policy_weights_nbytes(int32_t F) {
    const int kc1 = policy_kc1(F);
    if (!kc1) return fail(MAPF_ERR_UNSUPPORTED, "policy: feature_dim %d outside 1..64", F);
    const int s1 = 16 * kc1 + 8;
    return (int64_t)(mapf::POL_H * s1 + mapf::POL_H * mapf::POL_W2_STRIDE + 8 * mapf::POL_W2_STRIDE) * 2 + (2 * mapf::POL_H + 8) * 4;
}

int mapf_policy_pack_weights(int32_t F, const float *w1, const float *b1, const float *w2, const float *b2,
                             const float *wl, const float *bl, const float *wv, const float *bv, void *packed) {
    const int kc1 = policy_kc1(F);
    if (!kc1) return fail(MAPF_ERR_UNSUPPORTED, "policy: feature_dim %d outside 1..64", F);
    if (!w1 || !b1 || !w2 || !b2 || !wl || !bl || !wv || !bv || !packed) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    const int s1 = 16 * kc1 + 8, H = mapf::POL_H, S2 = mapf::POL_W2_STRIDE;
    memset(packed, 0, (size_t)mapf_policy_weights_nbytes(F));
    __nv_bfloat16 *p1 = static_cast<__nv_bfloat16 *>(packed), *p2 = p1 + H * s1, *p3 = p2 + H * S2;
    float *pb = reinterpret_cast<float *>(p3 + 8 * S2);
    for (int o = 0; o < H; ++o) {
        for (int i = 0; i < F; ++i) p1[o * s1 + i] = __float2bfloat16_rn(w1[o * F + i]);
        for (int i = 0; i < H; ++i) p2[o * S2 + i] = __float2bfloat16_rn(w2[o * H + i]);
        pb[o] = b1[o];
        pb[H + o] = b2[o];
    }
    for (int o = 0; o < 5; ++o) {
        for (int i = 0; i < H; ++i) p3[o * S2 + i] = __float2bfloat16_rn(wl[o * H + i]);
        pb[2 * H + o] = bl[o];
    }
    for (int i = 0; i < H; ++i) p3[5 * S2 + i] = __float2bfloat16_rn(wv[i]);
    pb[2 * H + 5] = bv[0];
    return MAPF_OK;
}

static int policy_launch(const mapf_policy_args *a, bool per_agent, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    const int kc1 = policy_kc1(a->feature_dim);
    if (!kc1 || a->v2 < 1 || a->feature_dim != a->v2 + 2 + (a->blocking_prev ? 1 : 0))
        return fail(MAPF_ERR_UNSUPPORTED, "policy: feature_dim %d does not match v2 %d (+2 goal delta, +1 pressure) or exceeds 64",
                    a->feature_dim, a->v2);
    if (a->num_envs < 1 || a->num_agents < 1 || !a->local_obs || !a->goal_delta || !a->weights)
        return fail(MAPF_ERR_INVALID_ARG, "policy: env outputs and weights are required");
    if (a->greedy != 0 && a->greedy != 1) return fail(MAPF_ERR_INVALID_ARG, "policy: greedy %d is neither 0 nor 1", a->greedy);
    if (per_agent && a->num_agents > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "policy: num_agents %d exceeds %d", a->num_agents, MAPF_MAX_AGENTS);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    const int threads = 256, warps = threads / 32;
    const size_t smem = (size_t)mapf_policy_weights_nbytes(a->feature_dim) + (size_t)warps * mapf::pol_warp_bytes(kc1, a->v2);
    // a per-agent tile holds one agent's rows: ceil(B / 32) tiles per agent
    const long long tiles = per_agent ? ((long long)a->num_envs + 31) / 32 * a->num_agents
                                      : ((long long)a->num_envs * a->num_agents + 31) / 32;
    long long blocks = (tiles + warps - 1) / warps;
    if (blocks > 148 * 8) blocks = 148 * 8;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    void (*const kernels[2][2][2])(const mapf_policy_args) = {
        {{mapf::mapf_policy_act_kernel<2, false>, mapf::mapf_policy_act_kernel<2, true>},
         {mapf::mapf_policy_act_kernel<4, false>, mapf::mapf_policy_act_kernel<4, true>}},
        {{mapf::mapf_policy_act_kernel<2, false, true>, mapf::mapf_policy_act_kernel<2, true, true>},
         {mapf::mapf_policy_act_kernel<4, false, true>, mapf::mapf_policy_act_kernel<4, true, true>}}};
    const auto kernel = kernels[per_agent][kc1 == 4][a->greedy];
    CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<(unsigned)blocks, threads, smem, st>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_policy_act(const mapf_policy_args *a, void *stream) { return policy_launch(a, false, stream); }
int mapf_policy_act_per_agent(const mapf_policy_args *a, void *stream) { return policy_launch(a, true, stream); }

int64_t mapf_lstm_policy_weights_nbytes(int32_t F) {
    const int kc1 = policy_kc1(F);
    if (!kc1) return fail(MAPF_ERR_UNSUPPORTED, "lstm policy: feature_dim %d outside 1..64", F);
    return mapf::lstm_weight_bytes(kc1);
}

int mapf_lstm_policy_pack_weights(int32_t F, const float *w1, const float *b1, const float *w2, const float *b2,
                                  const float *w_ih, const float *w_hh, const float *b_ih, const float *b_hh,
                                  const float *wl, const float *bl, const float *wv, const float *bv, void *packed) {
    const int kc1 = policy_kc1(F);
    if (!kc1) return fail(MAPF_ERR_UNSUPPORTED, "lstm policy: feature_dim %d outside 1..64", F);
    if (!w1 || !b1 || !w2 || !b2 || !w_ih || !w_hh || !b_ih || !b_hh || !wl || !bl || !wv || !bv || !packed)
        return fail(MAPF_ERR_INVALID_ARG, "null argument");
    const int s1 = 16 * kc1 + 8, H = mapf::POL_H, S2 = mapf::POL_W2_STRIDE, SG = mapf::LSTM_SG, KI = H + 5 + 1;
    memset(packed, 0, (size_t)mapf::lstm_weight_bytes(kc1));
    __nv_bfloat16 *p1 = static_cast<__nv_bfloat16 *>(packed), *p2 = p1 + H * s1, *p3 = p2 + H * S2, *pg = p3 + 8 * S2;
    float *pb = reinterpret_cast<float *>(pg + 4 * H * SG);
    for (int o = 0; o < H; ++o) {
        for (int i = 0; i < F; ++i) p1[o * s1 + i] = __float2bfloat16_rn(w1[o * F + i]);
        for (int i = 0; i < H; ++i) p2[o * S2 + i] = __float2bfloat16_rn(w2[o * H + i]);
        pb[o] = b1[o];
        pb[H + o] = b2[o];
    }
    for (int o = 0; o < 5; ++o) {
        for (int i = 0; i < H; ++i) p3[o * S2 + i] = __float2bfloat16_rn(wl[o * H + i]);
        pb[2 * H + o] = bl[o];
    }
    for (int i = 0; i < H; ++i) p3[5 * S2 + i] = __float2bfloat16_rn(wv[i]);
    pb[2 * H + 5] = bv[0];
    for (int o = 0; o < 4 * H; ++o) {   // [W_ih (70 cols) | 10 zero cols | W_hh (64 cols)]
        for (int i = 0; i < KI; ++i) pg[o * SG + i] = __float2bfloat16_rn(w_ih[o * KI + i]);
        for (int i = 0; i < H; ++i) pg[o * SG + mapf::LSTM_KX + i] = __float2bfloat16_rn(w_hh[o * H + i]);
        pb[2 * H + 8 + o] = b_ih[o] + b_hh[o];
    }
    return MAPF_OK;
}

static int lstm_policy_launch(const mapf_lstm_policy_args *a, bool per_agent, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    const int kc1 = policy_kc1(a->feature_dim);
    if (!kc1 || a->v2 < 1 || a->feature_dim != a->v2 + 2 + (a->blocking_prev ? 1 : 0))
        return fail(MAPF_ERR_UNSUPPORTED, "lstm policy: feature_dim %d does not match v2 %d (+2 goal delta, +1 pressure) or exceeds 64",
                    a->feature_dim, a->v2);
    if (a->num_envs < 1 || a->num_agents < 1 || !a->local_obs || !a->goal_delta || !a->weights)
        return fail(MAPF_ERR_INVALID_ARG, "lstm policy: env outputs and weights are required");
    if (!a->prev_action || !a->prev_reward || !a->h_in || !a->c_in)
        return fail(MAPF_ERR_INVALID_ARG, "lstm policy: prev_action, prev_reward, h_in and c_in are required");
    if (!a->h_out != !a->c_out)
        return fail(MAPF_ERR_INVALID_ARG, "lstm policy: h_out and c_out are given together (both NULL = state not advanced)");
    if (a->greedy != 0 && a->greedy != 1)
        return fail(MAPF_ERR_INVALID_ARG, "lstm policy: greedy %d is neither 0 nor 1", a->greedy);
    if (per_agent && a->num_agents > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "lstm policy: num_agents %d exceeds %d", a->num_agents, MAPF_MAX_AGENTS);
    int ndev = 0, dev = 0, sms = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int threads = mapf::LSTM_THREADS, warps = threads / 32;
    const size_t smem = (size_t)mapf::lstm_weight_bytes(kc1) + (size_t)warps * mapf::pol_warp_bytes(kc1, a->v2);
    const long long tiles = per_agent ? ((long long)a->num_envs + 31) / 32 * a->num_agents
                                      : ((long long)a->num_envs * a->num_agents + 31) / 32;
    long long blocks = (tiles + warps - 1) / warps;
    // one resident block per SM loads the weights once (per agent: once per agent of its tile range) and loops over
    // the tiles
    if (blocks > sms) blocks = sms;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    void (*const kernels[2][2][2])(const mapf_lstm_policy_args) = {
        {{mapf::mapf_lstm_policy_act_kernel<2, false>, mapf::mapf_lstm_policy_act_kernel<2, true>},
         {mapf::mapf_lstm_policy_act_kernel<4, false>, mapf::mapf_lstm_policy_act_kernel<4, true>}},
        {{mapf::mapf_lstm_policy_act_kernel<2, false, true>, mapf::mapf_lstm_policy_act_kernel<2, true, true>},
         {mapf::mapf_lstm_policy_act_kernel<4, false, true>, mapf::mapf_lstm_policy_act_kernel<4, true, true>}}};
    const auto kernel = kernels[per_agent][kc1 == 4][a->greedy];
    CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<(unsigned)blocks, threads, smem, st>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_lstm_policy_act(const mapf_lstm_policy_args *a, void *stream) { return lstm_policy_launch(a, false, stream); }
int mapf_lstm_policy_act_per_agent(const mapf_lstm_policy_args *a, void *stream) { return lstm_policy_launch(a, true, stream); }

static bool cte_policy_shape_ok(int cells, int n) {
    return cells >= 1 && cells <= MAPF_CTE_POLICY_MAX_CELLS && n >= 1 && n <= MAPF_MAX_AGENTS;
}

int64_t mapf_cte_policy_weights_nbytes(int32_t cells, int32_t num_agents) {
    if (!cte_policy_shape_ok(cells, num_agents))
        return fail(MAPF_ERR_UNSUPPORTED, "cte policy: cells %d / num_agents %d outside 1..%d / 1..%d", cells, num_agents,
                    MAPF_CTE_POLICY_MAX_CELLS, MAPF_MAX_AGENTS);
    return mapf::cte_weight_bytes(cells, num_agents);
}

int mapf_cte_policy_pack_weights(int32_t cells, int32_t num_agents, const float *w1, const float *b1, const float *w2,
                                 const float *b2, const float *wl, const float *bl, const float *wv, const float *bv,
                                 void *packed) {
    const int64_t nbytes = mapf_cte_policy_weights_nbytes(cells, num_agents);
    if (nbytes < 0) return (int)nbytes;
    if (!w1 || !b1 || !w2 || !b2 || !wl || !bl || !wv || !bv || !packed) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    const int s1 = mapf::cte_s1(cells), H = mapf::POL_H, S2 = mapf::POL_W2_STRIDE, A = 5 * num_agents;
    memset(packed, 0, (size_t)nbytes);
    __nv_bfloat16 *p1 = static_cast<__nv_bfloat16 *>(packed), *p2 = p1 + H * s1, *p3 = p2 + H * S2;
    float *pb = reinterpret_cast<float *>(p3 + 8 * mapf::cte_head_tiles(num_agents) * S2);
    for (int o = 0; o < H; ++o) {
        for (int i = 0; i < cells; ++i) p1[(size_t)o * s1 + i] = __float2bfloat16_rn(w1[(size_t)o * cells + i]);
        for (int i = 0; i < H; ++i) p2[o * S2 + i] = __float2bfloat16_rn(w2[o * H + i]);
        pb[o] = b1[o];
        pb[H + o] = b2[o];
    }
    for (int o = 0; o < A; ++o) {   // head rows: 5N logits, then the value
        for (int i = 0; i < H; ++i) p3[o * S2 + i] = __float2bfloat16_rn(wl[o * H + i]);
        pb[2 * H + o] = bl[o];
    }
    for (int i = 0; i < H; ++i) p3[A * S2 + i] = __float2bfloat16_rn(wv[i]);
    pb[2 * H + A] = bv[0];
    return MAPF_OK;
}

int mapf_cte_policy_act(const mapf_cte_policy_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (!cte_policy_shape_ok(a->cells, a->num_agents))
        return fail(MAPF_ERR_UNSUPPORTED, "cte policy: cells %d / num_agents %d outside 1..%d / 1..%d", a->cells,
                    a->num_agents, MAPF_CTE_POLICY_MAX_CELLS, MAPF_MAX_AGENTS);
    if (a->num_envs < 1 || !a->obs_grid || !a->action_mask || !a->weights)
        return fail(MAPF_ERR_INVALID_ARG, "cte policy: num_envs >= 1, obs_grid, action_mask and weights are required");
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "cte policy: reserved is %d, must be 0", a->reserved);
    if (a->greedy != 0 && a->greedy != 1) return fail(MAPF_ERR_INVALID_ARG, "cte policy: greedy %d is neither 0 nor 1", a->greedy);
    int ndev = 0, dev = 0, sms = 0, per_sm = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int threads = mapf::CTE_THREADS, warps = threads / 32;
    const size_t smem = (size_t)mapf::cte_weight_bytes(a->cells, a->num_agents) + (size_t)warps * mapf::CTE_WARP_BYTES;
    const auto kernel = a->greedy ? mapf::mapf_cte_policy_act_kernel<true> : mapf::mapf_cte_policy_act_kernel<false>;
    CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    if (per_sm < 1) return fail(MAPF_ERR_UNSUPPORTED, "cte policy: %zu bytes of shared memory do not fit one SM", smem);
    // resident blocks load the weights once and loop over the 32-env tiles
    const long long tiles = ((long long)a->num_envs + 31) / 32;
    long long blocks = (tiles + warps - 1) / warps;
    if (blocks > (long long)sms * per_sm) blocks = (long long)sms * per_sm;
    kernel<<<(unsigned)blocks, threads, smem, static_cast<cudaStream_t>(stream)>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int64_t mapf_cte_lstm_policy_weights_nbytes(int32_t cells, int32_t num_agents) {
    if (!cte_policy_shape_ok(cells, num_agents))
        return fail(MAPF_ERR_UNSUPPORTED, "cte lstm policy: cells %d / num_agents %d outside 1..%d / 1..%d", cells,
                    num_agents, MAPF_CTE_POLICY_MAX_CELLS, MAPF_MAX_AGENTS);
    return mapf::ctel_trunk_bytes(cells) + mapf::ctel_step_bytes(num_agents);
}

int mapf_cte_lstm_policy_pack_weights(int32_t cells, int32_t num_agents, const float *w1, const float *b1, const float *w2,
                                      const float *b2, const float *w_ih, const float *w_hh, const float *b_ih,
                                      const float *b_hh, const float *wl, const float *bl, const float *wv, const float *bv,
                                      void *packed) {
    const int64_t nbytes = mapf_cte_lstm_policy_weights_nbytes(cells, num_agents);
    if (nbytes < 0) return (int)nbytes;
    if (!w1 || !b1 || !w2 || !b2 || !w_ih || !w_hh || !b_ih || !b_hh || !wl || !bl || !wv || !bv || !packed)
        return fail(MAPF_ERR_INVALID_ARG, "null argument");
    const int s1 = mapf::cte_s1(cells), H = mapf::POL_H, S2 = mapf::POL_W2_STRIDE, A = 5 * num_agents;
    const int SG = mapf::ctel_sg(num_agents), KH = mapf::ctel_kh(num_agents), KI = H + A + 1;
    memset(packed, 0, (size_t)nbytes);
    // trunk part: w1 [64][S1] | w2 [64][72] | b1 b2
    __nv_bfloat16 *p1 = static_cast<__nv_bfloat16 *>(packed), *p2 = p1 + H * s1;
    float *pb = reinterpret_cast<float *>(p2 + H * S2);
    for (int o = 0; o < H; ++o) {
        for (int i = 0; i < cells; ++i) p1[(size_t)o * s1 + i] = __float2bfloat16_rn(w1[(size_t)o * cells + i]);
        for (int i = 0; i < H; ++i) p2[o * S2 + i] = __float2bfloat16_rn(w2[o * H + i]);
        pb[o] = b1[o];
        pb[H + o] = b2[o];
    }
    // step part: wg [256][SG] | w3 [8 NT][72] | bg[256] wr[256] b3[8 NT]
    const int NT = mapf::cte_head_tiles(num_agents);
    __nv_bfloat16 *pg = reinterpret_cast<__nv_bfloat16 *>(static_cast<unsigned char *>(packed) + mapf::ctel_trunk_bytes(cells));
    __nv_bfloat16 *p3 = pg + 4 * H * SG;
    float *pbg = reinterpret_cast<float *>(p3 + 8 * NT * S2), *pwr = pbg + 4 * H, *pb3 = pbg + 8 * H;
    for (int o = 0; o < 4 * H; ++o) {   // [W_ih y and one-hot columns | zero to 64 + KH | W_hh]; reward column in f32
        for (int i = 0; i < H + A; ++i) pg[(size_t)o * SG + i] = __float2bfloat16_rn(w_ih[(size_t)o * KI + i]);
        for (int i = 0; i < H; ++i) pg[(size_t)o * SG + H + KH + i] = __float2bfloat16_rn(w_hh[o * H + i]);
        pwr[o] = w_ih[(size_t)o * KI + H + A];
        pbg[o] = b_ih[o] + b_hh[o];
    }
    for (int o = 0; o < A; ++o) {   // head rows: 5N logits, then the value
        for (int i = 0; i < H; ++i) p3[o * S2 + i] = __float2bfloat16_rn(wl[o * H + i]);
        pb3[o] = bl[o];
    }
    for (int i = 0; i < H; ++i) p3[A * S2 + i] = __float2bfloat16_rn(wv[i]);
    pb3[A] = bv[0];
    return MAPF_OK;
}

int mapf_cte_lstm_policy_act(const mapf_cte_lstm_policy_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (!cte_policy_shape_ok(a->cells, a->num_agents))
        return fail(MAPF_ERR_UNSUPPORTED, "cte lstm policy: cells %d / num_agents %d outside 1..%d / 1..%d", a->cells,
                    a->num_agents, MAPF_CTE_POLICY_MAX_CELLS, MAPF_MAX_AGENTS);
    if (a->num_envs < 1 || !a->obs_grid || !a->action_mask || !a->weights || !a->trunk)
        return fail(MAPF_ERR_INVALID_ARG, "cte lstm policy: num_envs >= 1, obs_grid, action_mask, trunk and weights are required");
    if (!a->prev_action || !a->prev_reward || !a->h_in || !a->c_in)
        return fail(MAPF_ERR_INVALID_ARG, "cte lstm policy: prev_action, prev_reward, h_in and c_in are required");
    if (!a->h_out != !a->c_out)
        return fail(MAPF_ERR_INVALID_ARG, "cte lstm policy: h_out and c_out are given together (both NULL = state not advanced)");
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "cte lstm policy: reserved is %d, must be 0", a->reserved);
    if (a->greedy != 0 && a->greedy != 1)
        return fail(MAPF_ERR_INVALID_ARG, "cte lstm policy: greedy %d is neither 0 nor 1", a->greedy);
    int ndev = 0, dev = 0, sms = 0, per_sm[2] = {0, 0};
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    void (*const kernels[2])(const mapf_cte_lstm_policy_args) = {
        mapf::mapf_cte_lstm_trunk_kernel, a->greedy ? mapf::mapf_cte_lstm_step_kernel<true> : mapf::mapf_cte_lstm_step_kernel<false>};
    const int threads[2] = {mapf::CTE_THREADS, mapf::CTEL_THREADS};
    const size_t smem[2] = {(size_t)mapf::ctel_trunk_bytes(a->cells) + (size_t)(mapf::CTE_THREADS / 32) * mapf::CTE_WARP_BYTES,
                            (size_t)mapf::ctel_step_bytes(a->num_agents) + (size_t)(mapf::CTEL_THREADS / 32) * mapf::CTEL_WARP_BYTES};
    for (int k = 0; k < 2; ++k) {
        CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(kernels[k]), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem[k]));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[k], kernels[k], threads[k], smem[k]));
        if (per_sm[k] < 1) return fail(MAPF_ERR_UNSUPPORTED, "cte lstm policy: %zu bytes of shared memory do not fit one SM", smem[k]);
    }
    // resident blocks load their weights once and loop over the 32-env tiles
    const long long tiles = ((long long)a->num_envs + 31) / 32;
    for (int k = 0; k < 2; ++k) {
        const int warps = threads[k] / 32;
        long long blocks = (tiles + warps - 1) / warps;
        if (blocks > (long long)sms * per_sm[k]) blocks = (long long)sms * per_sm[k];
        kernels[k]<<<(unsigned)blocks, threads[k], smem[k], static_cast<cudaStream_t>(stream)>>>(*a);
        CUDA_TRY(cudaGetLastError());
    }
    return MAPF_OK;
}

int mapf_gae(const float *rewards, const float *values, const uint8_t *dones, const float *last_value, float *adv,
             float *ret, int32_t T, int64_t B, int32_t N, float gamma, float lam, void *stream) {
    if (!rewards || !values || !dones || !last_value || !adv || !ret || T < 1 || B < 1 || N < 1)
        return fail(MAPF_ERR_INVALID_ARG, "gae: null or empty argument");
    const long long BN = (long long)B * N;
    mapf::mapf_gae_kernel<<<(unsigned)((BN + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        rewards, values, dones, last_value, adv, ret, T, BN, N, gamma, lam);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_vtrace(const mapf_vtrace_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "vtrace: null argument");
    if (!a->rewards || !a->behaviour_logp || !a->dones || !a->bootstrap_value || !a->target_logp || !a->values || !a->vs ||
        !a->pg_advantages)
        return fail(MAPF_ERR_INVALID_ARG, "vtrace: null required pointer");
    if (a->T < 1 || a->M < 1 || a->num_agents < 1)
        return fail(MAPF_ERR_INVALID_ARG, "vtrace: T %d, M %lld and num_agents %d must be >= 1", a->T, (long long)a->M,
                    a->num_agents);
    if (a->num_columns < 1 || a->num_columns % a->num_agents != 0)
        return fail(MAPF_ERR_INVALID_ARG, "vtrace: num_columns %lld is not a positive multiple of num_agents %d",
                    (long long)a->num_columns, a->num_agents);
    if (!a->columns && a->M != a->num_columns)
        return fail(MAPF_ERR_INVALID_ARG, "vtrace: columns is NULL but M %lld != num_columns %lld", (long long)a->M,
                    (long long)a->num_columns);
    if (!(a->gamma >= 0.f && a->gamma <= 1.f)) return fail(MAPF_ERR_INVALID_ARG, "vtrace: gamma %g outside [0, 1]", a->gamma);
    if (!(std::isfinite(a->clip_rho) && a->clip_rho > 0.f) || !(std::isfinite(a->clip_pg_rho) && a->clip_pg_rho > 0.f))
        return fail(MAPF_ERR_INVALID_ARG, "vtrace: clip_rho %g and clip_pg_rho %g must be finite and positive", a->clip_rho,
                    a->clip_pg_rho);
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "vtrace: reserved is %d, must be 0", a->reserved);
    const long long blocks = (a->M + mapf::VTRACE_THREADS - 1) / mapf::VTRACE_THREADS;
    if (blocks > 0x7fffffffLL) return fail(MAPF_ERR_UNSUPPORTED, "vtrace: M %lld needs more than 2^31 - 1 blocks", (long long)a->M);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    mapf::mapf_vtrace_kernel<<<(unsigned)blocks, mapf::VTRACE_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

static int q_act_launch(const mapf_q_act_args *a, bool per_agent, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "q_act: null argument");
    if (!a->local_obs || !a->goal_delta || !a->action_mask || !a->weights || !a->actions)
        return fail(MAPF_ERR_INVALID_ARG, "q_act: local_obs, goal_delta, action_mask, weights and actions are required");
    if (a->num_envs < 1 || a->num_agents < 1)
        return fail(MAPF_ERR_INVALID_ARG, "q_act: num_envs %d and num_agents %d must be >= 1", a->num_envs, a->num_agents);
    if (!(a->epsilon >= 0.f && a->epsilon <= 1.f)) return fail(MAPF_ERR_INVALID_ARG, "q_act: epsilon %g outside [0, 1]", a->epsilon);
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "q_act: reserved is %d, must be 0", a->reserved);
    const int kc1 = policy_kc1(a->feature_dim);
    if (!kc1 || a->v2 < 1 || a->feature_dim != a->v2 + 2 + (a->blocking_prev ? 1 : 0))
        return fail(MAPF_ERR_UNSUPPORTED, "q_act: feature_dim %d does not match v2 %d (+2 goal delta, +1 pressure) or exceeds 64",
                    a->feature_dim, a->v2);
    if (per_agent && a->num_agents > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "q_act: num_agents %d exceeds %d", a->num_agents, MAPF_MAX_AGENTS);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    const int threads = 256, warps = threads / 32;
    const size_t smem = (size_t)mapf_policy_weights_nbytes(a->feature_dim) + (size_t)warps * mapf::pol_warp_bytes(kc1, a->v2);
    const long long tiles = per_agent ? ((long long)a->num_envs + 31) / 32 * a->num_agents
                                      : ((long long)a->num_envs * a->num_agents + 31) / 32;
    long long blocks = (tiles + warps - 1) / warps;
    if (blocks > 148 * 8) blocks = 148 * 8;
    void (*const kernels[2][2])(const mapf_q_act_args) = {
        {mapf::mapf_q_act_kernel<2, false>, mapf::mapf_q_act_kernel<4, false>},
        {mapf::mapf_q_act_kernel<2, true>, mapf::mapf_q_act_kernel<4, true>}};
    const auto kernel = kernels[per_agent][kc1 == 4];
    CUDA_TRY(cudaFuncSetAttribute(reinterpret_cast<const void *>(kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<(unsigned)blocks, threads, smem, static_cast<cudaStream_t>(stream)>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_q_act(const mapf_q_act_args *a, void *stream) { return q_act_launch(a, false, stream); }
int mapf_q_act_per_agent(const mapf_q_act_args *a, void *stream) { return q_act_launch(a, true, stream); }

// the leaf count L = N' K' B' of a ring shape, or an error (the shape checks every replay entry point shares)
static int64_t replay_leaves(int32_t B, int32_t N, int32_t K, const char *who) {
    if (B < 1 || N < 1 || K < 2)
        return fail(MAPF_ERR_INVALID_ARG, "%s: num_envs %d and num_agents %d must be >= 1 and capacity %d >= 2", who, B, N, K);
    const int bits = mapf::replay_log2_ceil(B) + mapf::replay_log2_ceil(K) + mapf::replay_log2_ceil(N);
    if (bits > 40) return fail(MAPF_ERR_UNSUPPORTED, "%s: 2^%d leaves", who, bits);
    return (int64_t)1 << bits;
}

int64_t mapf_replay_tree_leaves(int32_t B, int32_t N, int32_t K) { return replay_leaves(B, N, K, "replay"); }

static int replay_tree_check(const mapf_replay_tree &t, const char *who) {
    const int64_t L = replay_leaves(t.num_envs, t.num_agents, t.capacity, who);
    if (L < 0) return (int)L;
    if (!t.leaves || !t.sums || !t.mins || !t.max_priority) return fail(MAPF_ERR_INVALID_ARG, "%s: null tree array", who);
    return MAPF_OK;
}

static int replay_exponent_check(float x, const char *name, const char *who) {
    if (!(std::isfinite(x) && x >= 0.f)) return fail(MAPF_ERR_INVALID_ARG, "%s: %s %g must be finite and >= 0", who, name, x);
    return MAPF_OK;
}

static int device_check() {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    return MAPF_OK;
}

int mapf_replay_advance(const mapf_replay_advance_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "replay_advance: null argument");
    if (int rc = replay_tree_check(a->tree, "replay_advance")) return rc;
    if (int rc = replay_exponent_check(a->alpha, "alpha", "replay_advance")) return rc;
    const int K = a->tree.capacity;
    if (a->complete < 0 || a->complete >= K || a->clear < 0 || a->clear >= K || a->complete == a->clear)
        return fail(MAPF_ERR_INVALID_ARG, "replay_advance: complete %d and clear %d must be distinct slots of [0, %d)",
                    a->complete, a->clear, K);
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "replay_advance: reserved is %d, must be 0", a->reserved);
    if (int rc = device_check()) return rc;
    const long long Bp = 1ll << mapf::replay_log2_ceil(a->tree.num_envs);
    const int ch = (int)(Bp < mapf::REPLAY_CHUNK ? Bp : mapf::REPLAY_CHUNK);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    mapf::mapf_replay_advance_kernel<<<(unsigned)(2 * a->tree.num_agents * (Bp / ch)), ch, 0, st>>>(*a);
    CUDA_TRY(cudaGetLastError());
    mapf::mapf_replay_advance_top_kernel<<<1, mapf::REPLAY_THREADS, 0, st>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_replay_sample(const mapf_replay_sample_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "replay_sample: null argument");
    if (int rc = replay_tree_check(a->tree, "replay_sample")) return rc;
    if (!a->indices || !a->weights) return fail(MAPF_ERR_INVALID_ARG, "replay_sample: indices and weights are required");
    if (a->M < 1) return fail(MAPF_ERR_INVALID_ARG, "replay_sample: M %lld must be >= 1", (long long)a->M);
    if (int rc = replay_exponent_check(a->beta, "beta", "replay_sample")) return rc;
    if (a->per_agent != 0 && a->per_agent != 1)
        return fail(MAPF_ERR_INVALID_ARG, "replay_sample: per_agent %d is neither 0 nor 1", a->per_agent);
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "replay_sample: reserved is %d, must be 0", a->reserved);
    const long long blocks = (a->M + 255) / 256;
    if (blocks > 0x7fffffffLL) return fail(MAPF_ERR_UNSUPPORTED, "replay_sample: M %lld is too large", (long long)a->M);
    if (int rc = device_check()) return rc;
    mapf::mapf_replay_sample_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_replay_update(const mapf_replay_update_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "replay_update: null argument");
    if (int rc = replay_tree_check(a->tree, "replay_update")) return rc;
    if (!a->indices || !a->td_abs) return fail(MAPF_ERR_INVALID_ARG, "replay_update: indices and td_abs are required");
    if (a->M < 1) return fail(MAPF_ERR_INVALID_ARG, "replay_update: M %lld must be >= 1", (long long)a->M);
    if (int rc = replay_exponent_check(a->alpha, "alpha", "replay_update")) return rc;
    if (a->reserved != 0) return fail(MAPF_ERR_INVALID_ARG, "replay_update: reserved is %d, must be 0", a->reserved);
    if (int rc = device_check()) return rc;
    mapf::mapf_replay_update_kernel<<<1, mapf::REPLAY_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_eval_accumulate(const mapf_eval_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (a->num_envs < 1 || a->num_agents < 1 || !a->reward || !a->terminated || !a->truncated || !a->info || !a->active ||
        !a->episode_reward || !a->agent_reward || !a->timesteps || !a->success || !a->last_info || !a->active_count)
        return fail(MAPF_ERR_INVALID_ARG, "eval: null or empty argument");
    if (a->num_agents > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "eval: num_agents %d exceeds %d", a->num_agents, MAPF_MAX_AGENTS);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    int P = 1;   // lanes per env: N rounded up to a power of two
    while (P < a->num_agents) P <<= 1;
    const int envs_per_block = mapf::EVAL_THREADS / 32 * (32 / P);
    long long blocks = ((long long)a->num_envs + envs_per_block - 1) / envs_per_block;
    if (blocks > 148 * 8) blocks = 148 * 8;   // one resident wave; the count then costs one atomic per block
    mapf::mapf_eval_accumulate_kernel<<<(unsigned)blocks, mapf::EVAL_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*a, P);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int mapf_cte_eval_accumulate(const mapf_cte_eval_args *a, void *stream) {
    if (!a) return fail(MAPF_ERR_INVALID_ARG, "null argument");
    if (a->num_envs < 1 || a->num_agents < 1 || a->rows < 1 || a->cols < 1 || !a->positions || !a->reward ||
        !a->terminated || !a->truncated || !a->info || !a->active || !a->episode_reward || !a->timesteps || !a->success ||
        !a->last_info || !a->occupancy || !a->active_count)
        return fail(MAPF_ERR_INVALID_ARG, "cte eval: null or empty argument");
    if (a->num_agents > MAPF_MAX_AGENTS)
        return fail(MAPF_ERR_UNSUPPORTED, "cte eval: num_agents %d exceeds %d", a->num_agents, MAPF_MAX_AGENTS);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(MAPF_ERR_CUDA, "no CUDA device (libmapf_b200 has no CPU fallback)");
    // an int16 [B,N,2] (row, col) pair is, byte for byte on a little-endian device, the packed uint32 the heat-map
    // kernel decodes (prow: low half, pcol: high half); the heat-map reads `active` before the next launch clears it
    static_assert(sizeof(int16_t) * 2 == sizeof(uint32_t), "an agent's (row, col) pair is one packed position word");
    occupancy_launch(reinterpret_cast<const uint32_t *>(a->positions), a->active, a->num_envs, a->num_agents, a->rows,
                     a->cols, a->occupancy, stream);
    CUDA_TRY(cudaGetLastError());
    long long blocks = ((long long)a->num_envs + mapf::EVAL_THREADS - 1) / mapf::EVAL_THREADS;
    if (blocks > 148 * 8) blocks = 148 * 8;   // one resident wave, as mapf_eval_accumulate
    mapf::mapf_cte_eval_accumulate_kernel<<<(unsigned)blocks, mapf::EVAL_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(*a);
    CUDA_TRY(cudaGetLastError());
    return MAPF_OK;
}

int64_t mapf_launch_count(const mapf_handle *h) { return h ? h->launches : 0; }

int mapf_step_kernel_kind(const mapf_handle *h) { return h ? (h->use_env_kernel ? (h->pair_kernel ? 3 : 2) : 1) : 0; }

}  // extern "C"
