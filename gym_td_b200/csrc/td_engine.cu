// td_engine.cu -- C-ABI entry points (include/td_b200.h) over the kernels in td_kernels.cuh.
// Host logic only: buffer layout, validation, launches on the caller's stream, error reporting.
// There is no CPU fallback: every compute entry point needs a CUDA device.
#include "td_kernels.cuh"
#include "td_rollout.cuh"

#include <cuda.h>          // driver API types only: entry points are resolved at run time (no libcuda link dependency)

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

using namespace td;

struct HostCopy { void *dst; const void *src; size_t bytes; };     // one copy of td_step_host (either direction)

struct td_handle {
    int device = 0, kind = 0, L = 0, cells = 0, cells_pad = 0, n_envs = 0;
    int n_maps = 0, map_stride = 0, difficulty = 1;
    int record_bytes = 0, map_bytes = 0, smem_per_warp = 0, scratch_off = 0;
    int old_lists_off = 0, act_stage_off = 0;
    const float *obs_synced = nullptr;   // buffer that holds the current observation of every env (NULL: none known)
    int off_static = 0, off_towers = 0, off_enemies = 0, off_map6 = 0, rng_cache_words = 0;
    uint8_t *records = nullptr;
    uint8_t *maps = nullptr;
    uint32_t *mt = nullptr;
    EnvStats *stats = nullptr;
    td_stats *stats_dev = nullptr;
    bool opponent_seeded = false;
    long long steps = 0;
    // td_step_host: the whole host-buffer step (action copies, chunk kernels, output copies) is one CUDA graph,
    // cached per distinct set of buffers
    struct HostGraph { std::vector<unsigned char> key; cudaGraphExec_t exec; unsigned long long used; };
    std::vector<HostGraph> host_graphs;
    unsigned long long host_graph_clock = 0;
    cudaStream_t host_stream = nullptr;  // stands in for the legacy default stream, which cannot launch graphs
    int host_chunks = 0;                 // 0 = automatic
    int host_graph = 1;                  // 1 = graph launch (default), 0 = plain stream launches
    bool generic_kernels = false;        // td_set_option: never pick the opponent-specialised step kernels
    bool host_chain = false;             // td_step_host graph: chunk kernels chained, or independent branches (default)
    int host_first_chunk = -1;           // td_step_host: envs in the first chunk (chunks grow x3); 0 = equal chunks, -1 = automatic
    unsigned long long cfg_generation = 0;
    std::vector<unsigned char> host_key;   // td_step_host: lookup key of the call in progress
    std::vector<HostCopy> host_in, host_out;   // td_step_host: copy lists of the call in progress
    int host_zero_copy = -1;             // td_step_host inputs read by the kernel from host memory: -1 automatic (8-byte actions), 0 never, 1 always
    td_config cfg = {};
    DevConfig dev_cfg = {};              // derived tables of cfg; copied into the parameters of every launch (per handle)
    std::string err;
};

static std::string g_create_error;

static int fail(td_handle *h, int code, const std::string &msg)
{
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}

#define TD_CUDA(h, call)                                                                         \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail((h), TD_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));     \
    } while (0)

static int round16(int x) { return (x + 15) & ~15; }

extern "C" int td_abi_version(void) { return TD_ABI_VERSION; }

extern "C" int td_packed_stride(int env_kind) { return env_kind == TD_KIND_DEF ? 32 : (int)sizeof(td_step_packed); }

extern "C" const char *td_last_error(const td_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

// gym_TD/envs/TDParam.py:1-94, 105-111
extern "C" void td_default_config(td_config *c)
{
    static const double eLP[4][2] = {{820, 1700}, {2050, 3000}, {6000, 8000}, {8000, 12000}};
    static const double espd[4][2] = {{.25, .25}, {.13, .13}, {.1, .1}, {.1, .1}};
    static const double edef[4][2] = {{0, 0}, {200, 250}, {600, 800}, {80, 100}};
    static const double ecost[4][2] = {{8, 8}, {15, 15}, {40, 40}, {30, 30}};
    static const double tatk[4][2] = {{454, 540}, {651, 771}, {566, 691}, {358, 424}};
    static const int trge[4][2] = {{3, 3}, {2, 2}, {4, 4}, {3, 3}};
    static const int tspl[4][2] = {{0, 0}, {0, 0}, {1, 1}, {0, 0}};
    static const double tcost[4][2] = {{10, 10}, {17, 17}, {23, 23}, {12, 12}};
    static const double tintv[4][2] = {{2, 2}, {4, 4}, {7, 7}, {4.75, 4.75}};
    memset(c, 0, sizeof(*c));
    for (int t = 0; t < TD_NTYPES; ++t)
        for (int l = 0; l < TD_NLV; ++l) {
            c->enemy_LP[t][l] = eLP[t][l];
            c->enemy_speed[t][l] = espd[t][l];
            c->enemy_defense[t][l] = edef[t][l];
            c->enemy_cost[t][l] = ecost[t][l];
            c->tower_attack[t][l] = tatk[t][l];
            c->tower_range[t][l] = trge[t][l];
            c->tower_splash_range[t][l] = tspl[t][l];
            c->tower_cost[t][l] = tcost[t][l];
            c->tower_attack_interval[t][l] = tintv[t][l];
        }
    c->tower_destruct_return = .5;
    c->frozen_time = 2;
    c->frozen_ratio = .2;
    c->attacker_init_cost = 0;
    c->defender_init_cost = 10;
    c->base_LP = 5;
    c->max_cost = 100;
    c->reward_kill = 0.1;
    c->penalty_leak = 10.;
    c->reward_time = 0.001;
    c->attacker_cost_init_rate = .5;
    c->attacker_cost_final_rate = 1;
    c->defender_cost_rate = .2;
    c->tower_distance = 2;
    c->enemy_upgrade_at = 0.75;
    c->attacker_action_interval = 1;
    c->defender_action_interval = 1;
    c->max_episode_steps = 1200;
    c->max_tower_lv = 1;
}

static int validate_config(td_handle *h, const td_config *c)
{
    if (!c) return fail(h, TD_E_INVALID, "config is NULL");
    if (c->max_tower_lv != 1) return fail(h, TD_E_INVALID, "this build supports max_tower_lv == 1 only");
    if (c->tower_distance < 0 || c->tower_distance > 8) return fail(h, TD_E_INVALID, "tower_distance out of range [0, 8]");
    if (c->max_episode_steps < 1) return fail(h, TD_E_INVALID, "max_episode_steps < 1");
    if (c->base_LP > 0x7fff) return fail(h, TD_E_INVALID, "base_LP too large");
    if (c->attacker_action_interval < 0 || c->attacker_action_interval > 0x7fff ||
        c->defender_action_interval < 0 || c->defender_action_interval > 0x7fff)
        return fail(h, TD_E_INVALID, "action interval out of range");
    if (c->frozen_time < 0 || c->frozen_time > 255) return fail(h, TD_E_INVALID, "frozen_time out of range [0, 255]");
    for (int t = 0; t < TD_NTYPES; ++t)
        for (int l = 0; l < TD_NLV; ++l)
            if (c->tower_range[t][l] < 0 || c->tower_splash_range[t][l] < 0 || !(c->enemy_LP[t][l] > 0))
                return fail(h, TD_E_INVALID, "negative range or non-positive enemy LP in config tables");
    // observation planes 11-12 divide by max_cost, 41-44 by enemy_cost[t][0]: the reference divides Python numbers
    // there (TDBoard.py:118,123-125,142) and raises ZeroDivisionError, so it cannot run such a config (DESIGN.md 5)
    if (!(c->max_cost > 0)) return fail(h, TD_E_INVALID, "max_cost must be > 0 (and not NaN)");
    for (int t = 0; t < TD_NTYPES; ++t)
        if (c->enemy_cost[t][0] == 0 || c->enemy_cost[t][0] != c->enemy_cost[t][0])
            return fail(h, TD_E_INVALID, "enemy_cost[t][0] must not be 0 or NaN");
    return TD_OK;
}

// progress = steps / max_steps is monotone in steps (correctly rounded division of exact integers), so the first
// step count whose f64 quotient reaches the threshold decides the enemy level exactly like
// `self.progress >= config.enemy_upgrade_at` does, for every step count, also past the end of the episode.
// ceil(at * max) is within a few counts of it; the two walks land on the first count that passes the test itself.
extern "C" int td_upgrade_step(int max_episode_steps, double enemy_upgrade_at)
{
    const int kNever = 0x7fffffff;
    if (max_episode_steps < 1) return kNever;
    const double m = (double)max_episode_steps, at = enemy_upgrade_at;
    if (!(at > 0.0)) return at <= 0.0 ? 0 : kNever;            // 0 / max >= at; NaN never compares true
    auto reaches = [m, at](long long s) { volatile double q = (double)s / m; return q >= at; };
    const double guess = std::ceil(at * m);
    long long s = guess < (double)kNever ? (long long)guess : (long long)kNever;
    while (s > 0 && reaches(s - 1)) --s;
    while (s < kNever && !reaches(s)) ++s;
    return (int)s;
}

// td_config -> the derived tables the kernels read.  The result lives in the handle and rides in the kernel
// parameters of every launch, so handles with different configs coexist on one device.
static int derive_config(td_handle *h, const td_config *c)
{
    DevConfig &d = h->dev_cfg;
    memset(&d, 0, sizeof(d));
    for (int t = 0; t < TD_NTYPES; ++t)
        for (int l = 0; l < TD_NLV; ++l) {
            d.enemy_LP[t][l] = c->enemy_LP[t][l];
            d.enemy_speed[t][l] = c->enemy_speed[t][l];
            d.enemy_defense[t][l] = c->enemy_defense[t][l];
            d.enemy_cost[t][l] = c->enemy_cost[t][l];
            d.tower_attack[t][l] = c->tower_attack[t][l];
            d.tower_cost[t][l] = c->tower_cost[t][l];
            d.tower_range[t][l] = c->tower_range[t][l];
            d.tower_splash[t][l] = c->tower_splash_range[t][l];
        }
    for (int t = 0; t < TD_NTYPES; ++t) {
        // TDElements.py:152-170 passes (.., tower_cost, tower_attack_interval) into lvup(.., intv, cost):
        // after LvUp the interval is tower_cost[t][1] and Tower.cost grows by tower_attack_interval[t][1].
        d.tower_intv[t][0] = c->tower_attack_interval[t][0];
        d.tower_intv[t][1] = c->tower_cost[t][1];
        d.tower_refund[t][0] = c->tower_cost[t][0];
        volatile double grown = c->tower_cost[t][0] + c->tower_attack_interval[t][1];
        d.tower_refund[t][1] = grown;
    }
    d.destruct_return = c->tower_destruct_return;
    d.frozen_ratio = c->frozen_ratio;
    d.atk_init_cost = c->attacker_init_cost;
    d.def_init_cost = c->defender_init_cost;
    d.max_cost = c->max_cost;
    d.reward_kill = c->reward_kill;
    d.penalty_leak = c->penalty_leak;
    d.reward_time = c->reward_time;
    d.rate_init = c->attacker_cost_init_rate;
    d.rate_final = c->attacker_cost_final_rate;
    d.def_rate = c->defender_cost_rate;
    d.upgrade_at = c->enemy_upgrade_at;
    d.upgrade_step = td_upgrade_step(c->max_episode_steps, c->enemy_upgrade_at);
    for (int lv = 0; lv < TD_NLV; ++lv) {
        d.min_enemy_cost[lv] = d.enemy_cost[0][lv];
        for (int t = 1; t < TD_NTYPES; ++t) d.min_enemy_cost[lv] = std::min(d.min_enemy_cost[lv], d.enemy_cost[t][lv]);
    }
    d.frozen_time = c->frozen_time;
    d.base_LP = c->base_LP < 0 ? -1 : c->base_LP;
    d.tower_distance = c->tower_distance;
    d.atk_interval = c->attacker_action_interval;
    d.def_interval = c->defender_action_interval;
    d.max_steps = c->max_episode_steps;
    h->cfg = *c;
    h->cfg_generation += 1;      // cached host-step graphs carry the old tables in their kernel parameters
    return TD_OK;
}

static void fill_params(const td_handle *h, StepParams &p)
{
    memset(&p, 0, sizeof(p));
    p.records = h->records;
    p.maps = h->maps;
    p.mt = h->mt;
    p.stats = h->stats;
    p.n_envs = h->n_envs;
    p.n_maps = h->n_maps;
    p.map_stride = h->map_stride;
    p.L = h->L;
    p.cells = h->cells;
    p.cells_pad = h->cells_pad;
    p.record_bytes = h->record_bytes;
    p.map_bytes = h->map_bytes;
    p.smem_per_warp = h->smem_per_warp;
    p.scratch_off = h->scratch_off;
    p.off_static = h->off_static;
    p.off_towers = h->off_towers;
    p.off_enemies = h->off_enemies;
    p.rng_cache_words = h->rng_cache_words;
    p.difficulty = h->difficulty;
    p.opponent_seeded = h->opponent_seeded ? 1 : 0;
    p.old_lists_off = h->old_lists_off;
    p.act_stage_off = h->act_stage_off;
    p.cfg = h->dev_cfg;
}

static int grid_of(const td_handle *h) { return (h->n_envs + kWarpsPerCta - 1) / kWarpsPerCta; }
static size_t smem_of(const td_handle *h) { return (size_t)kWarpsPerCta * h->smem_per_warp; }

// Dynamic shared memory of one step CTA.  Boards whose observation is >= 128 KB ask for at least 75 KB so that
// three CTAs (12 warps = 12 open observation streams) share an SM instead of six: HBM write efficiency falls
// with the number of long streams written side by side (tools/storebench_sized.cu, test F: 162 KB regions at
// 4 / 12 / 24 warps per SM -> 7.0 / 6.3 / 5.75 TB/s), and the rules of a large board are a small part of the step.
static bool large_observation(const td_handle *h) { return (size_t)TD_NCHANNELS * h->cells * sizeof(float) >= 128 * 1024; }

static size_t step_smem_bytes(const td_handle *h)
{
    return large_observation(h) ? std::max(smem_of(h), (size_t)75 * 1024) : smem_of(h);
}

// Warps per step CTA.  The full-write kernels are insensitive to it (1 / 2 / 4 warps: def-small 0.2131 / 0.2129 /
// 0.2131 ms, 8 warps 0.2180); the in-place observation update is latency-bound and gains from single-warp CTAs,
// whose slots are re-filled as soon as ONE env is done (def-small 0.1765 -> 0.1580 ms, atk-small 0.2119 -> 0.1973).
static int step_warps_per_cta(const td_handle *h, bool incremental)
{
    // (10x10 boards only: at 20x20 it changes nothing, 0.1921 vs 0.1916 ms)
    return incremental && h->L == 10 ? 1 : kWarpsPerCta;
}

// The scripted opponent of level 1 draws from the device generator and no host-resolved opponent input is set:
// the case the opponent-specialised kernels (OPP = 1) are compiled for.
static bool scripted_lv1_on_device(const td_handle *h, const td_step_io *io)
{
    return !h->generic_kernels && h->kind != TD_KIND_2P && h->difficulty == 1 && h->opponent_seeded && h->mt != nullptr &&
           io->opponent_dev == nullptr && io->opponent_cluster_dev == nullptr &&
           (h->kind != TD_KIND_ATK || io->def_action_dev == nullptr);
}

using StepKernel = void (*)(StepParams);

// float32 observation kernels of one board specialisation.  `scripted`: the default scripted opponent (level 1 on
// the device generator) known at compile time, for the defender and the attacker env.
template <int CELLS, bool INC> static StepKernel f32_step_kernel(int kind, bool multi, bool scripted)
{
    switch (kind) {
    case TD_KIND_DEF:
        if (scripted)
            return multi ? td_step_kernel<TD_KIND_DEF, true, CELLS, INC, float, 1>
                         : td_step_kernel<TD_KIND_DEF, false, CELLS, INC, float, 1>;
        return multi ? td_step_kernel<TD_KIND_DEF, true, CELLS, INC> : td_step_kernel<TD_KIND_DEF, false, CELLS, INC>;
    case TD_KIND_ATK:
        return scripted ? td_step_kernel<TD_KIND_ATK, false, CELLS, INC, float, 1>
                        : td_step_kernel<TD_KIND_ATK, false, CELLS, INC>;
    default:
        return multi ? td_step_kernel<TD_KIND_2P, true, CELLS, INC> : td_step_kernel<TD_KIND_2P, false, CELLS, INC>;
    }
}

// reduced-precision observation kernels (td_step_io.obs_format): Discrete actions, full writes, opponent read at run time
template <int CELLS, class OT> static StepKernel reduced_step_kernel(int kind)
{
    switch (kind) {
    case TD_KIND_DEF: return td_step_kernel<TD_KIND_DEF, false, CELLS, false, OT>;
    case TD_KIND_ATK: return td_step_kernel<TD_KIND_ATK, false, CELLS, false, OT>;
    default: return td_step_kernel<TD_KIND_2P, false, CELLS, false, OT>;
    }
}

// The step kernel for a board size L, an env kind, Discrete / multi-action, the in-place observation update, an
// observation format (TD_OBS_F32 when no observation is written) and the opponent specialisation; NULL: none is
// compiled.  Boards other than 10 / 20 / 30 take the run-time-size kernels, which always write the observation in full.
static StepKernel step_kernel(int L, int kind, bool multi, bool incremental, int obs_format, bool scripted)
{
    if (obs_format != TD_OBS_F32) {
        if (multi) return nullptr;
        const bool bf16 = obs_format == TD_OBS_BF16;
        switch (L) {
        case 10: return bf16 ? reduced_step_kernel<100, __nv_bfloat16>(kind) : reduced_step_kernel<100, uint8_t>(kind);
        case 20: return bf16 ? reduced_step_kernel<400, __nv_bfloat16>(kind) : reduced_step_kernel<400, uint8_t>(kind);
        case 30: return bf16 ? reduced_step_kernel<900, __nv_bfloat16>(kind) : reduced_step_kernel<900, uint8_t>(kind);
        default: return nullptr;
        }
    }
    switch (L) {
    case 10:
        return incremental ? f32_step_kernel<100, true>(kind, multi, scripted) : f32_step_kernel<100, false>(kind, multi, scripted);
    case 20:
        return incremental ? f32_step_kernel<400, true>(kind, multi, scripted) : f32_step_kernel<400, false>(kind, multi, scripted);
    case 30:
        return incremental ? f32_step_kernel<900, true>(kind, multi, scripted) : f32_step_kernel<900, false>(kind, multi, scripted);
    default: return f32_step_kernel<0, false>(kind, multi, scripted);
    }
}

// The observation writer (td_observe_kernel) for a board size and format; NULL: none is compiled (reduced precision:
// boards 10 / 20 / 30 only).
template <class OT> static const void *specialised_observe_kernel(int L)
{
    switch (L) {
    case 10: return (const void *)td_observe_kernel<100, OT>;
    case 20: return (const void *)td_observe_kernel<400, OT>;
    case 30: return (const void *)td_observe_kernel<900, OT>;
    default: return nullptr;
    }
}

static const void *observe_kernel(int L, int obs_format)
{
    switch (obs_format) {
    case TD_OBS_F32: {
        const void *k = specialised_observe_kernel<float>(L);
        return k ? k : (const void *)td_observe_kernel<0>;
    }
    case TD_OBS_BF16: return specialised_observe_kernel<__nv_bfloat16>(L);
    case TD_OBS_U8: return specialised_observe_kernel<uint8_t>(L);
    default: return nullptr;
    }
}

// The action-mask kernel for a board size: specialised on 10 / 20 / 30, the run-time-size kernel otherwise.
static const void *action_mask_kernel(int L)
{
    switch (L) {
    case 10: return (const void *)td_action_mask_kernel<100>;
    case 20: return (const void *)td_action_mask_kernel<400>;
    case 30: return (const void *)td_action_mask_kernel<900>;
    default: return (const void *)td_action_mask_kernel<0>;
    }
}

static size_t mask_smem_of(const td_handle *h) { return (size_t)kWarpsPerCta * mask_smem_per_warp(h->cells_pad); }

template <typename K> static cudaError_t allow_smem(K kernel, size_t bytes)
{
    if (bytes <= 48 * 1024) return cudaSuccess;
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

extern "C" int td_create(const td_config *cfg, int env_kind, int map_size, int n_envs, int device, td_handle **out)
{
    if (!out) return fail(nullptr, TD_E_INVALID, "out is NULL");
    *out = nullptr;
    if (env_kind < TD_KIND_DEF || env_kind > TD_KIND_2P) return fail(nullptr, TD_E_INVALID, "unknown env kind");
    if (map_size < 4 || map_size > TD_MAX_L) return fail(nullptr, TD_E_INVALID, "map_size must be in [4, 64]");
    if (n_envs < 1) return fail(nullptr, TD_E_INVALID, "n_envs < 1");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0)
        return fail(nullptr, TD_E_CUDA, std::string("no CUDA device available (") +
                    (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") + "); there is no CPU fallback");
    if (device < 0 || device >= count) return fail(nullptr, TD_E_INVALID, "device index out of range");
    td_handle *h = new (std::nothrow) td_handle();
    if (!h) return fail(nullptr, TD_E_ALLOC, "out of host memory");
    h->device = device; h->kind = env_kind; h->L = map_size; h->cells = map_size * map_size;
    h->cells_pad = round16(h->cells); h->n_envs = n_envs; h->map_stride = n_envs;
    h->map_bytes = kMapHdrBytes + 2 * h->cells_pad;
    h->rng_cache_words = env_kind == TD_KIND_ATK ? kRngCacheAtk : kRngCacheDef;
    h->off_map6 = kOffRngCache + 4 * h->rng_cache_words;
    h->off_static = h->off_map6 + h->cells_pad;
    h->off_towers = h->off_static + h->map_bytes;
    h->off_enemies = h->off_towers + TD_CAP_TOWERS * kTowerBytes;
    h->record_bytes = h->off_enemies + TD_CAP_ENEMIES * kEnemyBytes;
    h->scratch_off = h->record_bytes;
    int scratch = std::max(1024, std::max(h->cells_pad, round16(2 * std::min(h->cells, 6 * map_size)) + 256));   // + shuffle word buffer
    // slice = [record | scratch | pre-step tower / enemy cells (incremental observation) | twist staging area]
    h->old_lists_off = h->record_bytes + scratch;
    scratch += kOldListBytes;
    h->act_stage_off = h->record_bytes + scratch;               // the attacker's action / RealAction (ATK, 2P)
    if (env_kind != TD_KIND_DEF) scratch += TD_ROADS * TD_CLUSTER * 8;
    if (env_kind != TD_KIND_2P) scratch += kTwistStageBytes;
    h->smem_per_warp = h->record_bytes + scratch;
    td_config def;
    if (!cfg) { td_default_config(&def); cfg = &def; }
    int rc = validate_config(h, cfg);
    auto bail = [&](int code) { g_create_error = h->err; td_destroy(h); return code; };
    if (rc != TD_OK) return bail(rc);
    if ((e = cudaSetDevice(device)) != cudaSuccess) { h->err = cudaGetErrorString(e); return bail(TD_E_CUDA); }
    const size_t smem = smem_of(h), step_smem = step_smem_bytes(h);
    if (step_smem > 227 * 1024) { h->err = "map too large for shared memory"; return bail(TD_E_INVALID); }
    // every kernel the handle can launch: the reset, and the observe and step kernels step_kernel / observe_kernel
    // pick for its board size and env kind
    auto allow = [&](auto kernel, size_t bytes) { if (kernel && e == cudaSuccess) e = allow_smem(kernel, bytes); };
    allow(td_reset_kernel, smem);
    allow(action_mask_kernel(h->L), mask_smem_of(h));
    for (int fmt : {TD_OBS_F32, TD_OBS_BF16, TD_OBS_U8}) {
        allow(observe_kernel(h->L, fmt), smem);
        for (bool multi : {false, true})
            for (bool incremental : {false, true})
                for (bool scripted : {false, true}) allow(step_kernel(h->L, env_kind, multi, incremental, fmt, scripted), step_smem);
    }
    if (e != cudaSuccess) {
        h->err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e);
        return bail(TD_E_CUDA);
    }
    size_t rec_total = (size_t)n_envs * h->record_bytes;
    // (the records gain nothing from a compressible allocation: def-small 0.1899 vs 0.1900 ms, 2p-large 0.3584 vs 0.3582)
    if ((e = cudaMalloc(&h->records, rec_total)) != cudaSuccess ||
        (e = cudaMemset(h->records, 0, rec_total)) != cudaSuccess ||
        (e = cudaMalloc(&h->stats, (size_t)n_envs * sizeof(EnvStats))) != cudaSuccess ||
        (e = cudaMemset(h->stats, 0, (size_t)n_envs * sizeof(EnvStats))) != cudaSuccess ||
        (e = cudaMalloc(&h->stats_dev, sizeof(td_stats))) != cudaSuccess) {
        h->err = std::string("device allocation failed: ") + cudaGetErrorString(e);
        return bail(TD_E_ALLOC);
    }
    rc = derive_config(h, cfg);
    if (rc != TD_OK) return bail(rc);
    *out = h;
    return TD_OK;
}

extern "C" int td_destroy(td_handle *h)
{
    if (!h) return TD_OK;
    if (h->records) cudaFree(h->records);
    if (h->maps) cudaFree(h->maps);
    if (h->mt) cudaFree(h->mt);
    if (h->stats) cudaFree(h->stats);
    if (h->stats_dev) cudaFree(h->stats_dev);
    for (auto &g : h->host_graphs) cudaGraphExecDestroy(g.exec);
    if (h->host_stream) cudaStreamDestroy(h->host_stream);
    delete h;
    return TD_OK;
}

extern "C" int td_set_config(td_handle *h, const td_config *cfg)
{
    if (!h) return TD_E_INVALID;
    int rc = validate_config(h, cfg);
    if (rc != TD_OK) return rc;
    return derive_config(h, cfg);       // takes effect with the next launch; kernels in flight keep their copy
}

extern "C" int td_get_layout(const td_handle *h, td_layout *out)
{
    if (!h || !out) return TD_E_INVALID;
    out->record_bytes = h->record_bytes;
    out->off_header = 0;
    out->off_towers = h->off_towers;
    out->off_enemies = h->off_enemies;
    out->off_map6 = h->off_map6;
    out->tower_stride = kTowerBytes;
    out->enemy_stride = kEnemyBytes;
    out->cap_towers = TD_CAP_TOWERS;
    out->cap_enemies = TD_CAP_ENEMIES;
    out->map_record_bytes = h->map_bytes;
    out->mt_words = kMtWords;
    out->pad_ = 0;
    return TD_OK;
}

extern "C" int td_upload_maps(td_handle *h, const td_map *maps, int n_maps)
{
    if (!h) return TD_E_INVALID;
    if (!maps || n_maps < 1) return fail(h, TD_E_INVALID, "td_upload_maps: no maps");
    std::vector<uint8_t> pool((size_t)n_maps * h->map_bytes, 0);
    for (int i = 0; i < n_maps; ++i) {
        const td_map &m = maps[i];
        if (m.map_size != h->L) return fail(h, TD_E_INVALID, "td_upload_maps: map_size differs from the handle's");
        if (m.num_roads < 1 || m.num_roads > TD_ROADS) return fail(h, TD_E_INVALID, "td_upload_maps: num_roads out of range");
        if (m.max_dist < 0 || m.max_dist > 254) return fail(h, TD_E_INVALID, "td_upload_maps: road too long");
        uint8_t *rec = pool.data() + (size_t)i * h->map_bytes;
        MapHdr hd;
        memset(&hd, 0, sizeof(hd));
        for (int r = 0; r < TD_ROADS; ++r) {
            int s = r < m.num_roads ? m.start[r] : 0;
            if (s < 0 || s >= h->cells) return fail(h, TD_E_INVALID, "td_upload_maps: start cell out of range");
            hd.start[r] = (uint16_t)s;
        }
        if (m.end < 0 || m.end >= h->cells) return fail(h, TD_E_INVALID, "td_upload_maps: end cell out of range");
        hd.end = (uint16_t)m.end;
        hd.num_roads = (uint8_t)m.num_roads;
        hd.maxd_p1 = (uint8_t)(m.max_dist + 1);
        memcpy(rec, &hd, sizeof(hd));
        memcpy(rec + kMapHdrBytes, m.cells, (size_t)h->cells);
        memcpy(rec + kMapHdrBytes + h->cells_pad, m.dist, (size_t)h->cells);
        // every road cell must lead somewhere inside the board (guards the on-device walk)
        for (int c = 0; c < h->cells; ++c) {
            if (!(m.cells[c] & 1) || c == m.end) continue;
            int d = (m.cells[c] >> 4) & 3, r = c / h->L, col = c % h->L;
            int nr = r + (d == 2) - (d == 3), nc = col + (d == 0) - (d == 1);
            if (nr < 0 || nr >= h->L || nc < 0 || nc >= h->L || !(m.cells[nr * h->L + nc] & 1))
                return fail(h, TD_E_INVALID, "td_upload_maps: a road cell points off the road");
        }
    }
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaDeviceSynchronize());
    if (h->maps) { cudaFree(h->maps); h->maps = nullptr; }
    TD_CUDA(h, cudaMalloc(&h->maps, pool.size()));
    TD_CUDA(h, cudaMemcpy(h->maps, pool.data(), pool.size(), cudaMemcpyHostToDevice));
    h->n_maps = n_maps;
    return TD_OK;
}

extern "C" int td_set_map_stride(td_handle *h, int stride)
{
    if (!h) return TD_E_INVALID;
    if (stride < 0) return fail(h, TD_E_INVALID, "stride < 0");
    h->map_stride = stride;
    return TD_OK;
}

extern "C" int td_set_difficulty(td_handle *h, int difficulty)
{
    if (!h) return TD_E_INVALID;
    const int top = h->kind == TD_KIND_ATK ? 2 : 1;      // random_enemy_lv0/1, random_tower_lv0/1/2 (TDGymBasic.py:81-292)
    if (difficulty < 0 || difficulty > top) return fail(h, TD_E_INVALID, "no scripted opponent of that level for this env kind");
    h->difficulty = difficulty;
    return TD_OK;
}

extern "C" int td_reset(td_handle *h, const uint8_t *mask_dev, const int32_t *map_ids_dev, float *obs_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (h->n_maps < 1) return fail(h, TD_E_STATE, "td_reset: upload maps first");
    TD_CUDA(h, cudaSetDevice(h->device));
    StepParams p;
    fill_params(h, p);
    td_reset_kernel<<<grid_of(h), kWarpsPerCta * 32, smem_of(h), (cudaStream_t)stream>>>(p, mask_dev, map_ids_dev, obs_dev);
    TD_CUDA(h, cudaGetLastError());
    if (!mask_dev) h->obs_synced = obs_dev;                      // every env restarted: obs_dev (if any) is current
    else if (obs_dev != h->obs_synced) h->obs_synced = nullptr;  // some envs restarted without updating the known buffer
    return TD_OK;
}

__global__ void td_rng_pos_kernel(uint8_t *records, int record_bytes, int first, int n, const int32_t *pos, int32_t *pos_out)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    td_env_header *h = reinterpret_cast<td_env_header *>(records + (size_t)(first + i) * record_bytes);
    if (pos) { h->rng_pos = pos[i]; h->pad0 = 0; h->pad1 = 0; }   // pad0 / pad1 = cached generator words valid / consumed: none
    if (pos_out) pos_out[i] = h->rng_pos;
}

extern "C" int td_seed_opponent(td_handle *h, const uint32_t *states, int first_env, int n)
{
    if (!h) return TD_E_INVALID;
    if (!states || first_env < 0 || n < 1 || first_env + n > h->n_envs) return fail(h, TD_E_INVALID, "td_seed_opponent: bad range");
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaDeviceSynchronize());
    if (!h->mt) {
        TD_CUDA(h, cudaMalloc(&h->mt, (size_t)h->n_envs * kMtWords * sizeof(uint32_t)));
        TD_CUDA(h, cudaMemset(h->mt, 0, (size_t)h->n_envs * kMtWords * sizeof(uint32_t)));
    }
    std::vector<uint32_t> words((size_t)n * kMtWords);
    std::vector<int32_t> pos((size_t)n);
    for (int i = 0; i < n; ++i) {
        memcpy(&words[(size_t)i * kMtWords], states + (size_t)i * (kMtWords + 1), kMtWords * sizeof(uint32_t));
        uint32_t p = states[(size_t)i * (kMtWords + 1) + kMtWords];
        if (p > (uint32_t)kMtWords) return fail(h, TD_E_INVALID, "td_seed_opponent: position > 624");
        pos[(size_t)i] = (int32_t)p;
    }
    int32_t *pos_dev = nullptr;
    TD_CUDA(h, cudaMalloc(&pos_dev, (size_t)n * sizeof(int32_t)));
    cudaError_t e = cudaMemcpy(pos_dev, pos.data(), (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = cudaMemcpy(h->mt + (size_t)first_env * kMtWords, words.data(), words.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        td_rng_pos_kernel<<<(n + 255) / 256, 256>>>(h->records, h->record_bytes, first_env, n, pos_dev, nullptr);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaFree(pos_dev);
    if (e != cudaSuccess) return fail(h, TD_E_CUDA, std::string("td_seed_opponent: ") + cudaGetErrorString(e));
    h->opponent_seeded = true;
    return TD_OK;
}

// CPython random.seed(int) for 0 <= seed < 2^32: init_by_array([seed]) (Modules/_randommodule.c)
static void python_seed_state(uint32_t seed, uint32_t *st625)
{
    uint32_t *mt = st625;
    mt[0] = 19650218u;
    for (int i = 1; i < kMtWords; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    int i = 1;
    for (int k = kMtWords; k; --k) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1664525u)) + seed;   // key = [seed], j stays 0
        if (++i >= kMtWords) { mt[0] = mt[kMtWords - 1]; i = 1; }
    }
    for (int k = kMtWords - 1; k; --k) {
        mt[i] = (mt[i] ^ ((mt[i - 1] ^ (mt[i - 1] >> 30)) * 1566083941u)) - (uint32_t)i;
        if (++i >= kMtWords) { mt[0] = mt[kMtWords - 1]; i = 1; }
    }
    mt[0] = 0x80000000u;
    st625[kMtWords] = (uint32_t)kMtWords;
}

extern "C" int td_seed_opponent_python(td_handle *h, const uint32_t *seeds, int first_env, int n)
{
    if (!h) return TD_E_INVALID;
    if (!seeds || n < 1) return fail(h, TD_E_INVALID, "td_seed_opponent_python: bad range");
    std::vector<uint32_t> states((size_t)n * (kMtWords + 1));
    for (int i = 0; i < n; ++i) python_seed_state(seeds[i], &states[(size_t)i * (kMtWords + 1)]);
    return td_seed_opponent(h, states.data(), first_env, n);
}

extern "C" int td_get_opponent(td_handle *h, int first_env, int n, uint32_t *states)
{
    if (!h) return TD_E_INVALID;
    if (!states || first_env < 0 || n < 1 || first_env + n > h->n_envs) return fail(h, TD_E_INVALID, "td_get_opponent: bad range");
    if (!h->mt) return fail(h, TD_E_STATE, "td_get_opponent: generators were never seeded");
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaDeviceSynchronize());
    std::vector<uint32_t> words((size_t)n * kMtWords);
    std::vector<int32_t> pos((size_t)n);
    int32_t *pos_dev = nullptr;
    TD_CUDA(h, cudaMalloc(&pos_dev, (size_t)n * sizeof(int32_t)));
    td_rng_pos_kernel<<<(n + 255) / 256, 256>>>(h->records, h->record_bytes, first_env, n, nullptr, pos_dev);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(pos.data(), pos_dev, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess)
        e = cudaMemcpy(words.data(), h->mt + (size_t)first_env * kMtWords, words.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaFree(pos_dev);
    if (e != cudaSuccess) return fail(h, TD_E_CUDA, std::string("td_get_opponent: ") + cudaGetErrorString(e));
    for (int i = 0; i < n; ++i) {
        memcpy(states + (size_t)i * (kMtWords + 1), &words[(size_t)i * kMtWords], kMtWords * sizeof(uint32_t));
        states[(size_t)i * (kMtWords + 1) + kMtWords] = (uint32_t)pos[(size_t)i];
    }
    return TD_OK;
}

// A bf16 / u8 observation buffer: a known format, a board the reduced-precision kernels are compiled for, and an
// address aligned for their stores.
static int check_reduced_obs(td_handle *h, const char *who, int obs_format, const void *obs_dev)
{
    const std::string w(who);
    if (obs_format != TD_OBS_BF16 && obs_format != TD_OBS_U8) return fail(h, TD_E_INVALID, w + ": unknown obs_format");
    if (!(h->L == 10 || h->L == 20 || h->L == 30))
        return fail(h, TD_E_INVALID, w + ": reduced-precision observations need a 10 / 20 / 30 board");
    if (reinterpret_cast<uintptr_t>(obs_dev) & (obs_format == TD_OBS_BF16 ? 7 : 3))
        return fail(h, TD_E_INVALID, w + ": obs_dev is not aligned for this obs_format");
    return TD_OK;
}

static int check_io(td_handle *h, const td_step_io *io)
{
    if (!io) return fail(h, TD_E_INVALID, "td_step: io is NULL");
    if (h->n_maps < 1) return fail(h, TD_E_STATE, "td_step: upload maps and reset first");
    if (h->kind != TD_KIND_ATK && !io->def_action_dev) return fail(h, TD_E_INVALID, "td_step: def_action_dev is required");
    if (h->kind != TD_KIND_DEF && !io->atk_action_dev) return fail(h, TD_E_INVALID, "td_step: atk_action_dev is required");
    if (h->kind == TD_KIND_ATK && io->multi_action) return fail(h, TD_E_INVALID, "td_step: multi_action does not apply to the attacker env");
    if (h->kind != TD_KIND_DEF && (io->opponent_dev || io->opponent_cluster_dev))
        return fail(h, TD_E_INVALID, "td_step: opponent_dev / opponent_cluster_dev belong to the defender env");
    if (io->opponent_dev && io->opponent_cluster_dev)
        return fail(h, TD_E_INVALID, "td_step: give opponent_dev or opponent_cluster_dev, not both");
    if (io->obs_format != TD_OBS_F32 && io->obs_dev) {
        if (io->multi_action) return fail(h, TD_E_INVALID, "td_step: reduced-precision observations need Discrete actions");
        return check_reduced_obs(h, "td_step", io->obs_format, io->obs_dev);
    }
    return TD_OK;
}

// launch the fused step for envs [begin, begin + count) on `s`
// td_step_io.obs_incremental is honoured only for the buffer the library itself filled last, and only when that buffer
// is 16-byte aligned: the in-place update stores float4 (obs_dense_incremental); elsewhere the full write takes its
// scalar path
static bool obs_is_current(const td_handle *h, const td_step_io *io)
{
    return io->obs_incremental != 0 && io->obs_format == TD_OBS_F32 && io->obs_dev != nullptr && io->obs_dev == h->obs_synced &&
           (reinterpret_cast<uintptr_t>(io->obs_dev) & 15) == 0;
}

// Where a step kernel goes: straight onto a stream, or into a graph under construction (td_step_host).
struct LaunchTarget {
    cudaStream_t stream = nullptr;
    cudaGraph_t graph = nullptr;
    const cudaGraphNode_t *deps = nullptr;
    size_t n_deps = 0;
    cudaGraphNode_t node = nullptr;      // out: the kernel node that was added
};

static int launch_step(td_handle *h, const td_step_io *io, int begin, int count, LaunchTarget &t, bool incremental)
{
    StepParams p;
    fill_params(h, p);
    p.io = *io;
    p.env_begin = begin;
    p.n_envs = begin + count;
    const int wpc = step_warps_per_cta(h, incremental);                   // one env per warp
    const int grid = (count + wpc - 1) / wpc, block = wpc * 32;
    const size_t smem = wpc == kWarpsPerCta ? step_smem_bytes(h) : (size_t)wpc * h->smem_per_warp;
    const StepKernel kernel = step_kernel(h->L, h->kind, io->multi_action != 0, incremental,
                                          io->obs_dev ? io->obs_format : TD_OBS_F32, scripted_lv1_on_device(h, io));
    if (!kernel) return fail(h, TD_E_INVALID, "td_step: no step kernel is compiled for this configuration");
    cudaError_t e;
    if (!t.graph) {
        kernel<<<grid, block, smem, t.stream>>>(p);
        e = cudaGetLastError();
    } else {
        void *args[] = {&p};
        cudaKernelNodeParams kp;
        memset(&kp, 0, sizeof(kp));
        kp.func = reinterpret_cast<void *>(kernel);
        kp.gridDim = dim3(grid);
        kp.blockDim = dim3(block);
        kp.sharedMemBytes = (unsigned)smem;
        kp.kernelParams = args;
        e = cudaGraphAddKernelNode(&t.node, t.graph, t.deps, t.n_deps, &kp);
    }
    if (e != cudaSuccess) return fail(h, TD_E_CUDA, std::string("td_step: ") + cudaGetErrorString(e));
    return TD_OK;
}

extern "C" int td_step(td_handle *h, const td_step_io *io, void *stream)
{
    if (!h) return TD_E_INVALID;
    int rc = check_io(h, io);
    if (rc != TD_OK) return rc;
    TD_CUDA(h, cudaSetDevice(h->device));
    LaunchTarget t;
    t.stream = (cudaStream_t)stream;
    rc = launch_step(h, io, 0, h->n_envs, t, obs_is_current(h, io));
    if (rc != TD_OK) return rc;
    h->obs_synced = io->obs_format == TD_OBS_F32 ? io->obs_dev : nullptr;
    h->steps += h->n_envs;
    return TD_OK;
}

// td_observe_kernel over the records [0, n) at records_dev (read only) into obs_dev, of a validated format
static int launch_observe(td_handle *h, const char *who, const void *records_dev, int n, int obs_format, void *obs_dev,
                          void *stream)
{
    StepParams p;
    fill_params(h, p);
    p.records = static_cast<uint8_t *>(const_cast<void *>(records_dev));
    p.n_envs = n;
    void *args[] = {&p, &obs_dev};
    const cudaError_t e = cudaLaunchKernel(observe_kernel(h->L, obs_format), dim3((n + kWarpsPerCta - 1) / kWarpsPerCta),
                                           dim3(kWarpsPerCta * 32), args, smem_of(h), (cudaStream_t)stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(h, TD_E_CUDA, std::string(who) + ": " + cudaGetErrorString(e));
    }
    return TD_OK;
}

extern "C" int td_observe(td_handle *h, float *obs_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!obs_dev) return fail(h, TD_E_INVALID, "td_observe: obs_dev is NULL");
    if (h->n_maps < 1) return fail(h, TD_E_STATE, "td_observe: upload maps and reset first");
    TD_CUDA(h, cudaSetDevice(h->device));
    const int rc = launch_observe(h, "td_observe", h->records, h->n_envs, TD_OBS_F32, obs_dev, stream);
    h->obs_synced = obs_dev;
    return rc;
}

extern "C" int td_observe_as(td_handle *h, int obs_format, void *obs_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (obs_format == TD_OBS_F32) return td_observe(h, static_cast<float *>(obs_dev), stream);
    if (!obs_dev) return fail(h, TD_E_INVALID, "td_observe_as: obs_dev is NULL");
    const int rc = check_reduced_obs(h, "td_observe_as", obs_format, obs_dev);
    if (rc != TD_OK) return rc;
    if (h->n_maps < 1) return fail(h, TD_E_STATE, "td_observe_as: upload maps and reset first");
    TD_CUDA(h, cudaSetDevice(h->device));
    return launch_observe(h, "td_observe_as", h->records, h->n_envs, obs_format, obs_dev, stream);
}

// td_action_mask_kernel over the handle's records
static int launch_action_mask(td_handle *h, uint8_t *def_mask_dev, uint8_t *atk_mask_dev, void *stream)
{
    StepParams p;
    fill_params(h, p);
    void *args[] = {&p, &def_mask_dev, &atk_mask_dev};
    const cudaError_t e = cudaLaunchKernel(action_mask_kernel(h->L), dim3(grid_of(h)), dim3(kWarpsPerCta * 32), args,
                                           mask_smem_of(h), (cudaStream_t)stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(h, TD_E_CUDA, std::string("td_action_mask: ") + cudaGetErrorString(e));
    }
    return TD_OK;
}

extern "C" int td_action_mask(td_handle *h, uint8_t *def_mask_dev, uint8_t *atk_mask_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!def_mask_dev && !atk_mask_dev) return fail(h, TD_E_INVALID, "td_action_mask: both masks are NULL");
    if (def_mask_dev && h->kind == TD_KIND_ATK)
        return fail(h, TD_E_INVALID, "td_action_mask: the attacker env has no defender mask (its defender is scripted)");
    if (atk_mask_dev && h->kind == TD_KIND_DEF)
        return fail(h, TD_E_INVALID, "td_action_mask: the defender env has no attacker mask (its attacker is scripted)");
    if (h->n_maps < 1) return fail(h, TD_E_STATE, "td_action_mask: upload maps and reset first");
    TD_CUDA(h, cudaSetDevice(h->device));
    return launch_action_mask(h, def_mask_dev, atk_mask_dev, stream);
}

// Compact snapshots (SURVEY 8(f) f4): the env records as they are, and observations rebuilt from them later.
extern "C" int td_snapshot(td_handle *h, void *records_out_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!records_out_dev) return fail(h, TD_E_INVALID, "td_snapshot: records_out_dev is NULL");
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaMemcpyAsync(records_out_dev, h->records, (size_t)h->n_envs * h->record_bytes,
                               cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return TD_OK;
}

extern "C" int td_observe_snapshot(td_handle *h, const void *records_dev, int n, float *obs_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!records_dev || !obs_dev || n < 1) return fail(h, TD_E_INVALID, "td_observe_snapshot: bad arguments");
    TD_CUDA(h, cudaSetDevice(h->device));
    const int rc = launch_observe(h, "td_observe_snapshot", records_dev, n, TD_OBS_F32, obs_dev, stream);
    if (obs_dev == h->obs_synced) h->obs_synced = nullptr;      // the buffer now shows the snapshot, not the live envs
    return rc;
}

// One host-buffer step (td_step_host).  Inputs the step kernel can read from the caller's page-locked buffer
// itself (small actions) and outputs it can store there itself (the packed record per env) need no copy at all: the
// call is then one kernel launch and the synchronisation.  Whatever is left is a list of operations per chunk of
// envs -- action copies (host -> device), the step kernel, output copies (device -> host); instances are
// independent, so a chunk is a complete unit of work.  The list is instantiated once as a CUDA graph whose chunk
// kernels are independent branches behind their own copies (or chained, TD_OPT_HOST_CHAIN) and replayed with one
// launch, or issued on the stream call by call (TD_OPT_HOST_GRAPH = 0, pageable host memory).

static void host_chunk_copies(const td_handle *h, const td_step_io *io, const td_host_io *host, size_t b, size_t n,
                              std::vector<HostCopy> &in, std::vector<HostCopy> &out)
{
    const size_t cells = (size_t)h->cells;
    const size_t def_w = io->multi_action ? 6 * cells : 1;               // int64 elements per env
    const size_t atk_w = TD_ROADS * TD_CLUSTER;
    in.clear();
    out.clear();
    // (a NULL host pointer here: the kernel reads that input straight from the caller's page-locked buffer, td_step_host)
    if (h->kind != TD_KIND_ATK && host->def_action_host)
        in.push_back({(int64_t *)io->def_action_dev + b * def_w, host->def_action_host + b * def_w, n * def_w * 8});
    if (h->kind != TD_KIND_DEF && host->atk_action_host)
        in.push_back({(int64_t *)io->atk_action_dev + b * atk_w, host->atk_action_host + b * atk_w, n * atk_w * 8});
    if (h->kind == TD_KIND_ATK && io->def_action_dev && host->def_action_host)       // host-resolved scripted defender
        in.push_back({(int64_t *)io->def_action_dev + b, host->def_action_host + b, n * 8});
    if (io->opponent_dev && host->opponent_host)
        in.push_back({(uint8_t *)io->opponent_dev + b, host->opponent_host + b, n});
    if (io->opponent_cluster_dev && host->opponent_cluster_host)
        in.push_back({(uint32_t *)io->opponent_cluster_dev + b, host->opponent_cluster_host + b, n * 4});
    // device -> host: outputs that sit at matching offsets of one device slab and one host slab (as TDVecEnv
    // allocates them) are merged into a single copy when the chunk is the whole batch
    struct Seg { char *dst; const char *src; size_t bytes; };
    Seg segs[9];
    int ns = 0;
    auto add = [&](void *dst, const void *src, size_t elem_bytes) {
        if (dst && src)
            segs[ns++] = Seg{static_cast<char *>(dst) + b * elem_bytes, static_cast<const char *>(src) + b * elem_bytes,
                             n * elem_bytes};
    };
    add(host->obs_host, io->obs_dev, TD_NCHANNELS * cells * (io->obs_format == TD_OBS_BF16 ? 2 : io->obs_format == TD_OBS_U8 ? 1 : 4));
    add(host->reward_host, io->reward_dev, sizeof(double));
    add(host->done_host, io->done_dev, 1);
    add(host->win_host, io->win_dev, 1);
    add(host->allow_next_host, io->allow_next_dev, 1);
    if (h->kind != TD_KIND_ATK) add(host->real_def_host, io->real_def_dev, def_w * 8);
    if (h->kind != TD_KIND_DEF) add(host->real_atk_host, io->real_atk_dev, atk_w * 8);
    if (h->kind != TD_KIND_ATK) add(host->fail_def_host, io->fail_def_dev, sizeof(int32_t));
    if (h->kind != TD_KIND_DEF) add(host->fail_atk_host, io->fail_atk_dev, 4 * sizeof(int32_t));
    std::sort(segs, segs + ns, [](const Seg &x, const Seg &y) { return x.src < y.src; });
    for (int i = 0; i < ns;) {
        Seg m = segs[i];
        int j = i + 1;
        while (j < ns && segs[j].src >= m.src + m.bytes && segs[j].src - (m.src + m.bytes) <= 256 &&
               segs[j].src - m.src == segs[j].dst - m.dst) {
            m.bytes = (size_t)(segs[j].src - m.src) + segs[j].bytes;
            ++j;
        }
        out.push_back({m.dst, m.src, m.bytes});
        i = j;
    }
}

static bool host_pointer_is_pinned(const void *p)
{
    if (!p) return true;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

// How td_step_host cuts the batch.  Measured on B200 (tools/e2e_sweep.py, profiles/r02_e2e_sweep.txt; def-small, 65,536
// envs, device step 0.2135 ms): one chunk 0.2462 ms per call; CHAINED chunk kernels lose (every boundary costs ~10 us:
// 2 / 4 chunks 0.2512 / 0.2790 ms); INDEPENDENT chunk kernels -- graph branches that start as soon as their own
// actions are in, and fill the SMs the chunk before them leaves -- win when the first chunk is short: chunks of
// n/16, 3n/16, 9n/16, rest = 0.2380 ms (0.90 of the device step; 2p-large 0.5424 -> 0.4806 ms, def-middle 0.4489 ->
// 0.4387 ms).  When the action copy is as long as the step (>= 8 MB: the attacker's (3, 8) int64 action at 65,536 envs,
// Box actions) equal chunks are better (atk-small 0.5760 -> 0.4530 ms, PCIe-bound).
struct HostPlan { int chunks; int first; bool chain; };

static HostPlan host_plan(const td_handle *h, const td_step_io *io, const td_host_io *host, bool graph)
{
    HostPlan p;
    const size_t cells = (size_t)h->cells;
    // bytes per env that travel through copy nodes (inputs the kernel reads from host memory itself do not count)
    const size_t action_bytes = ((h->kind != TD_KIND_ATK && host->def_action_host) ? (io->multi_action ? 6 * cells * 8 : 8) : 0) +
                                ((h->kind != TD_KIND_DEF && host->atk_action_host) ? (size_t)TD_ROADS * TD_CLUSTER * 8 : 0);
    const bool automatic = h->host_chunks <= 0;
    p.chain = graph ? h->host_chain : true;                       // plain stream launches are ordered by the stream
    p.chunks = automatic ? ((graph && !p.chain && h->n_envs >= 8192 && action_bytes > 0) ? 4 : 1) : h->host_chunks;
    p.chunks = std::max(1, std::min(p.chunks, h->n_envs));
    // a copy about as long as the step (>= 8 MB) wants equal chunks, a short one a short first chunk
    p.first = h->host_first_chunk >= 0 ? h->host_first_chunk
                                       : ((automatic && action_bytes * (size_t)h->n_envs < ((size_t)8 << 20)) ? h->n_envs / 16 : 0);
    return p;
}

// envs per chunk: equal parts, or -- first = F > 0 -- chunks that grow by a factor of three (F, 3F, 9F, ..., the last
// one takes the rest): the first actions arrive after a few microseconds and every kernel finds its inputs in place
// when the one before it drains
static std::vector<int> host_chunk_sizes(const td_handle *h, const HostPlan &plan)
{
    std::vector<int> counts;
    int left = h->n_envs;
    if (plan.first > 0 && plan.chunks >= 2) {
        long long size = plan.first;
        while ((int)counts.size() < plan.chunks - 1 && size < left) {
            counts.push_back((int)size);
            left -= (int)size;
            size *= 3;
        }
        counts.push_back(left);
        return counts;
    }
    const int parts = std::max(1, std::min(plan.chunks, left));
    for (int c = 0; c < parts; ++c) counts.push_back(left / parts + (c < left % parts ? 1 : 0));
    return counts;
}

// The operations of one td_step_host call, chunk by chunk: input copies, the step kernel, output copies -- issued on
// t.stream, or added to t.graph.  In the graph the output copies wait for their kernel; the kernels are chained
// (each waits for its own input copies and the kernel before it), or -- plan.chain off -- independent branches that
// start as soon as their own inputs are in, with the input copies of successive chunks following each other (chunk
// order on the copy engine).
static int issue_host_chunks(td_handle *h, const td_step_io *io, const td_host_io *host, const HostPlan &plan,
                             bool incremental, LaunchTarget t)
{
    auto copy = [&](const HostCopy &cp, cudaMemcpyKind dir, const cudaGraphNode_t *deps, size_t n_deps, cudaGraphNode_t *node) {
        cudaError_t e = t.graph ? cudaGraphAddMemcpyNode1D(node, t.graph, deps, n_deps, cp.dst, cp.src, cp.bytes, dir)
                                : cudaMemcpyAsync(cp.dst, cp.src, cp.bytes, dir, t.stream);
        return e == cudaSuccess ? TD_OK : fail(h, TD_E_CUDA, std::string("td_step_host: copy: ") + cudaGetErrorString(e));
    };
    std::vector<HostCopy> &in = h->host_in, &out = h->host_out;
    std::vector<cudaGraphNode_t> prev_copies, deps;
    cudaGraphNode_t prev_kernel = nullptr;
    int begin = 0, rc;
    for (int count : host_chunk_sizes(h, plan)) {
        host_chunk_copies(h, io, host, (size_t)begin, (size_t)count, in, out);
        deps.clear();
        for (const HostCopy &cp : in) {
            cudaGraphNode_t n = nullptr;
            if ((rc = copy(cp, cudaMemcpyHostToDevice, plan.chain ? nullptr : prev_copies.data(), plan.chain ? 0 : prev_copies.size(), &n)) != TD_OK)
                return rc;
            deps.push_back(n);
        }
        prev_copies = deps;
        if (prev_kernel && plan.chain) deps.push_back(prev_kernel);
        t.deps = deps.data();
        t.n_deps = deps.size();
        if ((rc = launch_step(h, io, begin, count, t, incremental)) != TD_OK) return rc;
        for (const HostCopy &cp : out) {
            cudaGraphNode_t n = nullptr;
            if ((rc = copy(cp, cudaMemcpyDeviceToHost, &t.node, 1, &n)) != TD_OK) return rc;
        }
        prev_kernel = t.node;
        begin += count;
    }
    return TD_OK;
}

static int build_host_graph(td_handle *h, const td_step_io *io, const td_host_io *host, const HostPlan &plan, bool incremental,
                            cudaGraphExec_t *exec_out)
{
    LaunchTarget t;
    TD_CUDA(h, cudaGraphCreate(&t.graph, 0));
    int rc = issue_host_chunks(h, io, host, plan, incremental, t);
    if (rc == TD_OK) {
        const cudaError_t e = cudaGraphInstantiate(exec_out, t.graph, 0);
        if (e != cudaSuccess) rc = fail(h, TD_E_CUDA, std::string("td_step_host: cudaGraphInstantiate: ") + cudaGetErrorString(e));
    }
    cudaGraphDestroy(t.graph);
    return rc;
}

extern "C" int td_step_host(td_handle *h, const td_step_io *io, const td_host_io *host, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!host) return fail(h, TD_E_INVALID, "td_step_host: host is NULL");
    int rc = check_io(h, io);
    if (rc != TD_OK) return rc;
    if (h->kind != TD_KIND_ATK && !host->def_action_host) return fail(h, TD_E_INVALID, "td_step_host: def_action_host is required");
    if (h->kind != TD_KIND_DEF && !host->atk_action_host) return fail(h, TD_E_INVALID, "td_step_host: atk_action_host is required");
    TD_CUDA(h, cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    td_step_io io_local = *io;
    td_host_io host_local = *host;
    if (host->packed_host) {
        // zero-copy outputs: the kernel stores every env's packed record straight into the caller's page-locked buffer
        void *dptr = nullptr;
        if (cudaHostGetDevicePointer(&dptr, host->packed_host, 0) != cudaSuccess) {
            cudaGetLastError();
            return fail(h, TD_E_INVALID, "td_step_host: packed_host must be page-locked, device-mapped host memory");
        }
        io_local.packed_out_dev = dptr;
    }
    {
        // zero-copy inputs: the step kernel reads small actions from the caller's page-locked buffer itself.  For the
        // 8-byte Discrete action that costs +1.2 us per step at 65,536 envs against +13 us for a copy-engine node in
        // front of the kernel (tools/e2e_breakdown.py: def-small 0.2376 -> 0.2317 ms per call).  Kernel-side PCIe reads
        // sustain ~20 GB/s, so the rule is bytes per env against the env's share of the step (~ its observation):
        // 3 x action bytes <= cells.  That takes the (3, 8) int64 attacker action on 30x30 boards (2p-large 0.4868 ->
        // 0.4702 ms) and leaves it to the copy engine on 10x10 boards (atk-small: 0.4551 ms copied, 0.6117 ms zero-copy).
        auto mapped = [](const void *hp) -> void * {
            void *d = nullptr;
            if (!hp || cudaHostGetDevicePointer(&d, const_cast<void *>(hp), 0) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            return d;
        };
        const int zc = h->host_zero_copy;
        const size_t def_bytes = io->multi_action ? 6 * (size_t)h->cells * 8 : 8, atk_bytes = (size_t)TD_ROADS * TD_CLUSTER * 8;
        auto wanted = [&](size_t bytes_per_env) { return zc > 0 || (zc < 0 && 3 * bytes_per_env <= (size_t)h->cells); };
        if (h->kind != TD_KIND_ATK && wanted(def_bytes))
            if (void *d = mapped(host->def_action_host)) { io_local.def_action_dev = static_cast<const int64_t *>(d); host_local.def_action_host = nullptr; }
        if (h->kind != TD_KIND_DEF && wanted(atk_bytes))
            if (void *d = mapped(host->atk_action_host)) { io_local.atk_action_dev = static_cast<const int64_t *>(d); host_local.atk_action_host = nullptr; }
    }
    io = &io_local;
    host = &host_local;
    const bool incremental = obs_is_current(h, io);
    h->obs_synced = nullptr;                                    // until every chunk was launched

    // the PCIe-bound variant that also ships the observation (1.2 GB per step at 65,536 envs) gains nothing from a
    // graph and measured slower through graph memcpy nodes (1.9e6 vs 3.1e6 env-steps/s): plain stream copies
    bool use_graph = h->host_graph != 0 && host->obs_host == nullptr;
    {
        // nothing left to copy in either direction: the call is one kernel launch and the synchronisation
        std::vector<HostCopy> &in = h->host_in, &out = h->host_out;
        host_chunk_copies(h, io, host, 0, (size_t)h->n_envs, in, out);
        if (in.empty() && out.empty()) use_graph = false;
    }
    td_handle::HostGraph *hit = nullptr;
    std::vector<unsigned char> &key = h->host_key;              // scratch of the handle: no allocation per call
    HostPlan plan = {1, 0, true};
    if (use_graph) {
        // everything a graph bakes in: the buffers of both structs, the cut of the batch, the kernel that was picked,
        // map pool, generators, difficulty
        plan = host_plan(h, io, host, true);
        const unsigned long long extra[3] = {(unsigned long long)plan.chunks | ((unsigned long long)plan.first << 20) | (plan.chain ? 1ull << 52 : 0ull),
                                             incremental ? 1ull : 0ull, h->cfg_generation};
        const void *ptrs[3] = {h->maps, h->mt, h->records};
        const int ints[2] = {h->difficulty | (h->opponent_seeded ? 0x100 : 0) | (h->map_stride << 9), h->n_maps};
        key.resize(sizeof(td_step_io) + sizeof(td_host_io) + sizeof(extra) + sizeof(ints) + sizeof(ptrs));
        unsigned char *k = key.data();
        memcpy(k, io, sizeof(td_step_io)); k += sizeof(td_step_io);
        memcpy(k, host, sizeof(td_host_io)); k += sizeof(td_host_io);
        memcpy(k, extra, sizeof(extra)); k += sizeof(extra);
        memcpy(k, ints, sizeof(ints)); k += sizeof(ints);
        memcpy(k, ptrs, sizeof(ptrs));
        for (auto &g : h->host_graphs)
            if (g.key == key) { hit = &g; break; }
        if (!hit) {
            // a graph keeps raw host addresses: only page-locked buffers qualify (checked when the graph is built;
            // a cached graph vouches for its buffers as long as the caller keeps them allocated)
            const void *hp[] = {host->def_action_host, host->atk_action_host, host->opponent_host, host->obs_host,
                                host->reward_host, host->done_host, host->win_host, host->allow_next_host,
                                host->real_def_host, host->real_atk_host, host->fail_def_host, host->fail_atk_host,
                                host->opponent_cluster_host, host->packed_host};
            for (const void *q : hp) use_graph = use_graph && host_pointer_is_pinned(q);
        }
    }
    if (use_graph) {
        if (s == nullptr || s == cudaStreamLegacy) {
            // the legacy default stream cannot launch a graph: a blocking internal stream takes its place (work on
            // it is ordered after everything already in the legacy stream, and the call synchronises it below)
            if (!h->host_stream) TD_CUDA(h, cudaStreamCreateWithFlags(&h->host_stream, cudaStreamDefault));
            s = h->host_stream;
        }
        if (!hit) {
            cudaGraphExec_t exec = nullptr;
            rc = build_host_graph(h, io, host, plan, incremental, &exec);
            if (rc != TD_OK) return rc;
            if (h->host_graphs.size() >= 16) {                      // evict the least recently used
                size_t lru = 0;
                for (size_t i = 1; i < h->host_graphs.size(); ++i)
                    if (h->host_graphs[i].used < h->host_graphs[lru].used) lru = i;
                cudaGraphExecDestroy(h->host_graphs[lru].exec);
                h->host_graphs.erase(h->host_graphs.begin() + (long)lru);
            }
            h->host_graphs.push_back({key, exec, 0});
            hit = &h->host_graphs.back();
        }
        hit->used = ++h->host_graph_clock;
        TD_CUDA(h, cudaGraphLaunch(hit->exec, s));
    } else {
        // plain stream launches (pageable host memory or TD_OPT_HOST_GRAPH = 0)
        LaunchTarget t;
        t.stream = s;
        rc = issue_host_chunks(h, io, host, host_plan(h, io, host, false), incremental, t);
        if (rc != TD_OK) return rc;
    }
    h->obs_synced = io->obs_format == TD_OBS_F32 ? io->obs_dev : nullptr;
    h->steps += h->n_envs;
    TD_CUDA(h, cudaStreamSynchronize(s));
    return TD_OK;
}

extern "C" int td_invalidate_obs(td_handle *h)
{
    if (!h) return TD_E_INVALID;
    h->obs_synced = nullptr;
    return TD_OK;
}

extern "C" int td_set_option(td_handle *h, int option, int value)
{
    if (!h) return TD_E_INVALID;
    switch (option) {
    case TD_OPT_HOST_CHUNKS:
        if (value < 0) return fail(h, TD_E_INVALID, "td_set_option: host chunks < 0");
        h->host_chunks = value;
        return TD_OK;
    case TD_OPT_HOST_GRAPH: h->host_graph = value != 0; return TD_OK;
    case TD_OPT_HOST_CHAIN:
        h->host_chain = value != 0;
        h->cfg_generation += 1;      // cached host-step graphs were built with the other shape
        return TD_OK;
    case TD_OPT_HOST_FIRST_CHUNK:
        h->host_first_chunk = value < 0 ? -1 : value;
        h->cfg_generation += 1;
        return TD_OK;
    case TD_OPT_HOST_ZERO_COPY:
        h->host_zero_copy = value < 0 ? -1 : value > 0 ? 1 : 0;
        return TD_OK;
    case TD_OPT_GENERIC_KERNELS:
        h->generic_kernels = value != 0;
        h->cfg_generation += 1;      // cached host-step graphs hold the kernel that was picked when they were built
        return TD_OK;
    default: return fail(h, TD_E_INVALID, "td_set_option: unknown option");
    }
}

extern "C" int td_get_state(td_handle *h, int first_env, int n, void *blob)
{
    if (!h) return TD_E_INVALID;
    if (!blob || first_env < 0 || n < 1 || first_env + n > h->n_envs) return fail(h, TD_E_INVALID, "td_get_state: bad range");
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaDeviceSynchronize());
    TD_CUDA(h, cudaMemcpy(blob, h->records + (size_t)first_env * h->record_bytes, (size_t)n * h->record_bytes, cudaMemcpyDeviceToHost));
    return TD_OK;
}

extern "C" int td_set_state(td_handle *h, int first_env, int n, const void *blob)
{
    if (!h) return TD_E_INVALID;
    h->obs_synced = nullptr;                                    // no buffer shows the state being written
    if (!blob || first_env < 0 || n < 1 || first_env + n > h->n_envs) return fail(h, TD_E_INVALID, "td_set_state: bad range");
    const uint8_t *b = static_cast<const uint8_t *>(blob);
    const int enemy_cap = step_enemy_cap(h->L);
    for (int i = 0; i < n; ++i) {
        const uint8_t *rec = b + (size_t)i * h->record_bytes;
        const td_env_header *hd = reinterpret_cast<const td_env_header *>(rec);
        if (hd->n_towers > TD_CAP_TOWERS || hd->n_enemies > enemy_cap || hd->map_id < 0 ||
            (h->n_maps > 0 && hd->map_id >= h->n_maps) || hd->rng_pos < 0 || hd->rng_pos > kMtWords ||
            hd->pad0 > h->rng_cache_words || hd->pad1 < 0 || hd->pad1 > hd->pad0)
            return fail(h, TD_E_INVALID, "td_set_state: record header out of range");
        // road bits of the record's own static map: enemies walk the road (movement follows its direction bits and
        // would leave the board from any other cell, or from the end cell, where the reference removes them), towers
        // stand beside it
        const MapHdr *mh = reinterpret_cast<const MapHdr *>(rec + h->off_static);
        const uint8_t *road = rec + h->off_static + kMapHdrBytes;
        const td_tower_rec *tw = reinterpret_cast<const td_tower_rec *>(rec + h->off_towers);
        for (int t = 0; t < hd->n_towers; ++t)
            if (tw[t].loc >= h->cells || (tw[t].type_lv >> 2) >= TD_NLV || (road[tw[t].loc] & 1))
                return fail(h, TD_E_INVALID, "td_set_state: bad tower record");
        const td_enemy_rec *en = reinterpret_cast<const td_enemy_rec *>(rec + h->off_enemies);
        for (int e = 0; e < hd->n_enemies; ++e)
            if (en[e].loc >= h->cells || (en[e].type_lv >> 2) >= TD_NLV || !(road[en[e].loc] & 1) || en[e].loc == mh->end)
                return fail(h, TD_E_INVALID, "td_set_state: bad enemy record");
    }
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaDeviceSynchronize());
    TD_CUDA(h, cudaMemcpy(h->records + (size_t)first_env * h->record_bytes, blob, (size_t)n * h->record_bytes, cudaMemcpyHostToDevice));
    return TD_OK;
}

extern "C" int td_get_stats(td_handle *h, td_stats *out, void *stream)
{
    if (!h || !out) return TD_E_INVALID;
    TD_CUDA(h, cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    td_stats_kernel<<<1, 256, 0, s>>>(h->stats, h->n_envs, h->steps, h->stats_dev);
    TD_CUDA(h, cudaGetLastError());
    TD_CUDA(h, cudaMemcpyAsync(out, h->stats_dev, sizeof(td_stats), cudaMemcpyDeviceToHost, s));
    TD_CUDA(h, cudaStreamSynchronize(s));
    return TD_OK;
}

extern "C" int td_reset_stats(td_handle *h, void *stream)
{
    if (!h) return TD_E_INVALID;
    TD_CUDA(h, cudaSetDevice(h->device));
    TD_CUDA(h, cudaMemsetAsync(h->stats, 0, (size_t)h->n_envs * sizeof(EnvStats), (cudaStream_t)stream));
    h->steps = 0;
    return TD_OK;
}

// ------------------------------------------------------------------------------------------------
// rollout consumer (td_rollout.cuh)

extern "C" int td_rollout_mask(td_handle *h, int which, int64_t *action_dev, const uint8_t *allow_next_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!action_dev || !allow_next_dev || which < 0 || which > 1) return fail(h, TD_E_INVALID, "td_rollout_mask: bad arguments");
    TD_CUDA(h, cudaSetDevice(h->device));
    const int width = which == 0 ? 1 : TD_ROADS * TD_CLUSTER;
    const int total = h->n_envs * width;
    rollout_mask_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        action_dev, allow_next_dev, h->n_envs, width, which == 0 ? 1 : 2,
        which == 0 ? (int64_t)6 * h->cells : (int64_t)TD_NTYPES);
    TD_CUDA(h, cudaGetLastError());
    return TD_OK;
}

extern "C" int td_rollout_record(td_handle *h, int which, const int64_t *action_dev, const int64_t *real_action_dev,
                                 const double *reward_dev, const uint8_t *done_dev, double penalty,
                                 float *rewards_row_dev, uint8_t *dones_row_dev, int64_t *actions_row_dev, void *stream)
{
    if (!h) return TD_E_INVALID;
    if (!action_dev || !real_action_dev || !reward_dev || !done_dev || !rewards_row_dev || !dones_row_dev ||
        which < 0 || which > 1)
        return fail(h, TD_E_INVALID, "td_rollout_record: bad arguments");
    TD_CUDA(h, cudaSetDevice(h->device));
    const int width = which == 0 ? 1 : TD_ROADS * TD_CLUSTER;
    rollout_record_kernel<<<(h->n_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        action_dev, real_action_dev, reward_dev, done_dev, h->n_envs, width, penalty, rewards_row_dev,
        dones_row_dev, actions_row_dev);
    TD_CUDA(h, cudaGetLastError());
    return TD_OK;
}

extern "C" int td_gae(int horizon, int n, const float *rewards_dev, const uint8_t *dones_dev, const float *values_dev,
                      const float *next_value_dev, double gamma, double lam, float *advs_dev, float *returns_dev,
                      void *stream)
{
    if (horizon < 1 || n < 1 || !rewards_dev || !dones_dev || !values_dev || !next_value_dev || !advs_dev || !returns_dev)
        return fail(nullptr, TD_E_INVALID, "td_gae: bad arguments");
    // no handle here: launch on the device that owns the buffers, whatever device is current on this thread
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, rewards_dev) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        return fail(nullptr, TD_E_INVALID, "td_gae: rewards_dev is not a device pointer");
    }
    if (cudaSetDevice(attr.device) != cudaSuccess) return fail(nullptr, TD_E_CUDA, "td_gae: cudaSetDevice failed");
    gae_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(horizon, n, rewards_dev, dones_dev, values_dev,
                                                                next_value_dev, gamma, lam, advs_dev, returns_dev);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(nullptr, TD_E_CUDA, std::string("td_gae: ") + cudaGetErrorString(e));
    return TD_OK;
}

// ---- compressible observation memory (td_b200.h) ---------------------------------------------------------------
// The driver entry points are looked up through the runtime (cudaGetDriverEntryPoint), so the library keeps loading
// on hosts without a driver (the CPU-only ABI tests).
namespace {
struct CompAlloc { CUmemGenericAllocationHandle handle; size_t size; int device; };
std::mutex g_comp_mutex;
std::map<void *, CompAlloc> g_comp_allocs;

template <typename Fn> bool driver_fn(const char *name, Fn *out)
{
    void *p = nullptr;
    cudaDriverEntryPointQueryResult st;
    if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess || !p) {
        cudaGetLastError();
        return false;
    }
    *out = reinterpret_cast<Fn>(p);
    return true;
}
}  // namespace

extern "C" int td_alloc_compressible(int device, size_t bytes, void **ptr_out, int *compressed_out)
{
    if (!ptr_out || bytes == 0) return fail(nullptr, TD_E_INVALID, "td_alloc_compressible: bad arguments");
    *ptr_out = nullptr;
    if (compressed_out) *compressed_out = 0;
    if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, TD_E_CUDA, "td_alloc_compressible: no such CUDA device");
    }
    CUresult (*get_attr)(int *, CUdevice_attribute, CUdevice) = nullptr;
    CUresult (*get_gran)(size_t *, const CUmemAllocationProp *, CUmemAllocationGranularity_flags) = nullptr;
    CUresult (*create)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *, unsigned long long) = nullptr;
    CUresult (*get_prop)(CUmemAllocationProp *, CUmemGenericAllocationHandle) = nullptr;
    CUresult (*reserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*set_access)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t) = nullptr;
    CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*addr_free)(CUdeviceptr, size_t) = nullptr;
    if (!driver_fn("cuDeviceGetAttribute", &get_attr) || !driver_fn("cuMemGetAllocationGranularity", &get_gran) ||
        !driver_fn("cuMemCreate", &create) || !driver_fn("cuMemGetAllocationPropertiesFromHandle", &get_prop) ||
        !driver_fn("cuMemAddressReserve", &reserve) || !driver_fn("cuMemMap", &map) || !driver_fn("cuMemSetAccess", &set_access) ||
        !driver_fn("cuMemUnmap", &unmap) || !driver_fn("cuMemRelease", &release) || !driver_fn("cuMemAddressFree", &addr_free))
        return fail(nullptr, TD_E_STATE, "td_alloc_compressible: the driver lacks the virtual memory management entry points");
    int supported = 0;
    if (get_attr(&supported, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, (CUdevice)device) != CUDA_SUCCESS || !supported)
        return fail(nullptr, TD_E_STATE, "td_alloc_compressible: the device does not support compressible memory");
    CUmemAllocationProp prop;
    memset(&prop, 0, sizeof(prop));
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t gran = 0;
    if (get_gran(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || gran == 0)
        return fail(nullptr, TD_E_CUDA, "td_alloc_compressible: cuMemGetAllocationGranularity failed");
    const size_t size = (bytes + gran - 1) / gran * gran;
    CompAlloc a;
    a.size = size;
    a.device = device;
    if (create(&a.handle, size, &prop, 0) != CUDA_SUCCESS) return fail(nullptr, TD_E_ALLOC, "td_alloc_compressible: cuMemCreate failed (out of memory?)");
    CUmemAllocationProp got;
    memset(&got, 0, sizeof(got));
    const bool compressed = get_prop(&got, a.handle) == CUDA_SUCCESS && got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC;
    CUdeviceptr p = 0;
    if (reserve(&p, size, gran, 0, 0) != CUDA_SUCCESS) { release(a.handle); return fail(nullptr, TD_E_ALLOC, "td_alloc_compressible: cuMemAddressReserve failed"); }
    if (map(p, size, 0, a.handle, 0) != CUDA_SUCCESS) { addr_free(p, size); release(a.handle); return fail(nullptr, TD_E_ALLOC, "td_alloc_compressible: cuMemMap failed"); }
    CUmemAccessDesc acc;
    memset(&acc, 0, sizeof(acc));
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (set_access(p, size, &acc, 1) != CUDA_SUCCESS || cudaMemset(reinterpret_cast<void *>(p), 0, size) != cudaSuccess ||
        cudaDeviceSynchronize() != cudaSuccess) {
        cudaGetLastError();
        unmap(p, size); addr_free(p, size); release(a.handle);
        return fail(nullptr, TD_E_CUDA, "td_alloc_compressible: cuMemSetAccess / zero fill failed");
    }
    {
        std::lock_guard<std::mutex> lock(g_comp_mutex);
        g_comp_allocs[reinterpret_cast<void *>(p)] = a;
    }
    *ptr_out = reinterpret_cast<void *>(p);
    if (compressed_out) *compressed_out = compressed ? 1 : 0;
    return TD_OK;
}

extern "C" int td_free_compressible(void *ptr)
{
    if (!ptr) return TD_OK;
    CompAlloc a;
    {
        std::lock_guard<std::mutex> lock(g_comp_mutex);
        auto it = g_comp_allocs.find(ptr);
        if (it == g_comp_allocs.end()) return fail(nullptr, TD_E_INVALID, "td_free_compressible: not a pointer from td_alloc_compressible");
        a = it->second;
        g_comp_allocs.erase(it);
    }
    CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*addr_free)(CUdeviceptr, size_t) = nullptr;
    if (!driver_fn("cuMemUnmap", &unmap) || !driver_fn("cuMemRelease", &release) || !driver_fn("cuMemAddressFree", &addr_free))
        return fail(nullptr, TD_E_STATE, "td_free_compressible: the driver lacks the virtual memory management entry points");
    cudaSetDevice(a.device);
    cudaDeviceSynchronize();
    const CUdeviceptr p = reinterpret_cast<CUdeviceptr>(ptr);
    const bool ok = unmap(p, a.size) == CUDA_SUCCESS;
    const bool ok2 = release(a.handle) == CUDA_SUCCESS;
    const bool ok3 = addr_free(p, a.size) == CUDA_SUCCESS;
    return ok && ok2 && ok3 ? TD_OK : fail(nullptr, TD_E_CUDA, "td_free_compressible: unmap / release failed");
}
