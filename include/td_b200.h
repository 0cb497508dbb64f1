/*
 * td_b200.h -- C ABI of the B200-native batched gym-TD board step.
 *
 * This is the drop-in boundary: the entry points below are what a binding of the
 * reference's operator interface for this path would call.  The reference has no
 * FFI (it is pure Python); the interface being replaced is the `TDBoard` method
 * set plus the three env wrappers' step() bodies:
 *
 *   td_create / td_destroy      <- TDBoard.__init__            gym_TD/envs/TDBoard.py:14-79
 *                                  TDGymBasic.__init__          gym_TD/envs/TDGymBasic.py:18-28
 *   td_set_config               <- paramConfig / config         gym_TD/envs/TDParam.py:1-100
 *   td_mapgen*                  <- TDRoadGen.create_road_v2     gym_TD/envs/TDRoadGen.py:4-199
 *                                  + map planes                 gym_TD/envs/TDBoard.py:31-59
 *   td_upload_maps              <- (the np_random map stream of TDGymBasic.reset, :42-51)
 *   td_reset                    <- TDGymBasic.reset             gym_TD/envs/TDGymBasic.py:37-55
 *   td_step                     <- TDDefense.step               gym_TD/envs/TDDefense.py:34-87
 *                                  TDAttack.step                gym_TD/envs/TDAttack.py:27-56
 *                                  TDMulti.step                 gym_TD/envs/TDMulti.py:46-138
 *                                  (which call tower_build/lvup/destruct, summon_cluster, step,
 *                                   done, get_states: TDBoard.py:199-385, 85-144)
 *   td_observe                  <- TDBoard.get_states           gym_TD/envs/TDBoard.py:85-144
 *   td_get_state / td_set_state <- (direct attribute access on board/env objects)
 *   td_seed_opponent            <- random.seed / `random` module use in TDGymBasic.py:81-196
 *
 * Conventions: every function returns 0 on success or a negative TD_E_* code; no C++
 * exception crosses the boundary; td_last_error() gives the message for the last failure
 * on a handle (or of td_create when h == NULL).  All kernels are launched asynchronously
 * on the caller's stream (a cudaStream_t passed as void*).  Pointers named *_dev are device
 * pointers owned by the caller (e.g. torch tensors); *_host are host pointers.  A handle
 * belongs to one device and is not thread-safe: the caller serialises calls on it.
 * There is no CPU fallback: without a CUDA device every compute entry point fails with
 * TD_E_CUDA.
 */
#ifndef TD_B200_H
#define TD_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TD_ABI_VERSION 3   /* 2: td_step_io grew `obs_incremental` (+ reserved_) at its end; 3: td_set_option,
                              config per handle, td_step_host as one graph launch.  Added since, without a layout
                              change: TD_OPT_GENERIC_KERNELS / HOST_CHAIN / HOST_FIRST_CHUNK / HOST_ZERO_COPY,
                              td_alloc_compressible / td_free_compressible, td_env_header.ep_kills_hi / ep_leaks_hi
                              in the formerly unused pad2 word, td_action_mask */

enum { TD_OK = 0, TD_E_INVALID = -1, TD_E_CUDA = -2, TD_E_ALLOC = -3, TD_E_STATE = -4,
       TD_E_OVERFLOW = -5 };

/* observation element types (td_step_io.obs_format, td_observe_as) */
enum { TD_OBS_F32 = 0, TD_OBS_BF16 = 1, TD_OBS_U8 = 2 };

/* env kinds (TDDefense / TDAttack / TDMulti) */
enum { TD_KIND_DEF = 0, TD_KIND_ATK = 1, TD_KIND_2P = 2 };

/* gym_TD/utils/fail_code.py:1-6 */
enum { TD_FC_SUCCESS = 0, TD_FC_COST_SHORTAGE = 1, TD_FC_INVALID_POSITION = 2, TD_FC_LV_MAX = 3,
       TD_FC_UNKNOWN_TARGET = 4, TD_FC_IMPOSSIBLE_CLUSTER = 5 };

#define TD_NTYPES 4     /* enemy_types == tower_types (TDParam.py:6-7) */
#define TD_NLV 2        /* max_enemy_lv == max_tower_lv == 1 (TDParam.py:3-4) */
#define TD_CLUSTER 8    /* max_cluster_length (TDParam.py:110) */
#define TD_ROADS 3      /* max_num_of_roads (TDParam.py:111) */
#define TD_NCHANNELS 45 /* TDBoard.n_channels(), TDBoard.py:146-154 */
#define TD_CAP_TOWERS 32
#define TD_CAP_ENEMIES 64
#define TD_MAX_L 64

/* snapshot of TDParam.config + hyper_parameters (same field meaning as the reference) */
typedef struct td_config {
    double enemy_LP[TD_NTYPES][TD_NLV];
    double enemy_speed[TD_NTYPES][TD_NLV];
    double enemy_defense[TD_NTYPES][TD_NLV];
    double enemy_cost[TD_NTYPES][TD_NLV];
    double tower_attack[TD_NTYPES][TD_NLV];
    double tower_cost[TD_NTYPES][TD_NLV];
    double tower_attack_interval[TD_NTYPES][TD_NLV];
    int32_t tower_range[TD_NTYPES][TD_NLV];
    int32_t tower_splash_range[TD_NTYPES][TD_NLV];
    double tower_destruct_return;
    double frozen_ratio;
    double attacker_init_cost, defender_init_cost, max_cost;
    double reward_kill, penalty_leak, reward_time;
    double attacker_cost_init_rate, attacker_cost_final_rate, defender_cost_rate;
    double enemy_upgrade_at;
    int32_t frozen_time;
    int32_t base_LP;            /* < 0 means None (no leakage ending) */
    int32_t tower_distance;
    int32_t attacker_action_interval, defender_action_interval;
    int32_t max_episode_steps;
    int32_t max_tower_lv;       /* must be 1 in this build */
    int32_t pad_;
} td_config;

/* One generated map in transfer form (host).  cells[i]: bits 0-3 = map[0..3] (road, road1..3),
 * bits 4-5 = map[5] (direction 0..3); dist[i] = map[4].  TDBoard.py:31-59. */
typedef struct td_map {
    int32_t map_size;
    int32_t num_roads;
    int32_t start[TD_ROADS];    /* r*L + c */
    int32_t end;
    int32_t max_dist;           /* np.max(map[4]) */
    int32_t n_randint;          /* randint() calls the generator made (seed-skip budget accounting) */
    uint8_t cells[TD_MAX_L * TD_MAX_L];
    uint8_t dist[TD_MAX_L * TD_MAX_L];
} td_map;

typedef struct td_handle td_handle;

/* Per-step device buffers.  Unused pointers may be NULL.  Leading dimension is n_envs. */
typedef struct td_step_io {
    /* inputs */
    const int64_t *def_action_dev;   /* DEF/2P: [n] Discrete, or [n,6,L,L] when multi_action != 0.
                                        ATK: optional host-resolved scripted defender (random_tower_lv0 on the env's
                                        np_random, TDGymBasic.py:117-121): [n] build actions type * L*L + r*L + c,
                                        < 0 = defender does nothing; NULL = the on-device scripted defender */
    const int64_t *atk_action_dev;   /* ATK/2P: [n,3,8] */
    const uint8_t *opponent_dev;     /* DEF only, optional host-resolved scripted attacker (random_enemy_lv1):
                                        [n] bytes, type | road<<4, 0xFF = attacker does nothing.  When NULL the
                                        on-device CPython-compatible generator seeded by td_seed_opponent is used;
                                        if that was never seeded there is no scripted opponent. */
    int32_t multi_action;            /* hyper_parameters.allow_multiple_actions */
    int32_t auto_reset;              /* re-initialise finished envs from the map pool inside the step */
    /* outputs */
    float *obs_dev;                  /* [n,45,L,L] float32; may be NULL to skip the observation */
    double *reward_dev;              /* [n] */
    uint8_t *done_dev;               /* [n] */
    int8_t *win_dev;                 /* [n] -1 None / 0 / 1; 2P: defender view (attacker = !defender when done) */
    uint8_t *allow_next_dev;         /* [n] bit0 defender, bit1 attacker (AllowNextMove) */
    int64_t *real_def_dev;           /* [n] Discrete RealAction, or [n,6,L,L] in multi_action mode */
    int64_t *real_atk_dev;           /* [n,3,8] */
    int32_t *fail_def_dev;           /* [n] */
    int32_t *fail_atk_dev;           /* [n,4]: count, then up to 3 codes (FailCode list of TDAttack/TDMulti) */
    /* options */
    int32_t obs_incremental;         /* != 0: obs_dev is the buffer this handle wrote its previous observation to
                                        (td_reset / td_observe / the last td_step) and nobody changed it since: the
                                        step then rewrites only what changed -- the planes that carry per-step
                                        scalars, the buildable plane, the old and new tower / enemy cells -- and
                                        leaves the static map planes and the untouched zeros alone.  The resulting
                                        tensor is bit-identical to a full write.  Ignored (full write) whenever the
                                        library cannot vouch for the buffer: another pointer than last time, after
                                        td_set_state, for envs that were reset inside the step, for board sizes
                                        without a specialised kernel, for a buffer that is not 16-byte aligned. */
    int32_t obs_format;              /* TD_OBS_F32 (0, default): obs_dev is float32, the reference layout.  TD_OBS_BF16 /
                                        TD_OBS_U8 (ABI 3): obs_dev points to [n,45,L,L] bfloat16 / uint8 elements instead
                                        (SURVEY 8(f) f4, reduced-precision planes): bf16 = the float32 value rounded to
                                        nearest-even, u8 = rint(min(v * 255, 255)).  Board sizes 10 / 20 / 30, Discrete
                                        defender actions, full writes only (obs_incremental is ignored); obs_dev must
                                        be 8- / 4-byte aligned. */
    /* more inputs (ABI 3) */
    const uint32_t *opponent_cluster_dev; /* DEF only, optional host-resolved scripted attacker with a free cluster
                                        (random_enemy_lv0 on the env's np_random, TDGymBasic.py:87-89): [n] words,
                                        bits 2k..2k+1 = enemy type of slot k (k < 8), bits 16-17 = road,
                                        0xFFFFFFFF = attacker does nothing.  Takes the place of opponent_dev. */
    void *packed_out_dev;            /* optional: [n] td_step_packed records (td_packed_stride bytes apart), every
                                        small per-step output of an env in ONE coalesced store.  May be page-locked
                                        HOST memory (device-accessible under UVA): the outputs then reach the host
                                        while the kernel runs.  Written in addition to the arrays above. */
} td_step_io;

/* One env's small outputs in one record.  DEF envs use the first 32 bytes (stride 32), ATK / 2P envs all 256. */
typedef struct td_step_packed {
    double reward;
    int64_t real_def;                /* Discrete RealAction (0 in multi_action mode: see real_def_dev) */
    int32_t fail_def;
    uint8_t done;
    int8_t win;
    uint8_t allow_next;
    uint8_t pad0_;
    int32_t pad1_[2];                /* -- 32 bytes: end of a DEF record */
    int32_t fail_atk[4];
    int32_t pad2_[4];
    int64_t real_atk[TD_ROADS * TD_CLUSTER];
} td_step_packed;                    /* 256 bytes */
int td_packed_stride(int env_kind);   /* 32 for TD_KIND_DEF, 256 otherwise */

/* byte offsets inside one env record, for td_get_state / td_set_state blobs */
typedef struct td_layout {
    int32_t record_bytes;
    int32_t off_header, off_towers, off_enemies, off_map6;
    int32_t tower_stride, enemy_stride;
    int32_t cap_towers, cap_enemies;
    int32_t map_record_bytes;
    int32_t mt_words;           /* 624 */
    int32_t pad_;
} td_layout;

/* header of an env record (what td_get_state returns at off_header) */
typedef struct td_env_header {
    double cost_def;
    double cost_atk;
    double ep_return;
    int32_t base_LP;
    int32_t steps;
    int32_t map_id;
    int32_t episode;
    int16_t defender_cd;
    int16_t attacker_cd;
    uint8_t n_towers;
    uint8_t n_enemies;
    uint8_t flags;              /* bit0 enemy overflow, bit1 tower overflow (sticky) */
    uint8_t pad0;               /* internal: valid words of the record's generator word cache */
    uint16_t ep_kills;          /* kills / leaks of the running episode: low 16 bits ... */
    uint16_t ep_leaks;
    int32_t rng_pos;            /* position in the opponent MT19937 state (0..624) */
    int32_t pad1;               /* internal: consumed words of that cache */
    uint16_t ep_kills_hi;       /* ... and high 16 bits (an episode may last INT_MAX steps; this word was pad2) */
    uint16_t ep_leaks_hi;
} td_env_header;                /* 64 bytes */

typedef struct td_tower_rec {   /* 16 bytes, list order */
    double cd;
    uint16_t loc;
    uint8_t type_lv;            /* type | lv << 2 */
    uint8_t scratch[5];
} td_tower_rec;

typedef struct td_enemy_rec {   /* 24 bytes, list order */
    double LP;
    double margin;
    uint16_t loc;
    uint8_t type_lv;            /* type | lv << 2 */
    uint8_t slowdown;
    uint8_t scratch[4];
} td_enemy_rec;

/* episode statistics, summed over the handle's envs (deterministic reduction on device) */
typedef struct td_stats {
    double return_sum;
    int64_t episodes;
    int64_t length_sum;
    int64_t wins;               /* from the env's own perspective (2P: defender) */
    int64_t kills;
    int64_t leaks;
    int64_t overflow_envs;      /* envs whose tower/enemy capacity overflowed (results invalid) */
    int64_t steps;              /* env-steps executed since creation */
} td_stats;

int td_abi_version(void);
const char *td_last_error(const td_handle *h);
void td_default_config(td_config *cfg);
/* host-only: the first step count s with (double)s / max_episode_steps >= enemy_upgrade_at, from which summoned
 * enemies are level 1 (also past the end of an episode); 0x7fffffff when no smaller count reaches it (NaN, huge) */
int td_upgrade_step(int max_episode_steps, double enemy_upgrade_at);

/* host-only: reference-order road generator on a NumPy-legacy MT19937 stream.
 * num_roads <= 0: draw it first from the same stream like TDGymBasic.reset (:42).
 * Returns 1 if the seed is valid, 0 if the reference generator would raise or exceed
 * `budget` randint calls (seed-skip rule), <0 on error. */
int td_mapgen(uint32_t seed, int map_size, int num_roads, int budget, td_map *out);
/* same generator on an explicit stream: state625 = RandomState.get_state() key (624 words) + position,
 * updated in place, so successive resets keep drawing from one stream like self.np_random does. */
int td_mapgen_stream(uint32_t *state625_inout, int map_size, int num_roads, int budget, td_map *out);
/* n seeds in parallel on `threads` host threads; valid_out[i] as above. first-valid search:
 * if skip_invalid != 0, seed i is advanced (s <- s+1) until valid and seeds_inout[i] is updated. */
int td_mapgen_batch(uint32_t *seeds_inout, int n, int map_size, int num_roads, int budget,
                    int skip_invalid, int threads, td_map *out, int32_t *valid_out);

int td_create(const td_config *cfg, int env_kind, int map_size, int n_envs, int device, td_handle **out);
int td_destroy(td_handle *h);
int td_set_config(td_handle *h, const td_config *cfg);
int td_get_layout(const td_handle *h, td_layout *out);

/* replace the device map pool by n_maps host maps */
int td_upload_maps(td_handle *h, const td_map *maps_host, int n_maps);
/* auto-reset schedule: a finished env takes map (map_id + stride) % n_maps */
int td_set_map_stride(td_handle *h, int stride);

/* (re)start envs: mask_dev NULL = all; map_ids_dev NULL = env i takes map i % n_maps.
 * obs_dev may be NULL. */
int td_reset(td_handle *h, const uint8_t *mask_dev, const int32_t *map_ids_dev, float *obs_dev, void *stream);

/* seed the per-env scripted-opponent generators: states_host is [n_envs][625] uint32
 * (624 MT19937 words + position, i.e. random.Random(s).getstate()[1]). */
int td_seed_opponent(td_handle *h, const uint32_t *states_host, int first_env, int n);
/* same, from integer seeds: env i gets the state of CPython's random.seed(seeds_host[i]) (0 <= seed < 2^32) */
int td_seed_opponent_python(td_handle *h, const uint32_t *seeds_host, int first_env, int n);
/* scripted opponent level (difficulty kwarg of TDDefense/TDAttack); default 1 */
int td_set_difficulty(td_handle *h, int difficulty);

int td_step(td_handle *h, const td_step_io *io, void *stream);
/* obs_incremental bookkeeping: the library remembers the ADDRESS of the buffer it filled last.  If that memory was
 * freed and re-allocated, or written by anybody else, call this before the next step: it then writes all planes. */
int td_invalidate_obs(td_handle *h);
/* observation of the current state only (kernel (f) alone) */
int td_observe(td_handle *h, float *obs_dev, void *stream);
/* the same in a reduced-precision element type (TD_OBS_BF16 / TD_OBS_U8; TD_OBS_F32 = td_observe) */
int td_observe_as(td_handle *h, int obs_format, void *obs_dev, void *stream);

/* Action masks of the current state (new; the reference has none): which actions the NEXT td_step / td_step_host
 * would carry out.  The state is the one in the env records -- after the last td_step (including its auto-resets),
 * td_reset or td_set_state -- i.e. the one the current observation shows.  A separate kernel; the step is unchanged.
 *
 * def_mask_dev (TD_KIND_DEF, TD_KIND_2P): [n_envs, 6*L*L + 1] uint8, any alignment.  Entry a is 1 exactly when the
 *   Discrete action a given to the next step comes back with RealAction == a.  So the no-op 6*L*L is always 1, and
 *   every other entry is 0 unless the defender may act: defender_cd <= 1 in the header (AllowNextMove bit 0; the step
 *   lowers the cooldown by one before the defender acts).  When it may act, with cost_def the header's purse:
 *     build type t on loc (a = t*L*L + loc, t < 4):  !(cost_def < tower_cost[t][0]) && map6[loc] == 0
 *                                                    && n_towers < TD_CAP_TOWERS
 *     LvUp on loc (a = 4*L*L + loc):                 a tower stands on loc, its level lv is below max_tower_lv
 *                                                    && !(cost_def < tower_cost[type][lv + 1])
 *     Destruct on loc (a = 5*L*L + loc):             a tower stands on loc
 *   (the comparisons are the step's own, so NaN and infinite purses and prices agree with it).  The first 6*L*L
 *   entries are the channel-major (6, L, L) layout of the multi-action Box: with multi_action, entry (ch, r, c) is 1
 *   exactly when a Box action whose only flag is (ch, r, c) succeeds (real_def[ch, r, c] == 1).
 * atk_mask_dev (TD_KIND_ATK, TD_KIND_2P): [n_envs, 3, 4] uint8.  Entry (r, t) is 1 exactly when the next step, given a
 *   cluster whose only non-empty slot is type t on road r, summons that enemy: attacker_cd <= 1 (AllowNextMove bit 1),
 *   r < num_roads, and the purse affords the enemy at level lv = (steps >= the upgrade step of td_upgrade_step):
 *   !(cost_atk < c_min[lv]) && !(cost_atk < enemy_cost[t][lv]), c_min[lv] = the cheapest enemy_cost[.][lv] (the step
 *   tests the cheapest type first).  A per-slot mask: later slots of one cluster see a smaller purse.  A cluster
 *   that would exceed the enemy capacity (an error the statistics report as overflow_envs) is not modelled.
 * In the defender env (TD-def) the defender acts first; in TD-2p the attacker acts first, but a summon changes only
 * cost_atk and the enemy list, which no defender entry depends on.  Either pointer may be NULL, not both; the mask
 * of a scripted side (atk mask of TD-def, defender mask of TD-atk) is TD_E_INVALID. */
int td_action_mask(td_handle *h, uint8_t *def_mask_dev, uint8_t *atk_mask_dev, void *stream);

/* Host-buffer variant (the gym-facing call): copies the actions host->device, steps, copies
 * the small outputs (and the observation if obs_host != NULL) device->host, and synchronises.
 * The *_dev members of io are used as the device staging buffers; host pointers should be pinned. */
typedef struct td_host_io {
    const int64_t *def_action_host;
    const int64_t *atk_action_host;
    const uint8_t *opponent_host;
    float *obs_host;
    double *reward_host;
    uint8_t *done_host;
    int8_t *win_host;
    uint8_t *allow_next_host;
    int64_t *real_def_host;
    int64_t *real_atk_host;
    int32_t *fail_def_host;
    int32_t *fail_atk_host;
    const uint32_t *opponent_cluster_host;   /* ABI 3: host side of td_step_io.opponent_cluster_dev */
    void *packed_host;               /* ABI 3: page-locked [n] td_step_packed records.  The step kernel writes them
                                        directly (zero-copy); leave the per-field host pointers above NULL and
                                        td_step_host issues no device->host copy at all. */
} td_host_io;
int td_step_host(td_handle *h, const td_step_io *io, const td_host_io *host, void *stream);
/* td_step_host runs as ONE CUDA-graph launch per call (copies in, the step kernels of 1..n chunks of the batch,
 * copies out), cached per distinct set of buffers; with pageable host memory, or TD_OPT_HOST_GRAPH = 0, the same
 * operations are issued on the stream one by one.  Large batches are cut automatically: the chunk kernels are
 * independent branches of the graph, each starts as soon as its own actions have arrived (the first chunk is short),
 * so the action copy hides behind the step.  Small actions are not copied at all: the step kernel reads them from
 * the page-locked host buffer (TD_OPT_HOST_ZERO_COPY), and io->def_action_dev / atk_action_dev, which only stage
 * the copy, are then left untouched.  Buffers of a cached graph must stay allocated (and page-locked) while the
 * handle lives.  Passing the legacy default stream (NULL) is fine. */

/* tuning knobs of a handle (no environment variables are read anywhere in the library) */
enum { TD_OPT_HOST_CHUNKS = 1,   /* td_step_host: chunks the batch is cut into; 0 = automatic (4 from 8,192 envs on) */
       TD_OPT_HOST_GRAPH = 2,    /* td_step_host: 1 = graph launch (default), 0 = plain stream launches */
       /* 3 and 4 are retired (former shared-memory experiments) and rejected; do not reuse them */
       TD_OPT_GENERIC_KERNELS = 5, /* 1 = never pick the step kernels specialised on the default scripted opponent
                                    (level 1 on the device generator); results are identical, for A/B runs and tests */
       TD_OPT_HOST_CHAIN = 6,    /* td_step_host graph with > 1 chunk: 0 = independent branches, each starts when its own
                                    actions have arrived (default), 1 = chunk kernels run one after the other */
       TD_OPT_HOST_FIRST_CHUNK = 7 }; /* td_step_host with > 1 chunk: F > 0 = chunks of F, 3F, 9F, ... envs (the last takes the
                                    rest), 0 = equal chunks, -1 = automatic (n/16 unless the copy is >= 8 MB) */
enum { TD_OPT_HOST_ZERO_COPY = 8 }; /* td_step_host inputs the step kernel reads straight from the caller's page-locked
                                    buffer instead of a copy in front of it: -1 = automatic (3 x action bytes per env <=
                                    cells: Discrete actions always, the (3, 8) attacker action on 30x30 boards),
                                    0 = never, 1 = every action */
int td_set_option(td_handle *h, int option, int value);

/* raw env records (td_layout) to/from host; blob is n * record_bytes */
int td_get_state(td_handle *h, int first_env, int n, void *blob_host);
int td_set_state(td_handle *h, int first_env, int n, const void *blob_host);
/* opponent generator states, [n][625] */
int td_get_opponent(td_handle *h, int first_env, int n, uint32_t *states_host);

int td_get_stats(td_handle *h, td_stats *out, void *stream);
int td_reset_stats(td_handle *h, void *stream);

/* ---- compact observations (SURVEY.md 8(f) f4): an env record (td_layout.record_bytes, ~2.5 KB at L=10) holds
 * everything the 18 KB float32 observation is a function of, including the static map.  A learner can keep
 * records instead of observations and rebuild any of them on demand:
 * td_snapshot          copies the n_envs current records to caller memory ([n_envs, record_bytes] bytes, device)
 * td_observe_snapshot  builds the (45, L, L) float32 observations of `n` stored records (kernel (f) alone,
 *                      TDBoard.get_states, gym_TD/envs/TDBoard.py:85-144) */
int td_snapshot(td_handle *h, void *records_out_dev, void *stream);
int td_observe_snapshot(td_handle *h, const void *records_dev, int n, float *obs_dev, void *stream);

/* ---- rollout consumer (SURVEY.md 8(f) f1): the per-step bookkeeping of the reference's training loop ----
 * td_rollout_mask    <- train/main.py:130-132       actions of envs that may not move become empty_action()
 * td_rollout_record  <- train/PPO/Callbacks.py:21-23 + train/PPO/Model.py:134-140
 *                       reward -= penalty when action != RealAction; row t of [horizon, n] buffers
 * td_gae             <- train/PPO/Model.py:166-192   GAE(gamma, lam) advantages and returns over one horizon
 * `which`: 0 = defender Discrete action ([n] int64, empty = 6*L*L), 1 = attacker cluster ([n,3,8], empty = 4).
 * All pointers are device pointers; buffers are [horizon, n(, width)] with the env index fastest. */
int td_rollout_mask(td_handle *h, int which, int64_t *action_dev, const uint8_t *allow_next_dev, void *stream);
int td_rollout_record(td_handle *h, int which, const int64_t *action_dev, const int64_t *real_action_dev,
                      const double *reward_dev, const uint8_t *done_dev, double penalty,
                      float *rewards_row_dev, uint8_t *dones_row_dev, int64_t *actions_row_dev, void *stream);
int td_gae(int horizon, int n, const float *rewards_dev, const uint8_t *dones_dev, const float *values_dev,
           const float *next_value_dev, double gamma, double lam, float *advs_dev, float *returns_dev, void *stream);
/* td_gae takes no handle: it runs on the device that owns rewards_dev (made current for the calling thread). */

/* ---- observation memory (new; no counterpart in the reference) ------------------------------------------------
 * Device memory for the observation tensor from a COMPRESSIBLE allocation (CUDA virtual memory management,
 * CU_MEM_ALLOCATION_COMP_GENERIC): B200 compresses lines in L2 on their way to HBM, losslessly and transparently to
 * every reader and writer.  60 % of an observation is zeros and 27 % are planes that broadcast one scalar, so the
 * step that writes it and the learner that reads it both move fewer HBM bytes (DESIGN.md section 7.2h).  The buffer
 * is zero-filled.  *compressed_out (optional) tells whether the driver granted compression; when the device does not
 * support it the call fails with TD_E_STATE and the caller allocates ordinary memory.  Any device pointer works as
 * td_step_io.obs_dev -- this is an allocator, not a requirement. */
int td_alloc_compressible(int device, size_t bytes, void **ptr_out, int *compressed_out);
int td_free_compressible(void *ptr);

#ifdef __cplusplus
}
#endif
#endif
