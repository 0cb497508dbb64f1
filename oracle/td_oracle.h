/*
 * td_oracle.h -- CPU restatement (plain C) of the gym-TD board step.
 *
 * TEST INFRASTRUCTURE ONLY.  This is the parity oracle for the CUDA product in
 * gym_td_b200/csrc.  Only tests/, __graft_entry__.smoke() and bench.py's
 * cpu_baseline / --impl reference legs may load it; the product never does.
 *
 * Parity status: PINNED.  The restatement is checked against
 *   (1) the reference's own golden vector (TDBoard.py:674-756: map + t=0 obs),
 *   (2) the reference itself executed in the build container (oracle/validate_oracle.py,
 *       tests/test_oracle_vs_reference.py), and
 *   (3) golden trajectories generated from the reference and committed under
 *       tests/golden/ (oracle/make_golden.py), which also travel to the GPU box.
 *
 * Every function cites the reference file:line it follows (paths relative to the
 * reference root, e.g. gym_TD/envs/TDBoard.py).
 */
#ifndef TD_ORACLE_H
#define TD_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TDO_MAX_L 64
#define TDO_MAX_CELLS (TDO_MAX_L * TDO_MAX_L)
#define TDO_CAP_TOWERS 1024
#define TDO_CAP_ENEMIES 2048
#define TDO_NTYPES 4   /* enemy_types == tower_types == 4 (TDParam.py:6-7) */
#define TDO_NLV 2      /* max_*_lv == 1 -> two levels (TDParam.py:3-4) */
#define TDO_CLUSTER 8  /* max_cluster_length (TDParam.py:110) */
#define TDO_ROADS 3    /* max_num_of_roads (TDParam.py:111) */

/* gym_TD/utils/fail_code.py:1-6 */
enum { TDO_SUCCESS = 0, TDO_COST_SHORTAGE = 1, TDO_INVALID_POSITION = 2,
       TDO_LV_MAX = 3, TDO_UNKNOWN_TARGET = 4, TDO_IMPOSSIBLE_CLUSTER = 5 };

/* gym_TD/envs/TDParam.py:1-94 (config) and :105-111 (hyper_parameters) */
typedef struct tdo_config {
    double enemy_LP[TDO_NTYPES][TDO_NLV];
    double enemy_speed[TDO_NTYPES][TDO_NLV];
    double enemy_defense[TDO_NTYPES][TDO_NLV];
    double enemy_cost[TDO_NTYPES][TDO_NLV];
    double tower_attack[TDO_NTYPES][TDO_NLV];
    double tower_cost[TDO_NTYPES][TDO_NLV];
    double tower_attack_interval[TDO_NTYPES][TDO_NLV];
    int32_t tower_range[TDO_NTYPES][TDO_NLV];
    int32_t tower_splash_range[TDO_NTYPES][TDO_NLV];
    double tower_destruct_return;
    double frozen_ratio;
    double attacker_init_cost, defender_init_cost, max_cost;
    double reward_kill, penalty_leak, reward_time;
    double attacker_cost_init_rate, attacker_cost_final_rate, defender_cost_rate;
    double enemy_upgrade_at;
    int32_t frozen_time;
    int32_t base_LP;            /* < 0 means None */
    int32_t tower_distance;
    int32_t attacker_action_interval, defender_action_interval;
    int32_t max_episode_steps;
    int32_t max_tower_lv;
    int32_t pad_;
} tdo_config;

typedef struct tdo_enemy {   /* TDElements.py:4-14 */
    double maxLP, LP, speed, defense, cost, margin;
    int32_t loc;             /* r*L + c */
    int32_t dist;
    int32_t slowdown;
    int32_t type;
    int32_t uid;             /* identity (Python object identity) */
    int32_t hit;             /* scratch */
} tdo_enemy;

typedef struct tdo_tower {   /* TDElements.py:45-55 */
    double atk, intv, cost, cd;
    int32_t rge, dmgrge;
    int32_t loc, lv, type, pad_;
} tdo_tower;

/* MT19937 word generator; used both as CPython `random.Random` and as NumPy legacy RandomState */
typedef struct tdo_mt {
    uint32_t mt[624];
    int32_t pos;
    int32_t pad_;
} tdo_mt;

typedef struct tdo_env {
    tdo_config cfg;
    int32_t L, num_roads;
    int32_t start[TDO_ROADS];
    int32_t end;
    /* map[0..3] road bits, map[4] dist, map[5] dir, map[6] towers nearby (TDBoard.py:31-59) */
    uint8_t road[TDO_MAX_CELLS];
    int32_t dist[TDO_MAX_CELLS];
    int32_t dir[TDO_MAX_CELLS];
    int32_t map6[TDO_MAX_CELLS];
    double cost_def, cost_atk, max_cost, progress;
    int32_t base_LP, max_base_LP, has_base_LP;
    int32_t steps, fail_code;
    int32_t attacker_cd, defender_cd;
    int32_t n_towers, n_enemies, next_uid;
    tdo_tower towers[TDO_CAP_TOWERS];
    tdo_enemy enemies[TDO_CAP_ENEMIES];
    float enemy_LP[4][TDO_NTYPES][TDO_MAX_CELLS]; /* TDBoard.py:63 */
    tdo_mt pyrand;   /* the global `random` module stream */
    tdo_mt nprand;   /* self.np_random */
    /* per-step counters (not in the reference; for statistics parity) */
    int32_t last_kills, last_leaks;
    /* longest tower / enemy list since the caller last set these (not in the reference; for the capacity tests) */
    int32_t peak_towers, peak_enemies;
} tdo_env;

/* outputs of one env-wrapper step: (obs,) reward, done, info */
typedef struct tdo_step_out {
    double reward;
    int32_t done;
    int32_t win;                 /* -1 None, 0 False, 1 True (defender view for TDMulti) */
    int32_t win_attacker;        /* TDMulti only */
    int32_t allow_next_def, allow_next_atk;
    int64_t real_def;            /* Discrete RealAction (defender) */
    int32_t fail_def;
    int32_t n_fail_atk;
    int32_t fail_atk[TDO_ROADS];
    int32_t real_is_def_only;    /* TDMulti.py:114 quirk: dict replaced by int */
    int64_t real_atk[TDO_ROADS][TDO_CLUSTER];
} tdo_step_out;

unsigned tdo_sizeof_env(void);
unsigned tdo_sizeof_config(void);
void tdo_default_config(tdo_config *c);

/* board construction from an already generated road list (TDBoard.py:14-79) */
void tdo_board_init(tdo_env *e, const tdo_config *cfg, int L, int num_roads,
                    const int32_t *road_cells, const int32_t *road_len);
/* same, but from packed planes (road bits, dist, dir) */
void tdo_board_init_planes(tdo_env *e, const tdo_config *cfg, int L, int num_roads,
                           const int32_t *start, int end, const uint8_t *road,
                           const int32_t *dist, const int32_t *dir);

int tdo_tower_build(tdo_env *e, int t, int loc);
int tdo_tower_lvup(tdo_env *e, int loc);
int tdo_tower_destruct(tdo_env *e, int loc);
int tdo_summon_enemy(tdo_env *e, int t, int start_id);
int tdo_summon_cluster(tdo_env *e, const int64_t *types, int start_id, int64_t *real_act);
double tdo_board_step(tdo_env *e);
void tdo_enemy_stats(tdo_env *e);   /* the enemy-statistics planes of the current lists (end of tdo_board_step) */
int tdo_done(const tdo_env *e);
void tdo_get_states(const tdo_env *e, float *out);
int tdo_n_channels(void);

/* scripted opponents (TDGymBasic.py:81-292); use_np selects self.np_random over `random` */
void tdo_random_enemy_lv0(tdo_env *e, int use_np);
void tdo_random_enemy_lv1(tdo_env *e, int use_np);
void tdo_random_tower_lv0(tdo_env *e, int use_np);
void tdo_random_tower_lv1(tdo_env *e, int use_np);
void tdo_random_tower_lv2(tdo_env *e, int use_np);

/* env wrappers.  opp: -1 = no scripted opponent call (caller injects it), else difficulty. */
void tdo_def_step(tdo_env *e, int64_t action, int difficulty, int use_np, tdo_step_out *o);
void tdo_def_step_multi(tdo_env *e, const int64_t *action, int64_t *real_act, int difficulty,
                        int use_np, tdo_step_out *o);
void tdo_atk_step(tdo_env *e, const int64_t *action, int difficulty, int use_np, tdo_step_out *o);
void tdo_multi_step(tdo_env *e, const int64_t *atk_action, int64_t def_action, tdo_step_out *o);
void tdo_multi_step_multi(tdo_env *e, const int64_t *atk_action, const int64_t *def_action,
                          int64_t *real_def, tdo_step_out *o);

/* cpu_baseline "port" leg: run n env-steps of TDDefense (Discrete, uniform random actions from a
 * xorshift stream, scripted attacker lv1 on e->pyrand), building the observation every step and
 * restarting the episode on the same map when done.  Returns a checksum so the work is not elided. */
double tdo_bench_def(tdo_env *e, int n_steps, uint64_t action_seed, float *obs_buf);

/* RNG helpers (exposed for tests) */
void tdo_mt_set(tdo_mt *m, const uint32_t *key624, int pos);
void tdo_mt_seed_numpy(tdo_mt *m, uint32_t seed);             /* RandomState(seed) */
void tdo_mt_seed_python(tdo_mt *m, uint32_t seed);            /* random.seed(int) (seed < 2^32) */
uint32_t tdo_mt_next(tdo_mt *m);
uint32_t tdo_py_randbelow(tdo_mt *m, uint32_t n);
double tdo_py_random(tdo_mt *m);
int64_t tdo_np_randint(tdo_mt *m, int64_t low, int64_t high); /* legacy RandomState.randint(low, high) */

#ifdef __cplusplus
}
#endif
#endif
