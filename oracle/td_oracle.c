/*
 * td_oracle.c -- CPU restatement (plain C) of the gym-TD board step.
 * TEST INFRASTRUCTURE ONLY; see td_oracle.h for the parity status ("pinned").
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math -shared -fPIC (oracle/Makefile).
 * All f64 arithmetic follows the reference's Python evaluation order with one
 * rounding per operation (never fused).
 */
#include "td_oracle.h"
#include <string.h>
#include <math.h>
#include <stdlib.h>

unsigned tdo_sizeof_env(void) { return (unsigned)sizeof(tdo_env); }
unsigned tdo_sizeof_config(void) { return (unsigned)sizeof(tdo_config); }
int tdo_n_channels(void) { return 15 + 2 * TDO_NTYPES + 1 + 1 + 5 * TDO_NTYPES; } /* TDBoard.py:154 */

/* gym_TD/envs/TDParam.py:1-94 */
void tdo_default_config(tdo_config *c)
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
    for (int t = 0; t < 4; ++t)
        for (int l = 0; l < 2; ++l) {
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
    c->max_episode_steps = 1200; /* TDParam.py:107 */
    c->max_tower_lv = 1;
}

/* ------------------------------------------------------------------ RNG */

static void mt_init_genrand(tdo_mt *m, uint32_t s)
{
    m->mt[0] = s;
    for (int i = 1; i < 624; ++i)
        m->mt[i] = 1812433253u * (m->mt[i - 1] ^ (m->mt[i - 1] >> 30)) + (uint32_t)i;
    m->pos = 624;
}

void tdo_mt_set(tdo_mt *m, const uint32_t *key624, int pos)
{
    memcpy(m->mt, key624, sizeof(m->mt));
    m->pos = pos;
}

/* numpy legacy RandomState(int seed): mt19937_seed == init_genrand */
void tdo_mt_seed_numpy(tdo_mt *m, uint32_t seed) { mt_init_genrand(m, seed); }

/* CPython random.seed(int): init_by_array([seed]) for 0 <= seed < 2^32 */
void tdo_mt_seed_python(tdo_mt *m, uint32_t seed)
{
    uint32_t key[1] = {seed};
    int i = 1, j = 0, k;
    mt_init_genrand(m, 19650218u);
    for (k = 624; k; --k) {
        m->mt[i] = (m->mt[i] ^ ((m->mt[i - 1] ^ (m->mt[i - 1] >> 30)) * 1664525u)) + key[j] + (uint32_t)j;
        ++i; ++j;
        if (i >= 624) { m->mt[0] = m->mt[623]; i = 1; }
        if (j >= 1) j = 0;
    }
    for (k = 623; k; --k) {
        m->mt[i] = (m->mt[i] ^ ((m->mt[i - 1] ^ (m->mt[i - 1] >> 30)) * 1566083941u)) - (uint32_t)i;
        ++i;
        if (i >= 624) { m->mt[0] = m->mt[623]; i = 1; }
    }
    m->mt[0] = 0x80000000u;
    m->pos = 624;
}

uint32_t tdo_mt_next(tdo_mt *m)
{
    uint32_t y;
    if (m->pos >= 624) {
        int kk;
        uint32_t *mt = m->mt;
        for (kk = 0; kk < 624 - 397; ++kk) {
            y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu);
            mt[kk] = mt[kk + 397] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        for (; kk < 623; ++kk) {
            y = (mt[kk] & 0x80000000u) | (mt[kk + 1] & 0x7fffffffu);
            mt[kk] = mt[kk + (397 - 624)] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        y = (mt[623] & 0x80000000u) | (mt[0] & 0x7fffffffu);
        mt[623] = mt[396] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        m->pos = 0;
    }
    y = m->mt[m->pos++];
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
}

static int bit_length(uint32_t n) { int k = 0; while (n) { ++k; n >>= 1; } return k; }

/* CPython Lib/random.py _randbelow_with_getrandbits; getrandbits(k<=32) = word >> (32-k) */
uint32_t tdo_py_randbelow(tdo_mt *m, uint32_t n)
{
    int k = bit_length(n);
    uint32_t r = tdo_mt_next(m) >> (32 - k);
    while (r >= n) r = tdo_mt_next(m) >> (32 - k);
    return r;
}
static int py_randint(tdo_mt *m, int a, int b) { return a + (int)tdo_py_randbelow(m, (uint32_t)(b - a + 1)); }

/* random.random() and RandomState.random_sample(): 53-bit double from two words */
double tdo_py_random(tdo_mt *m)
{
    uint32_t a = tdo_mt_next(m) >> 5, b = tdo_mt_next(m) >> 6;
    return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0);
}

/* legacy masked rejection (numpy/random/src/distributions: bounded_masked_uint32) */
static uint32_t np_interval(tdo_mt *m, uint32_t max)
{
    uint32_t mask = max, v;
    if (max == 0) return 0;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    while ((v = (tdo_mt_next(m) & mask)) > max) ;
    return v;
}
int64_t tdo_np_randint(tdo_mt *m, int64_t low, int64_t high)
{
    return low + (int64_t)np_interval(m, (uint32_t)(high - 1 - low));
}

/* ------------------------------------------------------------------ board */

static void board_common_init(tdo_env *e, const tdo_config *cfg, int L, int num_roads)
{
    /* keep RNG streams: the caller seeds them before or after */
    tdo_mt py = e->pyrand, np = e->nprand;
    memset(e, 0, sizeof(*e));
    e->pyrand = py; e->nprand = np;
    e->cfg = *cfg;
    e->L = L;
    e->num_roads = num_roads;
    /* TDBoard.py:66-79 with the arguments of TDGymBasic.py:43-51 */
    e->cost_def = cfg->defender_init_cost;
    e->cost_atk = cfg->attacker_init_cost;
    e->max_cost = cfg->max_cost;
    e->has_base_LP = cfg->base_LP >= 0;
    e->base_LP = cfg->base_LP;
    e->max_base_LP = cfg->base_LP;
    e->steps = 0;
    e->progress = 0.;
    e->fail_code = TDO_SUCCESS;
    e->attacker_cd = 0; /* TDGymBasic.py:52-53 */
    e->defender_cd = 0;
}

/* TDBoard.py:35-59: roads are lists of cells from start to end */
void tdo_board_init(tdo_env *e, const tdo_config *cfg, int L, int num_roads,
                    const int32_t *road_cells, const int32_t *road_len)
{
    board_common_init(e, cfg, L, num_roads);
    const int32_t *p = road_cells;
    for (int i = 0; i < num_roads; ++i) {
        int n = road_len[i];
        e->start[i] = p[0];
        if (i == 0) e->end = p[n - 1];
        for (int k = 0; k < n; ++k) {
            int c = p[k];
            e->road[c] |= (uint8_t)(1u | (2u << i)); /* map[0] and map[i+1] */
            e->map6[c] = 1;
            if (k > 0) {
                int last = p[k - 1];
                int dr = c / L - last / L, dc = c % L - last % L, d;
                if (dr == 0) d = (dc == 1) ? 0 : 1;
                else if (dr == 1) d = 2;
                else d = 3;
                e->dir[last] = d;
            }
        }
        for (int k = n - 1, dist = 0; k >= 0; --k, ++dist) e->dist[p[k]] = dist;
        p += n;
    }
}

void tdo_board_init_planes(tdo_env *e, const tdo_config *cfg, int L, int num_roads,
                           const int32_t *start, int end, const uint8_t *road,
                           const int32_t *dist, const int32_t *dir)
{
    board_common_init(e, cfg, L, num_roads);
    for (int i = 0; i < num_roads; ++i) e->start[i] = start[i];
    e->end = end;
    for (int c = 0; c < L * L; ++c) {
        e->road[c] = road[c];
        e->dist[c] = dist[c];
        e->dir[c] = dir[c];
        e->map6[c] = (road[c] & 1) ? 1 : 0;
    }
}

/* TDElements.py:33-43 */
static void create_enemy(const tdo_env *e, tdo_enemy *en, int t, int loc, int dist, int lv)
{
    en->maxLP = en->LP = e->cfg.enemy_LP[t][lv];
    en->speed = e->cfg.enemy_speed[t][lv];
    en->defense = e->cfg.enemy_defense[t][lv];
    en->cost = e->cfg.enemy_cost[t][lv];
    en->loc = loc;
    en->margin = 0.;
    en->dist = dist;
    en->slowdown = 0;
    en->type = t;
    en->hit = 0;
}

/* TDBoard.py:184-197 */
int tdo_summon_enemy(tdo_env *e, int t, int start_id)
{
    int start = e->start[start_id];
    int lv = e->progress >= e->cfg.enemy_upgrade_at ? 1 : 0;
    tdo_enemy en;
    create_enemy(e, &en, t, start, e->dist[start], lv);
    if (e->cost_atk < en.cost) { e->fail_code = TDO_COST_SHORTAGE; return 0; }
    en.uid = e->next_uid++;
    e->enemies[e->n_enemies++] = en;
    if (e->n_enemies > e->peak_enemies) e->peak_enemies = e->n_enemies;
    e->cost_atk -= en.cost;
    e->fail_code = TDO_SUCCESS;
    return 1;
}

/* TDBoard.py:199-224.  Returns the first element of the (bool, real_act) tuple. */
int tdo_summon_cluster(tdo_env *e, const int64_t *types, int start_id, int64_t *real_act)
{
    int start = e->start[start_id];
    int lv = e->progress >= e->cfg.enemy_upgrade_at ? 1 : 0;
    int tried = 0, summoned = 0;
    for (int k = 0; k < TDO_CLUSTER; ++k) {
        int64_t t = types[k];
        if (t == TDO_NTYPES) { if (real_act) real_act[k] = t; continue; }
        tried = 1;
        tdo_enemy en;
        create_enemy(e, &en, (int)t, start, e->dist[start], lv);
        if (e->cost_atk < en.cost) {
            if (real_act) real_act[k] = TDO_NTYPES;
        } else {
            e->cost_atk -= en.cost;
            en.uid = e->next_uid++;
            e->enemies[e->n_enemies++] = en;
            if (e->n_enemies > e->peak_enemies) e->peak_enemies = e->n_enemies;
            summoned = 1;
            if (real_act) real_act[k] = t;
        }
    }
    if (!summoned && tried) { e->fail_code = TDO_COST_SHORTAGE; return 0; }
    e->fail_code = TDO_SUCCESS;
    return 1;
}

static void diamond_add(tdo_env *e, int loc, int delta)
{
    int L = e->L, D = e->cfg.tower_distance, r0 = loc / L, c0 = loc % L;
    for (int i = -D; i <= D; ++i)
        for (int j = -D; j <= D; ++j)
            if (abs(i) + abs(j) <= D) {
                int r = r0 + i, c = c0 + j;
                if (r < 0 || r >= L || c < 0 || c >= L) continue;
                e->map6[r * L + c] += delta;
            }
}

/* TDBoard.py:226-247 + TDElements.py:134-150 */
int tdo_tower_build(tdo_env *e, int t, int loc)
{
    tdo_tower p;
    p.atk = e->cfg.tower_attack[t][0];
    p.rge = e->cfg.tower_range[t][0];
    p.dmgrge = e->cfg.tower_splash_range[t][0];
    p.intv = e->cfg.tower_attack_interval[t][0];
    p.loc = loc;
    p.cost = e->cfg.tower_cost[t][0];
    p.type = t; p.lv = 0; p.cd = 0; p.pad_ = 0;
    if (e->cost_def < p.cost) { e->fail_code = TDO_COST_SHORTAGE; return 0; }
    if (e->map6[loc] > 0) { e->fail_code = TDO_INVALID_POSITION; return 0; }
    e->towers[e->n_towers++] = p;
    if (e->n_towers > e->peak_towers) e->peak_towers = e->n_towers;
    e->cost_def -= p.cost;
    diamond_add(e, loc, +1);
    e->fail_code = TDO_SUCCESS;
    return 1;
}

/* TDBoard.py:249-271 + TDElements.py:152-170 (argument swap: intv <- tower_cost, cost += interval) */
int tdo_tower_lvup(tdo_env *e, int loc)
{
    for (int i = 0; i < e->n_towers; ++i) {
        tdo_tower *t = &e->towers[i];
        if (t->loc != loc) continue;
        if (t->lv >= e->cfg.max_tower_lv) { e->fail_code = TDO_LV_MAX; return 0; }
        double cost = e->cfg.tower_cost[t->type][t->lv + 1];
        if (e->cost_def < cost) { e->fail_code = TDO_COST_SHORTAGE; return 0; }
        int l = t->lv + 1, ty = t->type;
        t->lv += 1;
        t->atk = e->cfg.tower_attack[ty][l];
        t->rge = e->cfg.tower_range[ty][l];
        t->dmgrge = e->cfg.tower_splash_range[ty][l];
        t->intv = e->cfg.tower_cost[ty][l];                 /* sic: TDElements.py:167 vs :57 */
        t->cost += e->cfg.tower_attack_interval[ty][l];     /* sic: TDElements.py:168 vs :63 */
        e->cost_def -= cost;
        e->fail_code = TDO_SUCCESS;
        return 1;
    }
    e->fail_code = TDO_UNKNOWN_TARGET;
    return 0;
}

/* TDBoard.py:273-293 */
int tdo_tower_destruct(tdo_env *e, int loc)
{
    for (int i = 0; i < e->n_towers; ++i) {
        tdo_tower *t = &e->towers[i];
        if (t->loc != loc) continue;
        e->cost_def += t->cost * e->cfg.tower_destruct_return;
        e->cost_def = e->max_cost < e->cost_def ? e->max_cost : e->cost_def; /* min(cost_def, max_cost) */
        memmove(&e->towers[i], &e->towers[i + 1], sizeof(tdo_tower) * (size_t)(e->n_towers - i - 1));
        e->n_towers--;
        diamond_add(e, loc, -1);
        e->fail_code = TDO_SUCCESS;
        return 1;
    }
    e->fail_code = TDO_UNKNOWN_TARGET;
    return 0;
}

/* TDElements.py:67-69 (Chebyshev) */
static int cheb(int a, int b, int L)
{
    int dr = abs(a / L - b / L), dc = abs(a % L - b % L);
    return dr > dc ? dr : dc;
}

/* TDElements.py:19-28 */
static void enemy_damage(tdo_enemy *en, double atk, int magic)
{
    double dmg;
    if (magic) dmg = atk;
    else { dmg = atk - en->defense; if (!(dmg > 0)) dmg = 0; } /* max(atk - defense, 0) */
    double floor_ = atk * .05;
    if (dmg < floor_) dmg = floor_;
    en->LP -= dmg;
    if (en->LP <= 0) en->LP = 0;
    en->hit = 1;
}

/* TDBoard.py:355-365: enemy statistics of the current lists, float32 in list order (NumPy 2 / NEP 50 semantics).
 * The last part of tdo_board_step; also callable on its own for a state written field by field. */
void tdo_enemy_stats(tdo_env *e)
{
    const int cells = e->L * e->L;
    for (int t = 0; t < TDO_NTYPES; ++t)
        for (int c = 0; c < cells; ++c) {
            e->enemy_LP[0][t][c] = 1.f;
            e->enemy_LP[1][t][c] = 0.f;
            e->enemy_LP[2][t][c] = 0.f;
            e->enemy_LP[3][t][c] = 0.f;
        }
    for (int i = 0; i < e->n_enemies; ++i) {
        const tdo_enemy *en = &e->enemies[i];
        float r = (float)(en->LP / en->maxLP);
        float *mn = &e->enemy_LP[0][en->type][en->loc], *mx = &e->enemy_LP[1][en->type][en->loc];
        if (r < *mn) *mn = r;
        if (r > *mx) *mx = r;
        e->enemy_LP[2][en->type][en->loc] += r;
        e->enemy_LP[3][en->type][en->loc] += 1.f;
    }
    for (int t = 0; t < TDO_NTYPES; ++t)
        for (int c = 0; c < cells; ++c) {
            float cnt = e->enemy_LP[3][t][c];
            if (!(cnt > 0)) { e->enemy_LP[0][t][c] = 0.f; e->enemy_LP[2][t][c] = 0.f; }
            else e->enemy_LP[2][t][c] = e->enemy_LP[2][t][c] / cnt;
            e->enemy_LP[3][t][c] = cnt / (float)TDO_CLUSTER;
        }
}

/* TDBoard.py:295-368 */
double tdo_board_step(tdo_env *e)
{
    const int L = e->L;
    double reward = 0.;
    reward += e->cfg.reward_time;
    e->steps += 1;
    e->progress = (double)e->steps / (double)e->cfg.max_episode_steps;

    /* :305 stable in-place sort by dist - margin (insertion sort is stable) */
    for (int i = 1; i < e->n_enemies; ++i) {
        tdo_enemy x = e->enemies[i];
        double kx = (double)x.dist - x.margin;
        int j = i - 1;
        while (j >= 0 && ((double)e->enemies[j].dist - e->enemies[j].margin) > kx) {
            e->enemies[j + 1] = e->enemies[j];
            --j;
        }
        e->enemies[j + 1] = x;
    }
    for (int i = 0; i < e->n_enemies; ++i) e->enemies[i].hit = 0;

    /* :306-313 towers in list order; dead enemies stay targetable until :315-317 */
    for (int ti = 0; ti < e->n_towers; ++ti) {
        tdo_tower *t = &e->towers[ti];
        t->cd -= 1;
        if (t->cd > 0) continue;
        int target = -1;
        for (int i = 0; i < e->n_enemies; ++i)
            if (cheb(e->enemies[i].loc, t->loc, L) <= t->rge) { target = i; break; }
        if (target >= 0) {
            t->cd += t->intv;
            switch (t->type) {
            case 0: enemy_damage(&e->enemies[target], t->atk, 0); break;     /* TDElements.py:72-81 */
            case 1: enemy_damage(&e->enemies[target], t->atk, 1); break;     /* :83-93 */
            case 2:                                                           /* :95-110 */
                for (int i = 0; i < e->n_enemies; ++i)
                    if (cheb(e->enemies[target].loc, e->enemies[i].loc, L) <= t->dmgrge)
                        enemy_damage(&e->enemies[i], t->atk, 0);
                break;
            default:                                                          /* :112-132 */
                for (int i = 0; i < e->n_enemies; ++i)
                    if (cheb(e->enemies[target].loc, e->enemies[i].loc, L) <= t->dmgrge) {
                        enemy_damage(&e->enemies[i], t->atk, 1);
                        e->enemies[i].slowdown = e->cfg.frozen_time;
                        break;
                    }
                break;
            }
        }
        if (t->cd < 0) t->cd = 0;
    }
    /* :313-317 unique killed = hit this step and not alive */
    int kills = 0, n = 0;
    for (int i = 0; i < e->n_enemies; ++i) {
        if (e->enemies[i].hit && !(e->enemies[i].LP > 0)) { ++kills; continue; }
        e->enemies[n++] = e->enemies[i];
    }
    e->n_enemies = n;
    reward += e->cfg.reward_kill * kills;
    e->last_kills = kills;

    /* :319-346 movement and leakage */
    static const int dpr[4] = {0, 0, 1, -1}, dpc[4] = {1, -1, 0, 0};
    int leaks = 0;
    n = 0;
    for (int i = 0; i < e->n_enemies; ++i) {
        tdo_enemy *en = &e->enemies[i];
        int removed = 0;
        if (en->slowdown > 0) { en->margin += en->speed * e->cfg.frozen_ratio; en->slowdown -= 1; }
        else en->margin += en->speed;
        while (en->margin >= 1.) {
            en->margin -= 1.;
            int d = e->dir[en->loc];
            int r = en->loc / L + dpr[d], c = en->loc % L + dpc[d];
            en->loc = r * L + c;
            en->dist = e->dist[en->loc];
            if (en->loc == e->end) {
                if (e->has_base_LP && e->base_LP > 0) reward -= e->cfg.penalty_leak;
                removed = 1;
                ++leaks;
                if (e->has_base_LP) e->base_LP = e->base_LP - 1 > 0 ? e->base_LP - 1 : 0;
                break;
            }
        }
        if (!removed) e->enemies[n++] = *en;
    }
    e->n_enemies = n;
    e->last_leaks = leaks;

    /* :348-353 economy */
    double rate;
    if (e->progress >= 0.5) rate = e->cfg.attacker_cost_final_rate;
    else {
        double a = e->cfg.attacker_cost_init_rate * (1. - e->progress);
        double b = e->cfg.attacker_cost_final_rate * e->progress;
        rate = a + b;
    }
    double ca = e->cost_atk + rate;
    e->cost_atk = e->max_cost < ca ? e->max_cost : ca;
    double cd = e->cost_def + e->cfg.defender_cost_rate;
    e->cost_def = e->max_cost < cd ? e->max_cost : cd;

    tdo_enemy_stats(e);
    return reward;
}

/* TDBoard.py:370-385 */
int tdo_done(const tdo_env *e)
{
    return (e->has_base_LP && e->base_LP <= 0) || e->steps >= e->cfg.max_episode_steps;
}

/* TDBoard.py:85-144; out is (45, L, L) float32, C-contiguous */
void tdo_get_states(const tdo_env *e, float *s)
{
    const int L = e->L, cells = L * L, C = tdo_n_channels();
    memset(s, 0, sizeof(float) * (size_t)C * (size_t)cells);
#define PLANE(k) (s + (size_t)(k) * (size_t)cells)
    int maxd = 0;
    for (int c = 0; c < cells; ++c) if (e->dist[c] > maxd) maxd = e->dist[c];
    float v5 = e->has_base_LP ? (float)((double)e->base_LP / (double)e->max_base_LP) : 1.f;
    float v11 = (float)(e->cost_def / e->max_cost);
    float v12 = (float)(e->cost_atk / e->max_cost);
    float v13 = (float)e->progress;
    for (int c = 0; c < cells; ++c) {
        for (int k = 0; k < 4; ++k) PLANE(k)[c] = (float)((e->road[c] >> k) & 1);
        PLANE(5)[c] = v5;
        PLANE(9)[c] = (float)e->dist[c] / (float)(maxd + 1);   /* correctly rounded quotient, SURVEY 9.2 */
        PLANE(11)[c] = v11;
        PLANE(12)[c] = v12;
        PLANE(13)[c] = v13;
        PLANE(14)[c] = e->map6[c] == 0 ? 1.f : 0.f;
    }
    PLANE(4)[e->end] = 1.f;
    for (int i = 0; i < e->num_roads; ++i) PLANE(6 + i)[e->start[i]] = 1.f;
    /* channel 10 is never written (TDBoard.py:98 documented, never assigned) */
    const int lv_base = 15, type_base = lv_base + e->cfg.max_tower_lv + 1, build_base = type_base + TDO_NTYPES;
    for (int i = 0; i < e->n_towers; ++i) {
        PLANE(lv_base + e->towers[i].lv)[e->towers[i].loc] = 1.f;
        PLANE(type_base + e->towers[i].type)[e->towers[i].loc] = 1.f;
    }
    const int enemy_base = build_base + TDO_NTYPES, summon_base = enemy_base + 4 * TDO_NTYPES;
    for (int t = 0; t < TDO_NTYPES; ++t) {
        float b = e->cost_def >= e->cfg.tower_cost[t][0] ? 1.f : 0.f;
        float sm = (float)(e->cost_def / e->cfg.enemy_cost[t][0] / (double)TDO_CLUSTER); /* sic: cost_def, :142 */
        for (int c = 0; c < cells; ++c) { PLANE(build_base + t)[c] = b; PLANE(summon_base + t)[c] = sm; }
    }
    for (int k = 0; k < 4; ++k)
        for (int t = 0; t < TDO_NTYPES; ++t)
            memcpy(PLANE(enemy_base + k * TDO_NTYPES + t), e->enemy_LP[k][t], sizeof(float) * (size_t)cells);
#undef PLANE
}

/* ------------------------------------------------------------------ scripted opponents */

static int rnd_int(tdo_env *e, int use_np, int a, int b_inclusive)
{
    /* random.randint(a, b) vs np_random.randint(a, b+1) */
    if (use_np) return (int)tdo_np_randint(&e->nprand, a, (int64_t)b_inclusive + 1);
    return py_randint(&e->pyrand, a, b_inclusive);
}

/* TDGymBasic.py:81-93 */
void tdo_random_enemy_lv0(tdo_env *e, int use_np)
{
    if (e->attacker_cd != 0) return;
    int64_t cluster[TDO_CLUSTER];
    int road;
    if (!use_np) {
        for (int k = 0; k < TDO_CLUSTER; ++k) cluster[k] = py_randint(&e->pyrand, 0, TDO_NTYPES);
        road = py_randint(&e->pyrand, 0, e->num_roads - 1);
    } else {
        for (int k = 0; k < TDO_CLUSTER; ++k) cluster[k] = tdo_np_randint(&e->nprand, 0, TDO_NTYPES);
        road = (int)tdo_np_randint(&e->nprand, 0, e->num_roads);
    }
    tdo_summon_cluster(e, cluster, road, 0);
    e->attacker_cd = e->cfg.attacker_action_interval; /* tuple is always truthy, :90-93 */
}

/* TDGymBasic.py:95-108 */
void tdo_random_enemy_lv1(tdo_env *e, int use_np)
{
    if (e->attacker_cd != 0) return;
    int t = rnd_int(e, use_np, 0, TDO_NTYPES - 1);
    int road = rnd_int(e, use_np, 0, e->num_roads - 1);
    int64_t cluster[TDO_CLUSTER];
    for (int k = 0; k < TDO_CLUSTER; ++k) cluster[k] = t;
    tdo_summon_cluster(e, cluster, road, 0);
    e->attacker_cd = e->cfg.attacker_action_interval; /* tuple is always truthy, :105-108 */
}

/* TDGymBasic.py:111-122 */
void tdo_random_tower_lv0(tdo_env *e, int use_np)
{
    if (e->defender_cd != 0) return;
    int r = rnd_int(e, use_np, 0, e->L - 1);
    int c = rnd_int(e, use_np, 0, e->L - 1);
    int t = rnd_int(e, use_np, 0, TDO_NTYPES - 1);
    if (tdo_tower_build(e, t, r * e->L + c)) e->defender_cd = e->cfg.defender_action_interval;
}

static int collect_road_cells(const tdo_env *e, int *cells_out)
{
    int n = 0;
    for (int c = 0; c < e->L * e->L; ++c) if (e->road[c] & 1) cells_out[n++] = c;
    return n;
}

static void shuffle_cells(tdo_env *e, int use_np, int *x, int n)
{
    for (int i = n - 1; i >= 1; --i) {
        int j = use_np ? (int)np_interval(&e->nprand, (uint32_t)i)
                       : (int)tdo_py_randbelow(&e->pyrand, (uint32_t)(i + 1));
        int tmp = x[i]; x[i] = x[j]; x[j] = tmp;
    }
}

/* shared tail of random_tower_lv1/lv2: walk shuffled road cells, TDGymBasic.py:156-170 / :252-266 */
static void try_build_near_roads(tdo_env *e, int use_np, const int *roads, int n, int t)
{
    const int L = e->L;
    for (int k = 0; k < n; ++k) {
        int di = rnd_int(e, use_np, 0, 24);
        int r = roads[k] / L + (di / 5 - 2), c = roads[k] % L + (di % 5 - 2);
        if (r < 0 || r >= L || c < 0 || c >= L) continue;
        if (tdo_tower_build(e, t, r * L + c)) { e->defender_cd = e->cfg.defender_action_interval; return; }
        if (e->fail_code == TDO_COST_SHORTAGE) return; /* the wait-for-cost memo is dead code (name mangling) */
    }
}

static void lvup_or_destruct(tdo_env *e, int use_np, int act)
{
    if (e->n_towers == 0) return;
    if (act == 2) {
        double p = use_np ? tdo_py_random(&e->nprand) : tdo_py_random(&e->pyrand);
        if (p > .01) return;
    }
    /* note: the reference's np branch of act==2 raises (TDGymBasic.py:191); callers use use_np=0 */
    int id = rnd_int(e, act == 2 ? 0 : use_np, 0, e->n_towers - 1);
    int loc = e->towers[id].loc;
    int ok = act == 1 ? tdo_tower_lvup(e, loc) : tdo_tower_destruct(e, loc);
    if (ok) e->defender_cd = e->cfg.defender_action_interval;
}

/* TDGymBasic.py:124-196 */
void tdo_random_tower_lv1(tdo_env *e, int use_np)
{
    if (e->defender_cd != 0) return;
    int act = rnd_int(e, use_np, 0, 2);
    if (act == 0) {
        int roads[TDO_MAX_CELLS];
        int n = collect_road_cells(e, roads);
        shuffle_cells(e, use_np, roads, n);
        int t = rnd_int(e, use_np, 0, TDO_NTYPES - 1);
        try_build_near_roads(e, use_np, roads, n, t);
    } else lvup_or_destruct(e, use_np, act);
}

/* TDGymBasic.py:198-292 */
void tdo_random_tower_lv2(tdo_env *e, int use_np)
{
    if (e->defender_cd != 0) return;
    int act = rnd_int(e, use_np, 0, 2);
    if (act == 0) {
        if (e->n_enemies == 0) return;
        int nums[TDO_NTYPES] = {0, 0, 0, 0}, types[TDO_NTYPES], nu = 0, total = 0;
        for (int i = 0; i < e->n_enemies; ++i) nums[e->enemies[i].type]++;
        double ratio[TDO_NTYPES];
        for (int t = 0; t < TDO_NTYPES; ++t) total += nums[t];
        for (int t = 0; t < TDO_NTYPES; ++t)
            if (nums[t]) { types[nu] = t; ratio[nu] = (double)(float)nums[t] / (double)total; ++nu; } /* f32 array / np.int64 -> f64 */
        double p = use_np ? tdo_py_random(&e->nprand) : tdo_py_random(&e->pyrand);
        int t = types[nu - 1];
        for (int i = 0; i < nu; ++i) {
            if (p < ratio[i]) { t = types[i]; break; }
            p -= ratio[i];
        }
        static const int counter[4] = {2, 0, 1, 0};
        t = counter[t];
        p = use_np ? tdo_py_random(&e->nprand) : tdo_py_random(&e->pyrand);
        if (p < 0.2) t = 3;
        int roads[TDO_MAX_CELLS];
        int n = collect_road_cells(e, roads);
        shuffle_cells(e, use_np, roads, n);
        try_build_near_roads(e, use_np, roads, n, t);
    } else lvup_or_destruct(e, use_np, act);
}

static void call_enemy_opponent(tdo_env *e, int difficulty, int use_np)
{
    if (difficulty == 0) tdo_random_enemy_lv0(e, use_np);
    else if (difficulty == 1) tdo_random_enemy_lv1(e, use_np);
}
static void call_tower_opponent(tdo_env *e, int difficulty, int use_np)
{
    if (difficulty == 0) tdo_random_tower_lv0(e, use_np);
    else if (difficulty == 1) tdo_random_tower_lv1(e, use_np);
    else if (difficulty == 2) tdo_random_tower_lv2(e, use_np);
}

/* ------------------------------------------------------------------ env wrappers */

static void dec_cds(tdo_env *e)
{
    e->attacker_cd = e->attacker_cd - 1 > 0 ? e->attacker_cd - 1 : 0;
    e->defender_cd = e->defender_cd - 1 > 0 ? e->defender_cd - 1 : 0;
}

static void clear_out(tdo_step_out *o)
{
    memset(o, 0, sizeof(*o));
    o->win = -1;
    o->win_attacker = -1;
}

/* Discrete defender decode shared by TDDefense.py:61-77 and TDMulti.py:100-115 */
static int decode_discrete(tdo_env *e, int64_t action, tdo_step_out *o)
{
    const int L = e->L;
    const int64_t nop = (int64_t)L * L * 6;
    int success = 0;
    o->fail_def = 0;
    o->real_def = nop;
    if (e->defender_cd == 0 && action != nop) {
        int act = (int)(action / ((int64_t)L * L));
        int r = (int)((action / L) % L), c = (int)(action % L);
        int res;
        if (act < TDO_NTYPES) res = tdo_tower_build(e, act, r * L + c);
        else if (act == TDO_NTYPES) res = tdo_tower_lvup(e, r * L + c);
        else res = tdo_tower_destruct(e, r * L + c);
        if (res) { e->defender_cd = e->cfg.defender_action_interval; o->real_def = action; success = 1; }
        o->fail_def = e->fail_code;
    }
    return success;
}

/* multi-action decode shared by TDDefense.py:40-60 and TDMulti.py:65-84; action/real_act are (6, L, L) int64 */
static void decode_multi(tdo_env *e, const int64_t *action, int64_t *real_act)
{
    const int L = e->L, cells = L * L;
    memset(real_act, 0, sizeof(int64_t) * 6 * (size_t)cells);
    if (e->defender_cd != 0) return;
    for (int r = 0; r < L; ++r)
        for (int c = 0; c < L; ++c) {
            int loc = r * L + c;
            for (int t = 0; t < TDO_NTYPES; ++t)
                if (action[(size_t)t * cells + loc] == 1 && tdo_tower_build(e, t, loc)) {
                    e->defender_cd = e->cfg.defender_action_interval;
                    real_act[(size_t)t * cells + loc] = 1;
                }
            if (action[(size_t)4 * cells + loc] == 1 && tdo_tower_lvup(e, loc)) {
                e->defender_cd = e->cfg.defender_action_interval;
                real_act[(size_t)4 * cells + loc] = 1;
            }
            if (action[(size_t)5 * cells + loc] == 1 && tdo_tower_destruct(e, loc)) {
                e->defender_cd = e->cfg.defender_action_interval;
                real_act[(size_t)5 * cells + loc] = 1;
            }
        }
}

static void finish_def(tdo_env *e, tdo_step_out *o)
{
    o->reward = tdo_board_step(e);
    o->done = tdo_done(e);
    if (o->done) {
        o->win = (!e->has_base_LP || e->base_LP > 0) ? 1 : 0;
        o->win_attacker = (!e->has_base_LP || e->base_LP <= 0) ? 1 : 0;
    }
    o->allow_next_def = e->defender_cd <= 1;
    o->allow_next_atk = e->attacker_cd <= 1;
}

/* TDDefense.py:34-87, Discrete branch */
void tdo_def_step(tdo_env *e, int64_t action, int difficulty, int use_np, tdo_step_out *o)
{
    clear_out(o);
    dec_cds(e);
    decode_discrete(e, action, o);
    call_enemy_opponent(e, difficulty, use_np);
    finish_def(e, o);
}

/* TDDefense.py:40-60,79-86 (the reference raises at :87 in this mode; FailCode := 0, SURVEY 9.6) */
void tdo_def_step_multi(tdo_env *e, const int64_t *action, int64_t *real_act, int difficulty,
                        int use_np, tdo_step_out *o)
{
    clear_out(o);
    dec_cds(e);
    decode_multi(e, action, real_act);
    call_enemy_opponent(e, difficulty, use_np);
    finish_def(e, o);
}

static int all_skip(const int64_t *cluster)
{
    for (int k = 0; k < TDO_CLUSTER; ++k) if (cluster[k] != TDO_NTYPES) return 0;
    return 1;
}

/* TDAttack.py:27-56 */
void tdo_atk_step(tdo_env *e, const int64_t *action, int difficulty, int use_np, tdo_step_out *o)
{
    clear_out(o);
    dec_cds(e);
    memcpy(o->real_atk, action, sizeof(o->real_atk));
    if (e->attacker_cd == 0) {
        for (int i = 0; i < e->num_roads; ++i) {
            const int64_t *cluster = action + i * TDO_CLUSTER;
            if (all_skip(cluster)) { o->fail_atk[o->n_fail_atk++] = 0; continue; }
            int64_t real[TDO_CLUSTER];
            if (tdo_summon_cluster(e, cluster, i, real)) e->attacker_cd = e->cfg.attacker_action_interval;
            memcpy(o->real_atk[i], real, sizeof(real));
            o->fail_atk[o->n_fail_atk++] = e->fail_code;
        }
    }
    call_tower_opponent(e, difficulty, use_np);
    o->reward = -tdo_board_step(e);
    o->done = tdo_done(e);
    if (o->done) {
        o->win = (!e->has_base_LP || e->base_LP <= 0) ? 1 : 0;
        o->win_attacker = o->win;
    }
    o->allow_next_atk = e->attacker_cd <= 1;
    o->allow_next_def = e->defender_cd <= 1;
}

/* TDMulti.py:46-138, Discrete-defender branch (:85-115) */
void tdo_multi_step(tdo_env *e, const int64_t *atk_action, int64_t def_action, tdo_step_out *o)
{
    clear_out(o);
    dec_cds(e);
    memcpy(o->real_atk, atk_action, sizeof(o->real_atk));
    if (e->attacker_cd == 0) {
        for (int i = 0; i < e->num_roads; ++i) {
            const int64_t *cluster = atk_action + i * TDO_CLUSTER;
            if (all_skip(cluster)) { o->fail_atk[o->n_fail_atk++] = 0; continue; }
            tdo_summon_cluster(e, cluster, i, 0);
            e->attacker_cd = e->cfg.attacker_action_interval; /* tuple truthiness, :94 */
            o->fail_atk[o->n_fail_atk++] = e->fail_code;
        }
    }
    o->real_is_def_only = decode_discrete(e, def_action, o); /* :114 replaces the dict by the int */
    finish_def(e, o);
}

/* TDMulti.py:55-84 (the reference raises at :133-136 in this mode; FailCode := 0 / [], SURVEY 9.6) */
void tdo_multi_step_multi(tdo_env *e, const int64_t *atk_action, const int64_t *def_action,
                          int64_t *real_def, tdo_step_out *o)
{
    clear_out(o);
    dec_cds(e);
    memcpy(o->real_atk, atk_action, sizeof(o->real_atk));
    if (e->attacker_cd == 0) {
        for (int i = 0; i < e->num_roads; ++i) {
            tdo_summon_cluster(e, atk_action + i * TDO_CLUSTER, i, 0);
            e->attacker_cd = e->cfg.attacker_action_interval; /* tuple truthiness, :60 */
        }
    }
    decode_multi(e, def_action, real_def);
    finish_def(e, o);
}

/* ------------------------------------------------------------------ cpu_baseline "port" leg */

static void board_restart(tdo_env *e)
{
    /* TDGymBasic.reset on the same map: fresh TDBoard state (TDBoard.py:63-79) */
    const int cells = e->L * e->L;
    for (int c = 0; c < cells; ++c) e->map6[c] = (e->road[c] & 1) ? 1 : 0;
    memset(e->enemy_LP, 0, sizeof(e->enemy_LP));
    e->cost_def = e->cfg.defender_init_cost;
    e->cost_atk = e->cfg.attacker_init_cost;
    e->base_LP = e->cfg.base_LP;
    e->steps = 0;
    e->progress = 0.;
    e->n_towers = e->n_enemies = 0;
    e->attacker_cd = e->defender_cd = 0;
    e->fail_code = TDO_SUCCESS;
}

double tdo_bench_def(tdo_env *e, int n_steps, uint64_t s, float *obs_buf)
{
    const int64_t n_act = (int64_t)e->L * e->L * 6 + 1;
    double acc = 0.;
    tdo_step_out o;
    if (!s) s = 88172645463325252ull;
    for (int i = 0; i < n_steps; ++i) {
        s ^= s << 13; s ^= s >> 7; s ^= s << 17;
        tdo_def_step(e, (int64_t)(s % (uint64_t)n_act), 1, 0, &o);
        tdo_get_states(e, obs_buf);
        acc += o.reward + obs_buf[11 * e->L * e->L];
        if (o.done) board_restart(e);
    }
    return acc;
}
