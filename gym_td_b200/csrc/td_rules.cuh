// td_rules.cuh -- the game rules, warp-cooperative on the slice: (a) defender operations and action decode,
// (b) cluster summon, the scripted opponents, (c)(d)(e) TDBoard.step (sort, targeting, damage, movement, leak,
// reward, economy).  Reference lines are cited at each function.
#pragma once
#include "td_rng.cuh"

namespace td {

// ------------------------------------------------------------------------------------------------
// Legality: every test that decides whether a defender operation or a summon succeeds.  The rules below and the
// action masks (td_action_mask_kernel) both call these, so that a mask says exactly what the next step would do.

// A purse pays a price unless it is smaller: the reference's `if cost < price: fail`, so a NaN or infinite purse
// or price behaves as it does there.
__device__ __forceinline__ bool affords(double purse, double price) { return !(purse < price); }
// a tower may stand on a cell outside every tower's diamond and off the road: map[6] == 0 (TDBoard.py:229)
__device__ __forceinline__ bool cell_free(uint8_t map6_at) { return map6_at == 0; }
// the tower list holds TD_CAP_TOWERS towers; a build beyond that fails (and flags the env)
__device__ __forceinline__ bool tower_room(int nt) { return nt < TD_CAP_TOWERS; }
__device__ __forceinline__ bool below_max_lv(int lv) { return lv < TD_NLV - 1; }
// level of the enemies a summon creates: progress >= enemy_upgrade_at, progress = steps / max_steps (TDBoard.py:201)
__device__ __forceinline__ int summon_level(const DevConfig &cc, int steps) { return steps >= cc.upgrade_step ? 1 : 0; }
// A player whose header cooldown is `cd` may act in the next step: the step lowers it to max(cd - 1, 0) first
// (TDDefense.py:38-39), and an operation needs 0.  The same test gives AllowNextMove.
__device__ __forceinline__ bool acts_next(int cd) { return cd <= 1; }

// building type t on a cell succeeds (tower_build checks cost, then position, then capacity)
__device__ __forceinline__ bool can_build(const DevConfig &cc, double cost_def, int t, uint8_t map6_at, int nt)
{
    return affords(cost_def, cc.tower_cost[t][0]) && cell_free(map6_at) && tower_room(nt);
}
// LvUp of the tower with type_lv `tl` succeeds (tower_lvup, once it found the tower)
__device__ __forceinline__ bool can_lvup(const DevConfig &cc, double cost_def, int tl)
{
    const int ty = tl & 3, lv = tl >> 2;
    return below_max_lv(lv) && affords(cost_def, cc.tower_cost[ty][lv + 1]);
}
// a cluster slot of type t summons its enemy at level lv (summon_cluster tests the cheapest type first, then t)
__device__ __forceinline__ bool can_summon(const DevConfig &cc, double cost_atk, int t, int lv)
{
    return affords(cost_atk, cc.min_enemy_cost[lv]) && affords(cost_atk, cc.enemy_cost[t][lv]);
}

// ------------------------------------------------------------------------------------------------
// (a) defender operations -- all arguments and results are warp-uniform

// map[6] += delta on the Manhattan diamond around `loc` (TDBoard.py:239-245, 281-287).  Out of line: it is
// reached from several build / destruct sites and only on the rare successful operation.
__device__ __noinline__ void diamond_add_cells(uint8_t *map6, int loc, int delta, int L, int D, int lane)
{
    const int WD = 2 * D + 1;
    const int r0 = loc / L, c0 = loc - r0 * L;
    for (int k = lane; k < WD * WD; k += kLanes) {
        int i = k / WD - D, j = k % WD - D;
        int r = r0 + i, c = c0 + j;
        if (abs(i) + abs(j) <= D && r >= 0 && r < L && c >= 0 && c < L)
            map6[r * L + c] = (uint8_t)(map6[r * L + c] + delta);
    }
    __syncwarp();
}

template <class W>
__device__ __forceinline__ void diamond_add(W &w, int loc, int delta)
{
    diamond_add_cells(w.map6(), loc, delta, w.L(), w.pp->cfg.tower_distance, w.lane);
}

template <class W>
__device__ __forceinline__ bool tower_build(W &w, int t, int loc, bool &map6_dirty)   // TDBoard.py:226-247
{
    const DevConfig &cc = w.pp->cfg;
    const double cost = cc.tower_cost[t][0];
    if (!affords(w.cost_def, cost)) { w.fail = TD_FC_COST_SHORTAGE; return false; }
    if (!cell_free(w.map6()[loc])) { w.fail = TD_FC_INVALID_POSITION; return false; }
    if (!tower_room(w.nt)) { w.flags |= 2; w.fail = TD_FC_INVALID_POSITION; return false; }
    TD_CHECK(w, loc >= 0 && loc < w.ncells() && t >= 0 && t < TD_NTYPES);
    if (w.lane == 0) {
        td_tower_rec &r = w.tw()[w.nt];
        r.cd = 0.0;
        r.loc = (uint16_t)loc;
        r.type_lv = (uint8_t)t;
    }
    w.nt += 1;
    w.cost_def = __dsub_rn(w.cost_def, cost);
    diamond_add(w, loc, +1);
    map6_dirty = true;
    w.fail = TD_FC_SUCCESS;
    return true;
}

template <class W>
__device__ __forceinline__ int find_tower(const W &w, int loc)
{
    int idx = -1;
    for (int base = 0; base < w.nt; base += kLanes) {
        const int t = base + w.lane;
        const unsigned b = __ballot_sync(kFull, t < w.nt && w.tw()[t].loc == loc);
        if (b && idx < 0) idx = base + __ffs(b) - 1;
    }
    return idx;
}

template <class W>
__device__ __forceinline__ bool tower_lvup(W &w, int loc)                              // TDBoard.py:249-271
{
    const DevConfig &cc = w.pp->cfg;
    int idx = find_tower(w, loc);
    if (idx < 0) { w.fail = TD_FC_UNKNOWN_TARGET; return false; }
    int tl = w.tw()[idx].type_lv, ty = tl & 3, lv = tl >> 2;
    if (!below_max_lv(lv)) { w.fail = TD_FC_LV_MAX; return false; }
    const double cost = cc.tower_cost[ty][lv + 1];
    if (!affords(w.cost_def, cost)) { w.fail = TD_FC_COST_SHORTAGE; return false; }
    __syncwarp();
    if (w.lane == 0) w.tw()[idx].type_lv = (uint8_t)(ty | ((lv + 1) << 2));
    __syncwarp();
    w.cost_def = __dsub_rn(w.cost_def, cost);
    w.fail = TD_FC_SUCCESS;
    return true;
}

template <class W>
__device__ __forceinline__ bool tower_destruct(W &w, int loc, bool &map6_dirty)        // TDBoard.py:273-293
{
    const DevConfig &cc = w.pp->cfg;
    int idx = find_tower(w, loc);
    if (idx < 0) { w.fail = TD_FC_UNKNOWN_TARGET; return false; }
    int tl = w.tw()[idx].type_lv;
    double c = __dadd_rn(w.cost_def, __dmul_rn(cc.tower_refund[tl & 3][tl >> 2], cc.destruct_return));
    w.cost_def = cc.max_cost < c ? cc.max_cost : c;
    // remove from the list, keeping the order of the rest
    constexpr int kPasses = TD_CAP_TOWERS / kLanes;
    td_tower_rec mine[kPasses];
#pragma unroll
    for (int q = 0; q < kPasses; ++q) {
        const int t = w.lane + kLanes * q;
        if (t > idx && t < w.nt) mine[q] = w.tw()[t];
    }
    __syncwarp();
#pragma unroll
    for (int q = 0; q < kPasses; ++q) {
        const int t = w.lane + kLanes * q;
        if (t > idx && t < w.nt) w.tw()[t - 1] = mine[q];
    }
    __syncwarp();
    w.nt -= 1;
    diamond_add(w, loc, -1);
    map6_dirty = true;
    w.fail = TD_FC_SUCCESS;
    return true;
}

// Discrete action (TDDefense.py:61-77, TDMulti.py:100-115).  Returns success.
template <class W>
__device__ __forceinline__ bool decode_discrete(W &w, long long a, long long &real, int &failcode, bool &dirty)
{
    const DevConfig &cc = w.pp->cfg;
    const long long nop = 6ll * w.ncells();
    real = nop;
    failcode = 0;
    if (w.def_cd != 0 || a == nop || (unsigned long long)a > (unsigned long long)nop) return false;
    int ai = (int)a;
    int act = ai / w.ncells(), loc = ai - act * w.ncells();
    bool res;
    if (act < TD_NTYPES) res = tower_build(w, act, loc, dirty);
    else if (act == TD_NTYPES) res = tower_lvup(w, loc);
    else res = tower_destruct(w, loc, dirty);
    if (res) { w.def_cd = cc.def_interval; real = a; }
    failcode = w.fail;
    return res;
}

// Multi-action Box(6, L, L) (TDDefense.py:40-60, TDMulti.py:65-84): r-major, c, then build 0..3, LvUp,
// destruct inside a cell, every operation seeing the state left by the previous one.  32 cells are
// screened per pass; a cell is skipped when none of its flagged operations can succeed in the
// current state (no tower on it, and no flagged build that is both affordable and placeable).  The
// screen is recomputed after every success because cost and map6 then change.
template <class W>
__device__ __forceinline__ void decode_multi(W &w, const long long *act, long long *real, bool &dirty)
{
    const DevConfig &cc = w.pp->cfg;
    const int cells = w.ncells();
    uint8_t *tower_at = w.scratch();      // cells bytes: 1 where a tower stands (scratch >= cells_pad here)
    const bool enabled = w.def_cd == 0;
    for (int q = w.lane; q < (w.cells_pad() >> 2); q += kLanes) reinterpret_cast<uint32_t *>(tower_at)[q] = 0u;
    __syncwarp();
    for (int t = w.lane; t < w.nt; t += kLanes) tower_at[w.tw()[t].loc] = 1;
    __syncwarp();
    for (int base = 0; base < cells; base += kLanes) {
        const int cell = base + w.lane;
        unsigned flags = 0;          // bit ch set when action[ch][cell] == 1
        if (cell < cells) {
#pragma unroll
            for (int ch = 0; ch < 6; ++ch) {
                long long v = __ldcs(act + (size_t)ch * cells + cell);
                flags |= (v == 1 ? 1u : 0u) << ch;
            }
        }
        unsigned done_mask = 0;      // successes of this lane's cell
        if (enabled) {
            unsigned pending = __ballot_sync(kFull, flags != 0);
            while (pending) {
                // screen with the current state
                bool can = false;
                if (flags) {
                    if (tower_at[cell]) can = (flags & 0x30u) != 0 || false;
                    if (!can && (flags & 0x0fu) && cell_free(w.map6()[cell])) {
#pragma unroll
                        for (int t = 0; t < TD_NTYPES; ++t)
                            can = can || (((flags >> t) & 1u) && affords(w.cost_def, cc.tower_cost[t][0]));
                    }
                    // a flagged build on a free cell can create the tower that a flagged LvUp/destruct then hits
                }
                unsigned cand = __ballot_sync(kFull, can) & pending;
                if (!cand) break;
                int src = __ffs(cand) - 1;
                unsigned f = __shfl_sync(kFull, flags, src);
                int loc = base + src;
                unsigned ok = 0;
                for (int t = 0; t < TD_NTYPES; ++t)
                    if ((f >> t) & 1u) if (tower_build(w, t, loc, dirty)) { ok |= 1u << t; if (w.lane == 0) tower_at[loc] = 1; __syncwarp(); }
                if ((f >> 4) & 1u) if (tower_lvup(w, loc)) ok |= 1u << 4;
                if ((f >> 5) & 1u) if (tower_destruct(w, loc, dirty)) { ok |= 1u << 5; if (w.lane == 0) tower_at[loc] = 0; __syncwarp(); }
                if (ok) w.def_cd = cc.def_interval;
                if (w.lane == src) done_mask = ok;
                // cells up to and including src are finished
                pending &= ~((2u << src) - 1u);
            }
        }
        if (cell < cells && real) {
#pragma unroll
            for (int ch = 0; ch < 6; ++ch) __stcs(real + (size_t)ch * cells + cell, (long long)((done_mask >> ch) & 1u));
        }
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// (b) summon

template <class W>
__device__ __forceinline__ void append_enemy(W &w, int t, int lv, int start)
{
    const DevConfig &cc = w.pp->cfg;
    if (w.ne >= w.ecap) { w.flags |= 1; return; }
    if (w.lane == 0) {
        td_enemy_rec &e = w.en()[w.ne];
        e.LP = cc.enemy_LP[t][lv];
        e.margin = 0.0;
        e.loc = (uint16_t)start;
        e.type_lv = (uint8_t)(t | (lv << 2));
        e.slowdown = 0;
    }
    w.ne += 1;
}

// TDBoard.py:199-224 for one road.  `mine` is this lane's slot value (lanes lane_base..lane_base+7 hold the
// cluster); updated in place to the RealAction value.  Returns the bool of the (bool, list) tuple.
// The eight types are packed into three ballots, the f64 cost chain runs on uniform registers, and the
// affordable slots append their enemies in one parallel store (list order = slot order).
template <class W>
__device__ __forceinline__ bool summon_cluster(W &w, int road, long long &mine, int lane_base)
{
    const DevConfig &cc = w.pp->cfg;
    const int start = w.mh()->start[road];
    const int lv = summon_level(cc, w.steps);
    const int tv = (mine < 0 || mine >= TD_NTYPES) ? TD_NTYPES : (int)mine;     // 4 == enemy_types: empty slot
    const unsigned b0 = __ballot_sync(kFull, tv & 1) >> lane_base, b1 = __ballot_sync(kFull, tv & 2) >> lane_base,
                   b2 = __ballot_sync(kFull, tv & 4) >> lane_base;
    unsigned todo = ~b2 & 0xffu;                     // slots holding a real type (0..3)
    const bool tried = todo != 0;
    unsigned ok = 0, poor = 0;
    const double cheapest = cc.min_enemy_cost[lv];
    while (todo) {
        if (!affords(w.cost_atk, cheapest)) { poor |= todo; break; }      // an empty purse fails every remaining slot alike
        const int k = __ffs(todo) - 1;
        todo &= todo - 1;
        const int t = ((b0 >> k) & 1) | (((b1 >> k) & 1) << 1);
        const double cost = cc.enemy_cost[t][lv];
        if (!affords(w.cost_atk, cost)) poor |= 1u << k;
        else { w.cost_atk = __dsub_rn(w.cost_atk, cost); ok |= 1u << k; }
    }
    int n = __popc(ok);
    if (n > w.ecap - w.ne) { w.flags |= 1; n = w.ecap - w.ne; }
    const int k = w.lane - lane_base;
    if (k >= 0 && k < TD_CLUSTER) {
        if ((poor >> k) & 1u) mine = TD_NTYPES;
        const int idx = __popc(ok & ((1u << k) - 1u));
        if (((ok >> k) & 1u) && idx < n) {
            td_enemy_rec &e = w.en()[w.ne + idx];
            e.LP = cc.enemy_LP[tv][lv];
            e.margin = 0.0;
            e.loc = (uint16_t)start;
            e.type_lv = (uint8_t)(tv | (lv << 2));
            e.slowdown = 0;
        }
    }
    w.ne += n;
    __syncwarp();
    if (ok == 0 && tried) { w.fail = TD_FC_COST_SHORTAGE; return false; }
    w.fail = TD_FC_SUCCESS;
    return true;
}

// scripted attacker of the defender env: 8 x type t on one road (TDGymBasic.py:95-108 -> TDBoard.py:199-224).
// All eight slots cost the same, so the first unaffordable slot ends the cluster; the summoned enemies are
// appended by eight lanes at once.
template <class W>
__device__ __forceinline__ void summon_uniform(W &w, int t, int road)
{
    const DevConfig &cc = w.pp->cfg;
    const int start = w.mh()->start[road];
    const int lv = summon_level(cc, w.steps);
    const double cost = cc.enemy_cost[t][lv];
    int n = 0;
#pragma unroll 1
    for (int k = 0; k < TD_CLUSTER; ++k) {
        if (!affords(w.cost_atk, cost)) break;
        w.cost_atk = __dsub_rn(w.cost_atk, cost);
        ++n;
    }
    w.fail = n == 0 ? TD_FC_COST_SHORTAGE : TD_FC_SUCCESS;
    if (n > w.ecap - w.ne) { w.flags |= 1; n = w.ecap - w.ne; }
    if (w.lane < n) {
        td_enemy_rec &e = w.en()[w.ne + w.lane];
        e.LP = cc.enemy_LP[t][lv];
        e.margin = 0.0;
        e.loc = (uint16_t)start;
        e.type_lv = (uint8_t)(t | (lv << 2));
        e.slowdown = 0;
    }
    w.ne += n;
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// scripted opponents on the device generator (TDGymBasic.py:81-196, random_agent=True)

// host_cluster != 0xffffffff: the eight types and the road were drawn by the host (td_step_io.opponent_cluster_dev)
template <class W>
__device__ __forceinline__ void opponent_enemy(W &w, int difficulty, unsigned host_cluster)
{
    const DevConfig &cc = w.pp->cfg;
    if (w.atk_cd != 0) return;
    if (difficulty == 0) {                                   // random_enemy_lv0
        long long mine = 0;
        int road;
        if (host_cluster != 0xffffffffu) {
            mine = w.lane < TD_CLUSTER ? (long long)((host_cluster >> (2 * w.lane)) & 3u) : 0ll;
            road = min((int)((host_cluster >> 16) & 3u), w.mh()->num_roads - 1);
        } else {
            for (int k = 0; k < TD_CLUSTER; ++k) { int t = py_randbelow(w, TD_NTYPES + 1); if (w.lane == k) mine = t; }
            road = py_randbelow(w, w.mh()->num_roads);
        }
        summon_cluster(w, road, mine, 0);
    } else {                                                 // random_enemy_lv1
        int t = py_randbelow(w, TD_NTYPES);
        int road = py_randbelow(w, w.mh()->num_roads);
        summon_uniform(w, t, road);
    }
    w.atk_cd = cc.atk_interval;                              // the returned tuple is always truthy
}

template <class W>
__device__ __forceinline__ void opponent_tower(W &w, int difficulty, bool &dirty)
{
    const DevConfig &cc = w.pp->cfg;
    if (w.def_cd != 0) return;
    const int L = w.L();
    if (difficulty == 0) {                                   // random_tower_lv0
        int r = py_randbelow(w, L), c = py_randbelow(w, L), t = py_randbelow(w, TD_NTYPES);
        if (tower_build(w, t, r * L + c, dirty)) w.def_cd = cc.def_interval;
        return;
    }
    int act = py_randbelow(w, 3);                            // random_tower_lv1 / lv2
    if (act == 0) {
        int t = 0;
        if (difficulty == 2) {
            // TDGymBasic.py:216-240: counter the enemy type drawn in proportion to the live enemies
            if (w.ne == 0) return;
            int cnt[TD_NTYPES] = {0, 0, 0, 0};
            for (int base = 0; base < w.ne; base += kLanes) {
                const int e = base + w.lane;
                const int ty = e < w.ne ? (w.en()[e].type_lv & 3) : -1;
#pragma unroll
                for (int q = 0; q < TD_NTYPES; ++q) cnt[q] += __popc(__ballot_sync(kFull, ty == q));
            }
            double p = py_random(w);
            int pick = -1, last = 0;
#pragma unroll
            for (int q = 0; q < TD_NTYPES; ++q) {
                if (cnt[q] == 0 || pick >= 0) continue;
                const double ratio = (double)(float)cnt[q] / (double)w.ne;   // float32 counts / np.int64 sum -> f64
                last = q;
                if (p < ratio) pick = q;
                else p = __dsub_rn(p, ratio);
            }
            if (pick < 0) pick = last;
            t = pick == 0 ? 2 : pick == 2 ? 1 : 0;           // [2, 0, 1, 0][type]
            if (py_random(w) < 0.2) t = 3;
        }
        // road cells in row-major order
        uint16_t *list = reinterpret_cast<uint16_t *>(w.scratch());
        int n = 0;
        for (int base = 0; base < w.ncells(); base += kLanes) {
            int c = base + w.lane;
            bool on = c < w.ncells() && (w.cells()[c] & 1);
            unsigned b = __ballot_sync(kFull, on);
            TD_CHECK(w, 2 * (n + __popc(b)) <= max(768, w.cells_pad()));
            if (on) list[n + __popc(b & ((1u << w.lane) - 1u))] = (uint16_t)c;
            n += __popc(b);
        }
        __syncwarp();
        py_shuffle_u16(w, list, n);
        if (difficulty != 2) t = py_randbelow(w, TD_NTYPES);
        for (int k = 0; k < n; ++k) {
            int di = py_randbelow(w, 25);
            int cell = list[k];
            int r = cell / L + (di / 5 - 2), c = cell % L + (di % 5 - 2);
            if (r < 0 || r >= L || c < 0 || c >= L) continue;
            if (tower_build(w, t, r * L + c, dirty)) { w.def_cd = cc.def_interval; return; }
            if (w.fail == TD_FC_COST_SHORTAGE) return;
        }
    } else {
        if (w.nt == 0) return;
        if (act == 2 && py_random(w) > .01) return;
        int id = py_randbelow(w, w.nt);
        int loc = w.tw()[id].loc;
        bool ok = act == 1 ? tower_lvup(w, loc) : tower_destruct(w, loc, dirty);
        if (ok) w.def_cd = cc.def_interval;
    }
}

// ------------------------------------------------------------------------------------------------
// (c)(d)(e) TDBoard.step, returns the defender reward; kills/leaks for the statistics

struct EnemyRegs {
    double LP, margin;
    int loc, tl, slow, r, c;
    bool valid;
};

template <class W>
__device__ __forceinline__ double board_step(W &w, int &kills_out, int &leaks_out)
{
    constexpr int NCHUNK = step_enemy_cap(W::kL) / kLanes;     // enemies per lane
    const DevConfig &cc = w.pp->cfg;
    const int L = w.L(), lane = w.lane;
    double reward = __dadd_rn(0.0, cc.reward_time);
    w.steps += 1;
    const double progress = (double)w.steps / (double)cc.max_steps;

    const int ne = w.ne, nt = w.nt;
    EnemyRegs E[NCHUNK];
    double *keys = reinterpret_cast<double *>(w.scratch());    // [64]
    uint8_t *erow = w.scratch() + 512, *ecol = w.scratch() + 576;  // [64] each

    // ---- load enemies into registers, sort key = dist - margin (TDBoard.py:305)
    bool unsorted = false;
#pragma unroll
    for (int k = 0; k < NCHUNK; ++k) {
        int e = lane + kLanes * k;
        E[k].valid = e < ne;
        if (E[k].valid) {
            const td_enemy_rec &x = w.en()[e];
            E[k].LP = x.LP; E[k].margin = x.margin; E[k].loc = x.loc; E[k].tl = x.type_lv; E[k].slow = x.slowdown;
            keys[e] = __dsub_rn((double)w.dist()[E[k].loc], E[k].margin);
        }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NCHUNK; ++k) {
        int e = lane + kLanes * k;
        bool inv = E[k].valid && e > 0 && keys[e - 1] > keys[e];
        unsorted = unsorted || inv;
    }
    unsorted = __any_sync(kFull, unsorted);
    if (unsorted) {
        // stable rank = #(key smaller) + #(equal key, earlier position)
        int rank[NCHUNK];
#pragma unroll
        for (int k = 0; k < NCHUNK; ++k) rank[k] = 0;
        for (int j = 0; j < ne; ++j) {
            double kj = keys[j];
#pragma unroll
            for (int k = 0; k < NCHUNK; ++k) {
                int e = lane + kLanes * k;
                if (E[k].valid) { double ke = keys[e]; rank[k] += (kj < ke || (kj == ke && j < e)) ? 1 : 0; }
            }
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < NCHUNK; ++k)
            if (E[k].valid) {
                TD_CHECK(w, rank[k] >= 0 && rank[k] < ne);
                td_enemy_rec &x = w.en()[rank[k]];
                x.LP = E[k].LP; x.margin = E[k].margin; x.loc = (uint16_t)E[k].loc; x.type_lv = (uint8_t)E[k].tl;
                x.slowdown = (uint8_t)E[k].slow;
            }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < NCHUNK; ++k) {
            int e = lane + kLanes * k;
            if (E[k].valid) {
                const td_enemy_rec &x = w.en()[e];
                E[k].LP = x.LP; E[k].margin = x.margin; E[k].loc = x.loc; E[k].tl = x.type_lv; E[k].slow = x.slowdown;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < NCHUNK; ++k) {
        int e = lane + kLanes * k;
        if (E[k].valid) {
            E[k].r = E[k].loc / L; E[k].c = E[k].loc - E[k].r * L;
            erow[e] = (uint8_t)E[k].r; ecol[e] = (uint8_t)E[k].c;
        }
    }
    __syncwarp();

    // ---- towers choose targets: first enemy in list order within Chebyshev range, corpses included
    //      (TDBoard.py:306-312, TDElements.py:72-132).  Positions do not change inside the tower loop, so
    //      every tower's choice is independent: lane = tower.
    uint8_t *fire = w.scratch() + 640, *vict = w.scratch() + 672;     // [32] each
    for (int tt = lane; tt < nt; tt += kLanes) {
        td_tower_rec &T = w.tw()[tt];
        const int ty = T.type_lv & 3, lv = T.type_lv >> 2;
        double cd = __dsub_rn(T.cd, 1.0);
        int target = -1, victim = -1;
        if (!(cd > 0.0)) {
            const int rge = cc.tower_range[ty][lv];
            const int tr = T.loc / L, tc = T.loc - tr * L;
            for (int j = 0; j < ne; ++j) {
                int dr = abs((int)erow[j] - tr), dc = abs((int)ecol[j] - tc);
                if (max(dr, dc) <= rge) { target = j; break; }
            }
            if (target >= 0) {
                cd = __dadd_rn(cd, cc.tower_intv[ty][lv]);
                victim = target;
                if (ty == 3) {                                // Frozen: first enemy within splash of the target
                    const int sp = cc.tower_splash[ty][lv];
                    if (sp > 0) {
                        const int r0 = erow[target], c0 = ecol[target];
                        for (int j = 0; j < ne; ++j) {
                            int dr = abs((int)erow[j] - r0), dc = abs((int)ecol[j] - c0);
                            if (max(dr, dc) <= sp) { victim = j; break; }
                        }
                    }
                }
            }
            if (cd < 0.0) cd = 0.0;
        }
        T.cd = cd;
        fire[tt] = (uint8_t)(target < 0 ? 0xff : target);
        vict[tt] = (uint8_t)(victim < 0 ? 0xff : victim);
    }
    __syncwarp();

    // ---- damage in tower order: lane = enemy (TDElements.py:19-28)
    bool hit[NCHUNK];
#pragma unroll
    for (int k = 0; k < NCHUNK; ++k) hit[k] = false;
    if (ne > 0) {
        double defense[NCHUNK];
#pragma unroll
        for (int k = 0; k < NCHUNK; ++k) defense[k] = E[k].valid ? cc.enemy_defense[E[k].tl & 3][E[k].tl >> 2] : 0.0;
        for (int t = 0; t < nt; ++t) {
            const int f = fire[t];
            if (f == 0xff) continue;
            const int tl = w.tw()[t].type_lv, ty = tl & 3, lv = tl >> 2;
            const double atk = cc.tower_attack[ty][lv];
            const double floor_ = __dmul_rn(atk, .05);
            const bool magic = (ty == 1 || ty == 3);
            const int sp = cc.tower_splash[ty][lv];
            const int fr = erow[f], fc = ecol[f], v = vict[t];
#pragma unroll
            for (int k = 0; k < NCHUNK; ++k) {
                int e = lane + kLanes * k;
                bool h;
                if (ty == 2) h = E[k].valid && max(abs(E[k].r - fr), abs(E[k].c - fc)) <= sp;
                else if (ty == 3) h = E[k].valid && e == v;
                else h = E[k].valid && e == f;
                if (h) {
                    double dmg;
                    if (magic) dmg = atk;
                    else { dmg = __dsub_rn(atk, defense[k]); if (!(dmg > 0.0)) dmg = 0.0; }
                    if (dmg < floor_) dmg = floor_;
                    E[k].LP = __dsub_rn(E[k].LP, dmg);
                    if (E[k].LP <= 0.0) E[k].LP = 0.0;
                    if (ty == 3) E[k].slow = cc.frozen_time;
                    hit[k] = true;
                }
            }
        }
    }

    // ---- remove the killed, move the rest, remove the leaked (TDBoard.py:313-346)
    int kills = 0, leaks = 0, kept_before = 0;
    const int end = w.mh()->end;
    int newidx[NCHUNK];
    bool keep[NCHUNK];
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NCHUNK; ++k) {
        bool killed = E[k].valid && hit[k] && !(E[k].LP > 0.0);
        bool leaked = false;
        if (E[k].valid && !killed) {
            const double speed = cc.enemy_speed[E[k].tl & 3][E[k].tl >> 2];
            if (E[k].slow > 0) { E[k].margin = __dadd_rn(E[k].margin, __dmul_rn(speed, cc.frozen_ratio)); E[k].slow -= 1; }
            else E[k].margin = __dadd_rn(E[k].margin, speed);
            while (E[k].margin >= 1.0) {
                E[k].margin = __dsub_rn(E[k].margin, 1.0);
                int d = (w.cells()[E[k].loc] >> 4) & 3;
                E[k].loc += (d == 0) ? 1 : (d == 1) ? -1 : (d == 2) ? L : -L;
                TD_CHECK(w, E[k].loc >= 0 && E[k].loc < w.ncells() && (w.cells()[E[k].loc] & 1));
                if (E[k].loc == end) { leaked = true; break; }
            }
        }
        keep[k] = E[k].valid && !killed && !leaked;
        unsigned bk = __ballot_sync(kFull, killed), bl = __ballot_sync(kFull, leaked), bs = __ballot_sync(kFull, keep[k]);
        kills += __popc(bk);
        leaks += __popc(bl);
        newidx[k] = kept_before + __popc(bs & ((1u << lane) - 1u));
        kept_before += __popc(bs);
    }
#pragma unroll
    for (int k = 0; k < NCHUNK; ++k)
        if (keep[k]) {
            TD_CHECK(w, newidx[k] >= 0 && newidx[k] < w.ecap);
            td_enemy_rec &x = w.en()[newidx[k]];
            x.LP = E[k].LP; x.margin = E[k].margin; x.loc = (uint16_t)E[k].loc; x.type_lv = (uint8_t)E[k].tl;
            x.slowdown = (uint8_t)E[k].slow;
        }
    w.ne = kept_before;
    __syncwarp();

    reward = __dadd_rn(reward, __dmul_rn(cc.reward_kill, (double)kills));
    const bool has_base = cc.base_LP >= 0;
    for (int i = 0; i < leaks; ++i) {
        if (has_base && w.base_LP > 0) reward = __dsub_rn(reward, cc.penalty_leak);
        if (has_base) w.base_LP = max(w.base_LP - 1, 0);
    }

    // ---- economy (TDBoard.py:348-353)
    double rate;
    if (progress >= 0.5) rate = cc.rate_final;
    else rate = __dadd_rn(__dmul_rn(cc.rate_init, __dsub_rn(1.0, progress)), __dmul_rn(cc.rate_final, progress));
    double ca = __dadd_rn(w.cost_atk, rate);
    w.cost_atk = cc.max_cost < ca ? cc.max_cost : ca;
    double cd = __dadd_rn(w.cost_def, cc.def_rate);
    w.cost_def = cc.max_cost < cd ? cc.max_cost : cd;

    kills_out = kills;
    leaks_out = leaks;
    return reward;
}

} // namespace td
