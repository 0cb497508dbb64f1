// td_common.cuh -- shared definitions of the step kernels: record layout, derived config, kernel parameters, the
// per-warp context over its shared-memory slice, and the env record load / store / reset.
// Part of the kernel set described in td_kernels.cuh.
#pragma once
#include "../../include/td_b200.h"
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

// Debug build (-DTD_DEBUG_BOUNDS): index invariants are checked on the device and a violation sets the sticky
// flag bit 2 of the env, which TDVecEnv.stats() / the parity tests surface.  (compute-sanitizer is closed on
// the B200 pool, so this is the memory-safety net next to the bit-exact parity runs.)
#ifdef TD_DEBUG_BOUNDS
#define TD_CHECK(w, cond) do { if (!(cond)) (w).flags |= 4; } while (0)
#else
#define TD_CHECK(w, cond) do { } while (0)
#endif


namespace td {


// One warp advances one env: every lane loop of the kernels strides by kLanes, and the warp intrinsics run on kFull.
constexpr int kLanes = 32;
constexpr unsigned kFull = 0xffffffffu;
// Warps per CTA of the full-write step, reset and observe kernels (td_engine.cu: step_warps_per_cta).
constexpr int kWarpsPerCta = 4;
// Env record in HBM (mirrored byte for byte in the warp's shared-memory slice):
//   [ td_env_header 64 | opponent word cache 64 | map6 cells_pad | static map (MapHdr 16, cells, dist) |
//     towers 32 x 16 | enemies 64 x 24 ]
// Everything a step normally needs sits in two contiguous prefixes, fetched in ONE round trip: the first
// runs from the header to tower kSpecTowers, the second covers enemies [0, kSpecEnemies).
constexpr int kOffRngCache = 64;          // td_env_header, then the cached generator words, then map6
constexpr int kRngCacheDef = 16;          // words cached per env: the defender env's attacker draws ~4 per step,
constexpr int kRngCacheAtk = 64;          // the attacker env's scripted defender up to ~60 (shuffle of the road cells)
constexpr int kTowerBytes = 16;
constexpr int kEnemyBytes = 24;
constexpr int kMapHdrBytes = 16;
constexpr int kMtWords = 624;
// behind the scratch area of a slice: the tower / enemy cells of the env before the step (incremental observation)
constexpr int kOldListBytes = 16 + 4 * TD_CAP_TOWERS + 4 * TD_CAP_ENEMIES;
constexpr int kTwistStageBytes = kMtWords * 4;   // staging area of the generator regeneration (tail of a slice)
// Speculatively staged list prefixes.  Lists are short in practice (tools/state_hist.py: towers p99 = 10 in the
// defender env, 11-13 in the attacker env whose scripted defender keeps building; live enemies p99 = 6): 12 towers
// and 8 enemies cover almost every env and read 256 B less per env-step than 16 / 16 (def-small 0.2156 -> 0.2132 ms,
// atk-small 0.2435 -> 0.2397 ms; 8 / 8 is best for def-small alone, 0.2126 ms, and neutral for atk-small).
constexpr int kSpecTowers = 12;
constexpr int kSpecEnemies = 8;

// Live enemies a step kernel holds on a board of side L: one per lane on 10x10 boards (one register chunk in
// board_step), TD_CAP_ENEMIES (two chunks) on every other board.  td_set_state refuses records above it.
__host__ __device__ constexpr int step_enemy_cap(int L) { return L == 10 ? kLanes : TD_CAP_ENEMIES; }

// Derived constant tables (uploaded by td_set_config).
struct DevConfig {
    double enemy_LP[TD_NTYPES][TD_NLV];
    double enemy_speed[TD_NTYPES][TD_NLV];
    double enemy_defense[TD_NTYPES][TD_NLV];
    double enemy_cost[TD_NTYPES][TD_NLV];
    double tower_attack[TD_NTYPES][TD_NLV];
    double tower_cost[TD_NTYPES][TD_NLV];
    double tower_intv[TD_NTYPES][TD_NLV];     // effective interval by (type, lv): lv1 = tower_cost[t][1] (sic)
    double tower_refund[TD_NTYPES][TD_NLV];   // Tower.cost by (type, lv): lv1 = cost[t][0] + interval[t][1] (sic)
    int tower_range[TD_NTYPES][TD_NLV];
    int tower_splash[TD_NTYPES][TD_NLV];
    double destruct_return, frozen_ratio, atk_init_cost, def_init_cost, max_cost;
    double reward_kill, penalty_leak, reward_time, rate_init, rate_final, def_rate, upgrade_at;
    int frozen_time, base_LP, tower_distance, atk_interval, def_interval, max_steps;
    int upgrade_step;       // smallest s with (double)s / max_steps >= enemy_upgrade_at (TDBoard.py:201 without the division),
                            // INT_MAX when no step count below INT_MAX reaches it (td_upgrade_step)
    double min_enemy_cost[TD_NLV];   // cheapest enemy type per level: below it every remaining cluster slot fails
};

struct MapHdr {            // 16 bytes, head of a map-pool record
    uint16_t start[3];
    uint16_t end;
    uint8_t num_roads;
    uint8_t maxd_p1;       // max(map[4]) + 1
    uint8_t pad[6];
};

struct EnvStats {          // 32 bytes per env, written only when an episode ends
    double return_sum;
    uint32_t episodes, wins, length_sum, kills, leaks, flags;
};

struct StepParams {
    uint8_t *records;          // [n][record_bytes]
    const uint8_t *maps;       // [n_maps][map_bytes]
    uint32_t *mt;              // [n][624] scripted-opponent generator words (may be NULL)
    EnvStats *stats;           // [n]
    int n_envs, n_maps, map_stride;
    int env_begin;             // the step kernel covers envs [env_begin, n_envs) (chunked host-path launches)
    int L, cells, cells_pad, record_bytes, map_bytes, smem_per_warp, scratch_off;
    int off_static, off_towers, off_enemies, rng_cache_words;
    int difficulty;
    int opponent_seeded;
    int old_lists_off;         // offset of the pre-step tower / enemy cell lists inside a slice
    int act_stage_off;         // offset of the attacker's (3, 8) int64 action / RealAction inside a slice (ATK, 2P)
    td_step_io io;
    DevConfig cfg;             // per handle: travels with every launch in the kernel-parameter constant bank
};

// ------------------------------------------------------------------------------------------------
// per-warp context: pointers into the warp's shared-memory slice + uniform registers

// CELLS > 0: board size known at compile time -> every pointer into the slice is base + constant.
// CELLS == 0: layout read from the kernel parameters (constant bank).
template <int CELLS, int RC = 0>
struct Ctx {
    static constexpr int kCells = CELLS;
    static constexpr int kRngWords = RC;
    static constexpr int kL = CELLS == 100 ? 10 : CELLS == 400 ? 20 : CELLS == 900 ? 30 : 0;
    static constexpr int kPad = (CELLS + 15) & ~15;
    uint8_t *slice;            // the warp's shared-memory slice: [record | scratch]
    const StepParams *pp;
    int lane, ecap;
    // uniform copies of hot header fields (identical in all lanes of the warp)
    double cost_def, cost_atk;
    int nt, ne, base_LP, steps, def_cd, atk_cd, fail, flags;
    // opponent generator cursor
    uint32_t *mt;
    int mt_pos;
    int ck, cn;                 // consumed / valid words of the (tempered) word cache
    bool static_dirty;          // the record's static map was replaced (reset)
    bool cache_dirty;           // the word cache changed this step (it goes back to the record)
    bool cache_raw;             // ... by the asynchronous top-up: its words still have to be tempered

    __device__ __forceinline__ int L() const { return CELLS ? kL : pp->L; }
    __device__ __forceinline__ int ncells() const { return CELLS ? CELLS : pp->cells; }
    __device__ __forceinline__ int cells_pad() const { return CELLS ? kPad : pp->cells_pad; }
    __device__ __forceinline__ int map_bytes() const { return kMapHdrBytes + 2 * cells_pad(); }
    // RC > 0: cached generator words known at compile time; RC == 0: read from the kernel parameters
    __device__ __forceinline__ int rng_words() const { return RC ? RC : pp->rng_cache_words; }
    __device__ __forceinline__ int hdr_bytes() const { return kOffRngCache + 4 * rng_words(); }
    __device__ __forceinline__ int off_static() const { return hdr_bytes() + cells_pad(); }
    __device__ __forceinline__ int off_towers() const { return off_static() + map_bytes(); }
    __device__ __forceinline__ int off_enemies() const { return off_towers() + TD_CAP_TOWERS * kTowerBytes; }
    __device__ __forceinline__ int record_bytes() const { return off_enemies() + TD_CAP_ENEMIES * kEnemyBytes; }
    __device__ __forceinline__ td_env_header *hdr() const { return reinterpret_cast<td_env_header *>(slice); }
    __device__ __forceinline__ const uint32_t *rng_cache() const { return reinterpret_cast<const uint32_t *>(slice + kOffRngCache); }
    __device__ __forceinline__ uint8_t *map6() const { return slice + hdr_bytes(); }
    __device__ __forceinline__ MapHdr *mh() const { return reinterpret_cast<MapHdr *>(slice + off_static()); }
    __device__ __forceinline__ uint8_t *cells() const { return slice + off_static() + kMapHdrBytes; }
    __device__ __forceinline__ uint8_t *dist() const { return slice + off_static() + kMapHdrBytes + cells_pad(); }
    __device__ __forceinline__ td_tower_rec *tw() const { return reinterpret_cast<td_tower_rec *>(slice + off_towers()); }
    __device__ __forceinline__ td_enemy_rec *en() const { return reinterpret_cast<td_enemy_rec *>(slice + off_enemies()); }
    __device__ __forceinline__ uint8_t *scratch() const { return slice + record_bytes(); }
    __device__ __forceinline__ uint32_t *old_lists() const
    {
        return reinterpret_cast<uint32_t *>(slice + pp->old_lists_off);
    }
    // the attacker's cluster action, later its RealAction: 24 int64 staged with the record (ATK / 2P envs)
    __device__ __forceinline__ long long *act_stage() const
    {
        return reinterpret_cast<long long *>(slice + pp->act_stage_off);
    }
    // tail of the slice (envs with a scripted opponent only): staging area of the generator regeneration
    __device__ __forceinline__ uint32_t *twist_stage() const
    {
        return reinterpret_cast<uint32_t *>(slice + pp->smem_per_warp - kTwistStageBytes);
    }
};

// n16 <= MAXN int4 with a compile-time bound: one predicated load/store pair per pass instead of a loop.
template <int MAXN>
__device__ __forceinline__ void copy16_upto(void *dst, const void *src, int n16, int lane)
{
    int4 *d = reinterpret_cast<int4 *>(dst);
    const int4 *s = reinterpret_cast<const int4 *>(src);
#pragma unroll
    for (int k = 0; k < (MAXN + kLanes - 1) / kLanes; ++k) {
        const int q = lane + kLanes * k;
        if (q < n16) d[q] = s[q];
    }
}

__device__ __forceinline__ void warp_copy16(void *dst, const void *src, int n16, int lane)
{
    int4 *d = reinterpret_cast<int4 *>(dst);
    const int4 *s = reinterpret_cast<const int4 *>(src);
    for (int q = lane; q < n16; q += kLanes) d[q] = s[q];
}

// global -> shared, 16 bytes per lane per instruction, asynchronous (LDGSTS): every segment of a stage
// is in flight at once and no register is held while the data travels.
__device__ __forceinline__ void async_copy16(void *smem_dst, const void *gmem_src, int n16, int lane)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const char *s = reinterpret_cast<const char *>(gmem_src);
    for (int q = lane; q < n16; q += kLanes)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 16u * q), "l"(s + 16 * q) : "memory");
}
__device__ __forceinline__ void async_wait_all()
{
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    __syncwarp();
}

template <class W>
__device__ __forceinline__ void ctx_bind(W &w, uint8_t *slice, const StepParams &p)
{
    w.slice = slice;
    w.pp = &p;
    w.lane = threadIdx.x & 31;
    w.ecap = TD_CAP_ENEMIES;
    w.mt = nullptr;
    w.mt_pos = 0;
    w.ck = 0; w.cn = 0;
    w.static_dirty = false;
    w.cache_dirty = false;
    w.cache_raw = false;
}

template <class W>
__device__ __forceinline__ void load_static_map(W &w, const StepParams &p, int map_id)
{
    async_copy16(w.mh(), p.maps + (size_t)map_id * w.map_bytes(), w.map_bytes() >> 4, w.lane);
    w.static_dirty = true;
}

template <class W>
__device__ __forceinline__ void pull_header(W &w)
{
    const td_env_header *h = w.hdr();
    w.cost_def = h->cost_def;
    w.cost_atk = h->cost_atk;
    w.nt = h->n_towers;
    w.ne = h->n_enemies;
    w.base_LP = h->base_LP;
    w.steps = h->steps;
    w.def_cd = h->defender_cd;
    w.atk_cd = h->attacker_cd;
    w.flags = h->flags;
    w.fail = TD_FC_SUCCESS;
    w.mt_pos = h->rng_pos;
    w.ck = h->pad1;             // cached generator words already consumed / valid (the cache holds tempered words)
    w.cn = h->pad0;
}

template <class W>
__device__ __forceinline__ void push_header(W &w)
{
    if (w.lane == 0) {
        td_env_header *h = w.hdr();
        h->cost_def = w.cost_def;
        h->cost_atk = w.cost_atk;
        h->n_towers = (uint8_t)w.nt;
        h->n_enemies = (uint8_t)w.ne;
        h->base_LP = w.base_LP;
        h->steps = w.steps;
        h->defender_cd = (int16_t)w.def_cd;
        h->attacker_cd = (int16_t)w.atk_cd;
        h->flags = (uint8_t)w.flags;
        h->rng_pos = w.mt_pos;
        h->pad0 = (uint8_t)w.cn;
        h->pad1 = w.ck;
    }
}

// Stage one env in one round trip: [header .. tower kSpecTowers) and enemies [0, kSpecEnemies) are fetched
// speculatively; only envs with longer lists pay a second trip for the rest.
template <class W>
__device__ __forceinline__ void issue_env_load(W &w, const uint8_t *rec)
{
    async_copy16(w.slice, rec, (w.off_towers() + kSpecTowers * kTowerBytes) >> 4, w.lane);
    async_copy16(w.en(), rec + w.off_enemies(), (kSpecEnemies * kEnemyBytes) >> 4, w.lane);
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// The speculative part has landed (caller waited): read the header, fetch the rare remainder.
template <class W>
__device__ __forceinline__ void finish_env_load(W &w, const StepParams &p, const uint8_t *rec, uint32_t *mt_base)
{
    pull_header(w);
    w.mt = mt_base;
    if (__builtin_expect(w.nt > kSpecTowers || w.ne > kSpecEnemies, 0)) {
        if (w.nt > kSpecTowers)
            async_copy16(w.tw() + kSpecTowers, rec + w.off_towers() + kSpecTowers * kTowerBytes, w.nt - kSpecTowers, w.lane);
        if (w.ne > kSpecEnemies)
            async_copy16(w.en() + kSpecEnemies, rec + w.off_enemies() + kSpecEnemies * kEnemyBytes,
                         ((w.ne - kSpecEnemies) * 3 + 1) >> 1, w.lane);
        async_wait_all();
    }
}

template <class W>
__device__ __forceinline__ void load_env(W &w, const StepParams &p, const uint8_t *rec, uint32_t *mt_base = nullptr)
{
    issue_env_load(w, rec);
    async_wait_all();
    finish_env_load(w, p, rec, mt_base);
}

// Write back the header block (incl. the word cache), the changed maps and the live list prefixes.
// UNROLLED: predicated single-pass copies instead of loops -- 45 fewer instructions per env-step.  Measured on
// B200: attacker env 0.291 -> 0.273 ms, in-place observation update (def-small) 0.191 -> 0.167 ms, but the
// full-write defender step 0.2175 -> 0.2220 ms (same box, twice), so the caller chooses per kernel variant.
template <bool UNROLLED = false, class W>
__device__ __forceinline__ void store_env(W &w, const StepParams &p, uint8_t *rec, bool map6_dirty, bool push = true)
{
    if (push) push_header(w);
    __syncwarp();
    const int head = w.static_dirty ? w.off_towers() : (map6_dirty ? w.off_static() : w.hdr_bytes());
    // the word cache block [kOffRngCache, hdr_bytes) goes back only when it was refilled
    const int skip_lo = w.cache_dirty ? 0 : (kOffRngCache >> 4), skip_hi = w.cache_dirty ? 0 : (w.hdr_bytes() >> 4);
    if (!UNROLLED) {
        for (int q = w.lane; q < (head >> 4); q += kLanes)
            if (q < skip_lo || q >= skip_hi) reinterpret_cast<int4 *>(rec)[q] = reinterpret_cast<const int4 *>(w.slice)[q];
        warp_copy16(rec + w.off_towers(), w.tw(), w.nt, w.lane);
        warp_copy16(rec + w.off_enemies(), w.en(), (w.ne * 3 + 1) >> 1, w.lane);
        return;
    }
    if (W::kCells > 0 && W::kRngWords > 0) {
        constexpr int kHeadMax = (kOffRngCache + 4 * W::kRngWords + 3 * W::kPad + kMapHdrBytes) / 16;   // = off_towers / 16
#pragma unroll
        for (int k = 0; k < (kHeadMax + kLanes - 1) / kLanes; ++k) {
            const int q = w.lane + kLanes * k;
            if (q < (head >> 4) && (q < skip_lo || q >= skip_hi))
                reinterpret_cast<int4 *>(rec)[q] = reinterpret_cast<const int4 *>(w.slice)[q];
        }
    } else {
        for (int q = w.lane; q < (head >> 4); q += kLanes)
            if (q < skip_lo || q >= skip_hi) reinterpret_cast<int4 *>(rec)[q] = reinterpret_cast<const int4 *>(w.slice)[q];
    }
    copy16_upto<TD_CAP_TOWERS>(rec + w.off_towers(), w.tw(), w.nt, w.lane);
    copy16_upto<(TD_CAP_ENEMIES * 3 + 1) / 2>(rec + w.off_enemies(), w.en(), (w.ne * 3 + 1) >> 1, w.lane);
}

// TDGymBasic.reset (:37-55) + TDBoard.__init__ (:63-79): fresh episode on map `map_id`.
template <class W>
__device__ __forceinline__ void reset_env(W &w, const StepParams &p, int map_id, bool reload_map)
{
    const DevConfig &cc = w.pp->cfg;
    if (reload_map) {
        __syncwarp();
        load_static_map(w, p, map_id);
        async_wait_all();
    }
    for (int q = w.lane; q < (w.cells_pad() >> 2); q += kLanes) {
        uint32_t c4 = reinterpret_cast<const uint32_t *>(w.cells())[q];
        reinterpret_cast<uint32_t *>(w.map6())[q] = c4 & 0x01010101u;           // map[6] = 1 on road cells
    }
    w.cost_def = cc.def_init_cost;
    w.cost_atk = cc.atk_init_cost;
    w.nt = 0;
    w.ne = 0;
    w.base_LP = cc.base_LP;
    w.steps = 0;
    w.def_cd = 0;
    w.atk_cd = 0;
    w.fail = TD_FC_SUCCESS;
    if (w.lane == 0) {
        w.hdr()->map_id = map_id;
        w.hdr()->ep_return = 0.0;
        w.hdr()->ep_kills = 0;
        w.hdr()->ep_leaks = 0;
        w.hdr()->ep_kills_hi = 0;
        w.hdr()->ep_leaks_hi = 0;
    }
    __syncwarp();
}

} // namespace td
