// td_kernels.cuh -- sm_100a kernels for the batched gym-TD board step.
//
// One warp advances one game instance.  The env record (header, tower list, enemy list, map6)
// is staged from HBM into the warp's private shared-memory slice with asynchronous 16-byte copies
// (cp.async, one round trip), all game rules run warp-cooperatively on that slice (lanes = towers
// or enemies, ballots, matches and shuffles instead of loops where the reference loops), the
// (45, L, L) float32 observation is written with unrolled 128-bit stores (or updated in place,
// INC kernels), and the live prefix of the record is written back.  Nothing stays in registers
// across the observation stores.  No block-level synchronisation exists anywhere: warps never
// communicate.  DESIGN.md section 7 lists what was measured to get here, including the dead ends.
//
// Reference semantics followed (file:line under gym_TD/envs/):
//   (a) defender decode + build/LvUp/destruct  TDDefense.py:38-77, TDMulti.py:65-115, TDBoard.py:226-293,
//                                               TDElements.py:134-170 (incl. the lvup argument swap)
//   (b) cluster summon                          TDBoard.py:199-224, TDAttack.py:36-46, TDMulti.py:88-98
//   (c) advance / leak / end condition          TDBoard.py:319-346, 370-385
//   (d) sort, target selection, damage          TDBoard.py:305-317, TDElements.py:19-28, 67-132
//   (e) reward + economy                        TDBoard.py:298-299, 315, 337-338, 348-353
//   (f) enemy statistics + observation          TDBoard.py:355-365, 85-144
//   scripted opponents                          TDGymBasic.py:81-196 (CPython `random` semantics)
//
// Compile with -fmad=false: the reference never fuses a multiply-add, and costs, LP, margins and
// rewards are compared bit for bit.
#pragma once
#include "td_common.cuh"
#include "td_rng.cuh"
#include "td_rules.cuh"
#include "td_obs.cuh"

namespace td {

// ------------------------------------------------------------------------------------------------
// kernels

extern __shared__ __align__(16) uint8_t td_smem[];

// Minimum CTAs per SM of the step kernels (__launch_bounds__), which caps their registers.  7-10 instead of 6 made
// the rules faster but the step slower: the tighter register budget spills the uniform header scalars (DESIGN.md 7).
constexpr int kMinBlocks = 6;
// 10x10 boards: the attacker env is latency-bound (scripted defender): 32 warps per SM at 64 registers (24 B of
// spills): 6 / 7 / 8 CTAs per SM = 0.2490 / 0.2440 / 0.2376 ms on B200; the other kinds gain nothing or lose
// (multi-action: +5 % at 7).  Its in-place-observation variant is best at 7 (0.2075 vs 0.2195 ms at 8).
constexpr int kMinBlocksAtk = 8;
constexpr int kMinBlocksAtkInc = 7;
// 10x10 boards, Discrete defender env: 64 registers without spills, 8 CTAs per SM.  Lost while the step was HBM-bound
// (round 1); with the observation in compressible memory the SM side bounds it and 32 warps per SM win: def-small
// 0.1842 -> 0.1809 ms, in-place 0.1601 -> 0.1579 ms.
constexpr int kMinBlocksDefSmall = 8;

// One env's rules for one step: load the record, apply the actions / scripted opponent, advance the board, emit
// the per-env outputs, auto-reset.  Leaves the updated record in the slice and starts the asynchronous copy of
// the next step's generator words into the slice's word cache (the caller waits for it before store_env).
// OPP >= 0: the engine vouches that the scripted opponent of level OPP runs on the device generator and that no
// host-resolved opponent input is set, so the other levels and the host-opponent paths are not compiled in (the
// attacker kernel is instruction-fetch bound: 4,664 -> 4,088 SASS instructions, atk-small 0.2383 -> 0.2287 ms); OPP = -1 decides
// all of it at run time.
template <int KIND, bool MULTI, bool INC, int OPP, class W>
__device__ __forceinline__ void env_rules(const StepParams &p, const int env, W &w, uint8_t *rec, bool &dirty)
{
    const DevConfig &cc = p.cfg;
    const int lane = w.lane;
    const td_step_io &io = p.io;
    static_assert(OPP < 0 || KIND != TD_KIND_2P, "the two-player env has no scripted opponent");
    const bool host_opponent = OPP < 0 && ((KIND == TD_KIND_DEF && (io.opponent_dev != nullptr || io.opponent_cluster_dev != nullptr)) ||
                                           (KIND == TD_KIND_ATK && io.def_action_dev != nullptr));
    const bool device_opponent = OPP >= 0 || ((KIND != TD_KIND_2P) && p.opponent_seeded && p.mt != nullptr && !host_opponent);
    const int difficulty = OPP >= 0 ? OPP : p.difficulty;
    // the record and the inputs are requested together: one round trip
    issue_env_load(w, rec);
    long long in_def = 0;
    int in_opp = 0xff;
    if (KIND != TD_KIND_ATK && !MULTI) in_def = io.def_action_dev[env];
    if (KIND == TD_KIND_ATK && OPP < 0 && io.def_action_dev != nullptr) in_def = io.def_action_dev[env];     // host-resolved build
    unsigned in_cluster = 0xffffffffu;
    if (KIND == TD_KIND_DEF && OPP < 0 && io.opponent_cluster_dev != nullptr) in_cluster = io.opponent_cluster_dev[env];
    if (KIND != TD_KIND_DEF) {
        // the attacker's (3, 8) int64 action travels with the record: 12 asynchronous 16-byte copies into the slice,
        // where summon_cluster turns it into the RealAction in place (no registers held across the step)
        const long long *src = reinterpret_cast<const long long *>(io.atk_action_dev) + (size_t)env * TD_ROADS * TD_CLUSTER;
        if ((reinterpret_cast<uintptr_t>(io.atk_action_dev) & 15) == 0) {
            async_copy16(w.act_stage(), src, TD_ROADS * TD_CLUSTER / 2, lane);
            asm volatile("cp.async.commit_group;" ::: "memory");
        } else {
            for (int q = lane; q < TD_ROADS * TD_CLUSTER; q += kLanes) w.act_stage()[q] = src[q];
        }
    }
    if (KIND == TD_KIND_DEF && OPP < 0 && io.opponent_dev != nullptr) in_opp = io.opponent_dev[env];
    w.ecap = step_enemy_cap(W::kL);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    finish_env_load(w, p, rec, device_opponent ? p.mt + (size_t)env * kMtWords : nullptr);
    if (INC) {
        // remember where towers and enemies stand in the observation the caller's buffer still holds
        uint32_t *old = w.old_lists();
        if (lane == 0) { old[0] = (uint32_t)w.nt; old[1] = (uint32_t)w.ne; }
        for (int t = lane; t < w.nt; t += kLanes) old[4 + t] = w.tw()[t].loc | ((uint32_t)w.tw()[t].type_lv << 16);
        for (int e = lane; e < w.ne; e += kLanes) old[4 + TD_CAP_TOWERS + e] = w.en()[e].loc | ((uint32_t)(w.en()[e].type_lv & 3) << 16);
    }

    // cooldowns (TDDefense.py:38-39)
    w.atk_cd = max(w.atk_cd - 1, 0);
    w.def_cd = max(w.def_cd - 1, 0);

    long long real_def = 6ll * w.ncells();
    int fail_def = 0;
    bool def_ok = false;
    int fail_atk[TD_ROADS] = {0, 0, 0}, n_fail_atk = 0;

    auto defender = [&]() {
        if (MULTI) {
            decode_multi(w, reinterpret_cast<const long long *>(io.def_action_dev) + (size_t)env * 6 * w.ncells(),
                         io.real_def_dev ? reinterpret_cast<long long *>(io.real_def_dev) + (size_t)env * 6 * w.ncells() : nullptr,
                         dirty);
        } else {
            def_ok = decode_discrete(w, in_def, real_def, fail_def, dirty);
        }
    };
    auto attacker = [&]() {
        if (w.atk_cd == 0) {
            const int nr = w.mh()->num_roads;
            // one instance of the cluster code for all roads (kept rolled: the kernel is instruction-cache bound)
#pragma unroll 1
            for (int i = 0; i < nr; ++i) {
                long long cur = lane < TD_CLUSTER ? w.act_stage()[i * TD_CLUSTER + lane] : (long long)TD_NTYPES;
                int code = 0;
                bool skip = false;
                if (!(KIND == TD_KIND_2P && MULTI))
                    skip = __all_sync(kFull, lane >= TD_CLUSTER || cur == TD_NTYPES);           // TDAttack.py:39-41
                if (!skip) {
                    const long long before = cur;
                    const bool res = summon_cluster(w, i, cur, 0);
                    if (KIND == TD_KIND_2P) { cur = before; w.atk_cd = cc.atk_interval; }   // tuple truthiness
                    else if (res) w.atk_cd = cc.atk_interval;
                    code = w.fail;
                    if (lane < TD_CLUSTER) w.act_stage()[i * TD_CLUSTER + lane] = cur;          // RealAction
                }
                if (n_fail_atk == 0) fail_atk[0] = code; else if (n_fail_atk == 1) fail_atk[1] = code; else fail_atk[2] = code;
                ++n_fail_atk;
            }
            if (KIND == TD_KIND_2P && MULTI) n_fail_atk = 0;
        }
    };

    if (KIND == TD_KIND_DEF) {
        defender();
        if (OPP < 0 && io.opponent_dev != nullptr) {
            const int o = in_opp;
            if (o != 0xff && w.atk_cd == 0) {
                summon_uniform(w, o & 3, min((o >> 4) & 3, w.mh()->num_roads - 1));
                w.atk_cd = cc.atk_interval;
            }
        } else if (OPP < 0 && io.opponent_cluster_dev != nullptr) {
            if (in_cluster != 0xffffffffu) opponent_enemy(w, 0, in_cluster);
        } else if (device_opponent) opponent_enemy(w, difficulty, 0xffffffffu);
    } else if (KIND == TD_KIND_ATK) {
        attacker();
        if (OPP < 0 && io.def_action_dev != nullptr) {         // random_tower_lv0 resolved by the host (np_random)
            const long long top = (long long)TD_NTYPES * w.ncells();
            if (w.def_cd == 0 && in_def >= 0 && in_def < top) {
                const int t = (int)(in_def / w.ncells()), loc = (int)(in_def - (long long)t * w.ncells());
                if (tower_build(w, t, loc, dirty)) w.def_cd = cc.def_interval;
            }
        } else if (device_opponent) opponent_tower(w, difficulty, dirty);
    } else {
        attacker();
        defender();
    }
    auto refill = [&]() {
        // Generator words for the next step: copied global -> shared straight into the slice's word cache (this
        // step's draws are done with it), asynchronously, so that no register waits for them behind the observation.
        if (w.mt != nullptr && w.cn - w.ck < (w.rng_words() >> 1)) {
            w.cache_dirty = true;
            w.cache_raw = true;
            w.ck = 0;
            w.cn = min(w.rng_words(), max(kMtWords - w.mt_pos, 0));
            constexpr int kRefill = (W::kRngWords + kLanes - 1) / kLanes;
            const unsigned dst = (unsigned)__cvta_generic_to_shared(w.rng_cache());
#pragma unroll
            for (int q = 0; q < kRefill; ++q) {
                const int k = lane + kLanes * q;
                if (k < w.cn)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * k), "l"(w.mt + w.mt_pos + k) : "memory");
                else if (k < W::kRngWords)
                    const_cast<uint32_t *>(w.rng_cache())[k] = 0u;
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (INC) refill();          // in-place observation kernels write the record back first (see td_step_kernel)
    __syncwarp();

    int kills, leaks;
    double reward = board_step(w, kills, leaks);
    if (KIND == TD_KIND_ATK) reward = -reward;

    const bool has_base = cc.base_LP >= 0;
    const bool done = (has_base && w.base_LP <= 0) || w.steps >= cc.max_steps;
    const bool def_wins = !has_base || w.base_LP > 0;
    const bool atk_wins = !has_base || w.base_LP <= 0;
    const bool my_win = KIND == TD_KIND_ATK ? atk_wins : def_wins;

    if (lane == 0) {
        if (io.reward_dev) io.reward_dev[env] = reward;
        if (io.done_dev) io.done_dev[env] = done ? 1 : 0;
        if (io.win_dev) io.win_dev[env] = done ? (my_win ? 1 : 0) : -1;
        if (io.allow_next_dev) io.allow_next_dev[env] = (uint8_t)((w.def_cd <= 1 ? 1 : 0) | (w.atk_cd <= 1 ? 2 : 0));
        if (!MULTI && KIND != TD_KIND_ATK) {
            if (io.real_def_dev) io.real_def_dev[env] = real_def;
            if (io.fail_def_dev) io.fail_def_dev[env] = fail_def;
        } else if (io.fail_def_dev) io.fail_def_dev[env] = 0;
        if (KIND != TD_KIND_DEF && io.fail_atk_dev) {
            int4 f = make_int4(n_fail_atk, fail_atk[0], fail_atk[1], fail_atk[2]);
            reinterpret_cast<int4 *>(io.fail_atk_dev)[env] = f;
        }
        td_env_header *h = w.hdr();
        h->ep_return = __dadd_rn(h->ep_return, reward);
        // 32-bit episode counters kept as two 16-bit halves of the header
        const uint32_t ep_kills = ((uint32_t)h->ep_kills | ((uint32_t)h->ep_kills_hi << 16)) + (uint32_t)kills;
        const uint32_t ep_leaks = ((uint32_t)h->ep_leaks | ((uint32_t)h->ep_leaks_hi << 16)) + (uint32_t)leaks;
        h->ep_kills = (uint16_t)ep_kills;
        h->ep_kills_hi = (uint16_t)(ep_kills >> 16);
        h->ep_leaks = (uint16_t)ep_leaks;
        h->ep_leaks_hi = (uint16_t)(ep_leaks >> 16);
        // An episode counts once, on the step where it ends.  A finished env that is stepped on without a reset
        // (auto_reset off; the reference has no done latch) reports done again: the header in the slice still holds
        // the pre-step base_LP / steps, and an env that had already ended before this step is not counted again.
        const bool ended_before = h->steps > 0 && ((has_base && h->base_LP <= 0) || h->steps >= cc.max_steps);
        if (done && !ended_before) {
            EnvStats &s = p.stats[env];
            s.return_sum = __dadd_rn(s.return_sum, h->ep_return);
            s.episodes += 1;
            s.wins += my_win ? 1 : 0;
            s.length_sum += (uint32_t)w.steps;
            s.kills += ep_kills;
            s.leaks += ep_leaks;
        }
        if (w.flags) p.stats[env].flags |= (uint32_t)w.flags;
    }
    if (KIND != TD_KIND_DEF && io.real_atk_dev) {
        for (int q = lane; q < TD_ROADS * TD_CLUSTER; q += kLanes)
            io.real_atk_dev[(size_t)env * TD_ROADS * TD_CLUSTER + q] = w.act_stage()[q];
    }
    if (io.packed_out_dev != nullptr) {
        // every small output of the env in one record and one coalesced store (the buffer may be host memory)
        constexpr int kStride = KIND == TD_KIND_DEF ? 32 : 256;
        int4 *po = reinterpret_cast<int4 *>(static_cast<uint8_t *>(io.packed_out_dev) + (size_t)env * kStride);
        const long long rd = (MULTI || KIND == TD_KIND_ATK) ? 0ll : real_def;
        const long long rbits = __double_as_longlong(reward);
        const int win_v = done ? (my_win ? 1 : 0) : -1;
        const unsigned fl = (done ? 1u : 0u) | ((unsigned)(win_v & 0xff) << 8) |
                            ((unsigned)((w.def_cd <= 1 ? 1 : 0) | (w.atk_cd <= 1 ? 2 : 0)) << 16);
        int4 v = make_int4(0, 0, 0, 0);
        if (lane == 0) v = make_int4((int)rbits, (int)(rbits >> 32), (int)rd, (int)(rd >> 32));
        if (lane == 1) v = make_int4((MULTI || KIND == TD_KIND_ATK) ? 0 : fail_def, (int)fl, 0, 0);
        if (KIND != TD_KIND_DEF) {
            if (lane == 2) v = make_int4(n_fail_atk, fail_atk[0], fail_atk[1], fail_atk[2]);
            // lanes 4..15 carry real_atk[2q], real_atk[2q + 1] (q = lane - 4), straight from the slice
            if (lane >= 4 && lane < 16) v = reinterpret_cast<const int4 *>(w.act_stage())[lane - 4];
        }
        if (lane < kStride / 16) po[lane] = v;
    }
    (void)def_ok;
    __syncwarp();

    if (__builtin_expect(done && io.auto_reset, 0)) {
        int next = (w.hdr()->map_id + p.map_stride) % p.n_maps;
        if (lane == 0) w.hdr()->episode += 1;
        reset_env(w, p, next, true);
        dirty = true;
    }
    if (!INC) refill();
}

// INC: the observation is an in-place update of the previous one (td_step_io.obs_incremental, vouched for by the
// engine); a separate instantiation, so that the full-write kernels carry none of its code.
template <int KIND, bool MULTI, int CELLS, bool INC, class OT = float, int OPP = -1>
__global__ void __launch_bounds__(kWarpsPerCta * 32, (KIND == TD_KIND_ATK && CELLS == 100) ? (INC ? kMinBlocksAtkInc : kMinBlocksAtk)
                                                     : (KIND == TD_KIND_DEF && !MULTI && CELLS == 100) ? kMinBlocksDefSmall : kMinBlocks)
td_step_kernel(const __grid_constant__ StepParams p)
{
    const int warp = threadIdx.x / 32;
    const int env = p.env_begin + blockIdx.x * (blockDim.x / 32) + warp;      // any CTA size up to kWarpsPerCta warps
    if (env >= p.n_envs) return;
    constexpr int RC = KIND == TD_KIND_ATK ? kRngCacheAtk : kRngCacheDef;
    Ctx<CELLS, RC> w;
    ctx_bind(w, td_smem + (size_t)warp * p.smem_per_warp, p);               // [record | scratch] per warp
    uint8_t *rec = p.records + (size_t)env * w.record_bytes();
    bool dirty = false;
    env_rules<KIND, MULTI, INC, OPP>(p, env, w, rec, dirty);
    // The header scalars go back to the slice before the observation is written: their registers are free
    // during the store phase (a spilled one cost a local-memory reload behind 18 KB of stores: 8 % of the step).
    push_header(w);
    // In-place observation kernels write the record back before the observation (the generator words were
    // requested before board_step): 64 instead of 79 registers, def-small 0.167 -> 0.161 ms.  The full-write
    // kernels keep the record for last: 0.2175 vs 0.2206 ms on def-small.
    if (INC) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        if (w.cache_raw) { __syncwarp(); temper_cache(w); }
        store_env<true>(w, p, rec, dirty, false);
    }
    if (p.io.obs_dev) {
        OT *o = reinterpret_cast<OT *>(p.io.obs_dev) + (size_t)env * TD_NCHANNELS * w.ncells();
        if constexpr (INC && CELLS > 0) {
            obs_prepare(w);
            if (!w.static_dirty && (reinterpret_cast<uintptr_t>(o) & 15) == 0) obs_dense_incremental(w, o);
            else obs_dense(w, o);                          // envs restarted inside this step get all 45 planes
            obs_sparse(w, o);
        } else {
            write_obs(w, o);
        }
    }
    if (!INC) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");      // the next steps' generator words are in the slice
        if (w.cache_raw) { __syncwarp(); temper_cache(w); }
        store_env<(KIND == TD_KIND_ATK)>(w, p, rec, dirty, false);
    }
}

// reset (mask / explicit map ids) and observation-only kernels
__global__ void __launch_bounds__(kWarpsPerCta * 32)
td_reset_kernel(const __grid_constant__ StepParams p, const uint8_t *mask, const int32_t *map_ids, float *obs)
{
    const int warp = threadIdx.x >> 5;
    const int env = blockIdx.x * kWarpsPerCta + warp;
    if (env >= p.n_envs) return;
    if (mask && !mask[env]) return;
    Ctx<0> w;
    ctx_bind(w, td_smem + (size_t)warp * p.smem_per_warp, p);
    uint8_t *rec = p.records + (size_t)env * p.record_bytes;
    if (w.lane < (w.hdr_bytes() >> 4)) reinterpret_cast<int4 *>(w.hdr())[w.lane] = reinterpret_cast<const int4 *>(rec)[w.lane];
    __syncwarp();
    pull_header(w);
    int id = map_ids ? map_ids[env] : env % p.n_maps;
    id = ((id % p.n_maps) + p.n_maps) % p.n_maps;
    reset_env(w, p, id, true);
    if (obs) write_obs(w, obs + (size_t)env * TD_NCHANNELS * w.ncells());
    __syncwarp();
    store_env(w, p, rec, true);
}

template <int CELLS, class OT = float>
__global__ void __launch_bounds__(kWarpsPerCta * 32) td_observe_kernel(const __grid_constant__ StepParams p, OT *obs)
{
    const int warp = threadIdx.x >> 5;
    const int env = blockIdx.x * kWarpsPerCta + warp;
    if (env >= p.n_envs) return;
    Ctx<CELLS> w;
    ctx_bind(w, td_smem + (size_t)warp * p.smem_per_warp, p);
    load_env(w, p, p.records + (size_t)env * p.record_bytes);
    write_obs(w, obs + (size_t)env * TD_NCHANNELS * w.ncells());
}

// Action masks (td_action_mask): which defender actions and attacker summons the next step would carry out, decided
// from the env record by the legality predicates of td_rules.cuh.  The warp reads only what they need, into a slice
//   [ td_env_header 64 | map6 cells_pad | MapHdr 16 | towers 32 x 16 | per-cell table cells_pad ]
// (map6 and the MapHdr are adjacent in the record as well), not the generator words, enemies or static planes.
__host__ __device__ constexpr int mask_smem_per_warp(int cells_pad)
{
    return (int)sizeof(td_env_header) + cells_pad + kMapHdrBytes + TD_CAP_TOWERS * kTowerBytes + cells_pad;
}

// def_mask: [n, 6 cells + 1] bytes, entry a = 1 when the Discrete action a would come back as RealAction a (the
// first 6 cells are the (6, L, L) layout of the multi-action Box, one flag each).  atk_mask: [n, 3, 4] bytes, entry
// (r, t) = 1 when a cluster whose only slot is type t on road r would summon it.  Either may be NULL.
template <int CELLS>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
td_action_mask_kernel(const __grid_constant__ StepParams p, uint8_t *def_mask, uint8_t *atk_mask)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int env = blockIdx.x * kWarpsPerCta + warp;
    if (env >= p.n_envs) return;
    const DevConfig &cc = p.cfg;
    const int cells = CELLS > 0 ? CELLS : p.cells, cells_pad = CELLS > 0 ? ((CELLS + 15) & ~15) : p.cells_pad;
    uint8_t *slice = td_smem + (size_t)warp * mask_smem_per_warp(cells_pad);
    const td_env_header *hdr = reinterpret_cast<const td_env_header *>(slice);
    uint8_t *map6 = slice + sizeof(td_env_header);
    const MapHdr *mh = reinterpret_cast<const MapHdr *>(map6 + cells_pad);
    const td_tower_rec *tw = reinterpret_cast<const td_tower_rec *>(map6 + cells_pad + kMapHdrBytes);
    uint8_t *table = map6 + cells_pad + kMapHdrBytes + TD_CAP_TOWERS * kTowerBytes;
    const uint8_t *rec = p.records + (size_t)env * p.record_bytes;

    // header, then map6 + MapHdr (only the MapHdr without a defender mask): one round trip
    async_copy16(slice, rec, (int)sizeof(td_env_header) >> 4, lane);
    if (def_mask) async_copy16(map6, rec + p.off_static - cells_pad, (cells_pad + kMapHdrBytes) >> 4, lane);
    else async_copy16(map6 + cells_pad, rec + p.off_static, kMapHdrBytes >> 4, lane);
    async_wait_all();

    if (def_mask) {
        const double cost_def = hdr->cost_def;
        const int nt = hdr->n_towers;
        async_copy16(const_cast<td_tower_rec *>(tw), rec + p.off_towers, nt, lane);
        for (int q = lane; q < (cells_pad >> 2); q += kLanes) reinterpret_cast<uint32_t *>(table)[q] = 0u;
        async_wait_all();
        // lane = tower: the first tower of the list on a cell (the one find_tower picks) marks it in the table,
        // bit 0 = a tower stands there (Destruct), bit 1 = its LvUp succeeds
        static_assert(TD_CAP_TOWERS == kLanes, "one tower per lane");
        const bool have = lane < nt;
        const int loc = have ? tw[lane].loc : 0;
        const unsigned same = __match_any_sync(kFull, have ? (unsigned)loc : 0x10000u + lane);
        if (have && lane == __ffs(same) - 1) table[loc] = (uint8_t)(1u | (can_lvup(cc, cost_def, tw[lane].type_lv) ? 2u : 0u));
        __syncwarp();
        // lane = cell: bit ch of table[cell] = entry (ch, cell), build 0..3, LvUp, Destruct
        const bool acts = acts_next(hdr->defender_cd);
        for (int cell = lane; cell < cells; cell += kLanes) {
            const unsigned tower = table[cell];
            unsigned bits = 0;
            if (acts) {
#pragma unroll
                for (int t = 0; t < TD_NTYPES; ++t) bits |= (can_build(cc, cost_def, t, map6[cell], nt) ? 1u : 0u) << t;
                bits |= ((tower >> 1) & 1u) << 4 | (tower & 1u) << 5;
            }
            table[cell] = (uint8_t)bits;
        }
        __syncwarp();
        // The row (6 cells + 1 bytes, so rows of successive envs start at every alignment) in 16-byte chunks of the
        // aligned address space: whole chunks go out in one store, the partial chunks at either end byte by byte.
        const int row_bytes = 6 * cells + 1;
        uint8_t *row = def_mask + (size_t)env * row_bytes;
        const int head = (int)(reinterpret_cast<uintptr_t>(row) & 15);
        const int chunks = (head + row_bytes + 15) >> 4;
        for (int q = lane; q < chunks; q += kLanes) {
            const int i0 = 16 * q - head;             // row entry of the chunk's first byte (negative: before the row)
            int ch = 0, cell = i0;
            if (i0 > 0) { ch = i0 / cells; cell = i0 - ch * cells; }
            uint32_t v[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int i = i0 + j;
                if (i >= 0 && i < row_bytes) v[j >> 2] |= (ch < 6 ? (table[cell] >> ch) & 1u : 1u) << (8 * (j & 3));   // the no-op: always 1
                if (++cell == cells) { cell = 0; ++ch; }
            }
            uint8_t *dst = row - head + 16 * q;
            if (i0 >= 0 && i0 + 16 <= row_bytes) {
                *reinterpret_cast<uint4 *>(dst) = make_uint4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (i0 + j >= 0 && i0 + j < row_bytes) dst[j] = (uint8_t)(v[j >> 2] >> (8 * (j & 3)));
            }
        }
    }
    if (atk_mask && lane < TD_ROADS * TD_NTYPES) {
        const int r = lane / TD_NTYPES, t = lane % TD_NTYPES;
        const bool ok = acts_next(hdr->attacker_cd) && r < mh->num_roads &&
                        can_summon(cc, hdr->cost_atk, t, summon_level(cc, hdr->steps));
        atk_mask[(size_t)env * TD_ROADS * TD_NTYPES + lane] = ok ? 1 : 0;
    }
}

// deterministic reduction of the per-env statistics: one block, fixed order
__global__ void __launch_bounds__(256) td_stats_kernel(const EnvStats *s, int n, long long steps, td_stats *out)
{
    __shared__ double r[256];
    __shared__ long long acc[256][6];
    const int t = threadIdx.x;
    double rs = 0.0;
    long long a[6] = {0, 0, 0, 0, 0, 0};
    for (int i = t; i < n; i += 256) {
        rs += s[i].return_sum;
        a[0] += s[i].episodes; a[1] += s[i].length_sum; a[2] += s[i].wins;
        a[3] += s[i].kills; a[4] += s[i].leaks; a[5] += s[i].flags ? 1 : 0;
    }
    r[t] = rs;
    for (int k = 0; k < 6; ++k) acc[t][k] = a[k];
    __syncthreads();
    for (int stride = 128; stride > 0; stride >>= 1) {
        if (t < stride) {
            r[t] += r[t + stride];
            for (int k = 0; k < 6; ++k) acc[t][k] += acc[t + stride][k];
        }
        __syncthreads();
    }
    if (t == 0) {
        out->return_sum = r[0];
        out->episodes = acc[0][0]; out->length_sum = acc[0][1]; out->wins = acc[0][2];
        out->kills = acc[0][3]; out->leaks = acc[0][4]; out->overflow_envs = acc[0][5];
        out->steps = steps;
    }
}

} // namespace td
