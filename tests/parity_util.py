"""Shared machinery of the GPU parity tests: drive the CUDA engine (through the C ABI) and the CPU
oracle (oracle/td_oracle.c) with the same maps, actions and opponent randomness, and compare every
output and the whole board state after every step.

Comparison bar: integers, f64 costs / LP / margins / rewards and the float32 observation are all
compared BIT FOR BIT (stricter than the 1e-6 relative tolerance north_star allows for the float
LP ratios and averages).
"""
import ctypes as C
import random

import numpy as np

from gym_td_b200 import engine as E
from gym_td_b200 import mapgen
from oracle import td_oracle as TO


LAST_MAX = {"towers": 0, "enemies": 0}      # longest lists seen by the last run_parity (coverage evidence)
LAST_RUN = {}                                # what the last run_parity went through: post-done steps, overflows, episodes


def enemy_capacity(L):
    """Live enemies the step kernel holds: one per lane on 10x10 boards, 64 otherwise."""
    return 32 if L == 10 else E.CAP_ENEMIES


def stats_reduction_order(values):
    """Sum per-env f64 values in the order of td_stats_kernel (256 strided partial sums, then a halving tree)."""
    r = [0.0] * 256
    for i, v in enumerate(values):
        r[i % 256] += v
    stride = 128
    while stride:
        for t in range(stride):
            r[t] += r[t + stride]
        stride >>= 1
    return r[0]


def oracle_config_from_engine(cfg):
    """TdConfig (product) -> oracle Config; the two structs have the same field names."""
    o = TO.Config()
    for name, _ in E.TdConfig._fields_:
        src = getattr(cfg, name)
        if hasattr(src, "__len__"):
            for t in range(4):
                for l in range(2):
                    getattr(o, name)[t][l] = src[t][l]
        else:
            setattr(o, name, src)
    return o


def make_config(**overrides):
    c = E.TdConfig()
    E.lib().td_default_config(C.byref(c))
    for k, v in overrides.items():
        if k == "base_LP" and v is None:
            v = -1
        cur = getattr(c, k)
        if hasattr(cur, "__len__"):
            for t in range(4):
                for l in range(2):
                    cur[t][l] = v[t][l]
        else:
            setattr(c, k, v)
    return c


def oracle_env_from_map(m, ocfg):
    p = mapgen.planes(m)
    road_bits = (p["road"][0] | (p["road"][1] << 1) | (p["road"][2] << 2) | (p["road"][3] << 3)).astype(np.uint8)
    o = TO.OracleEnv(ocfg)
    o.init_from_planes(p["map_size"], p["num_roads"], p["start"], p["end"], road_bits, p["dist"], p["dir"])
    return o


def smart_defender_action(o, rs, p_nop=0.3, p_uniform=0.2):
    """Action generator that really exercises build / LvUp / destruct (uniform actions mostly fail)."""
    e = o.e
    L = e.L
    cells = L * L
    nop = 6 * cells
    u = rs.random_sample()
    if u < p_nop:
        return nop
    if u < p_nop + p_uniform:
        return int(rs.randint(nop + 1))
    kind = rs.randint(10)
    if kind < 6 or e.n_towers == 0:
        map6 = np.ctypeslib.as_array(e.map6)[:cells]
        free = np.flatnonzero(map6 == 0)
        if len(free) == 0:
            return nop
        road = (np.ctypeslib.as_array(e.road)[:cells] & 1).reshape(L, L)
        loc = int(free[rs.randint(len(free))])
        for _ in range(6):
            cand = int(free[rs.randint(len(free))])
            r, c = divmod(cand, L)
            if road[max(r - 2, 0):r + 3, max(c - 2, 0):c + 3].any():
                loc = cand
                break
        return int(rs.randint(4)) * cells + loc
    tw = e.towers[rs.randint(e.n_towers)]
    return (4 if kind < 9 else 5) * cells + tw.loc


def uniform_multi_action(L, rs):
    """Box(0, 2, (6, L, L), int64).sample(): the distribution of BASELINE config 3."""
    return rs.randint(0, 3, size=(6, L, L)).astype(np.int64)


def sparse_multi_action(L, rs, p=0.02):
    a = (rs.random_sample((6, L, L)) < p).astype(np.int64)
    a[rs.random_sample((6, L, L)) < p] = 2
    return a


def attacker_action(rs):
    mode = rs.randint(4)
    if mode == 0:
        return rs.randint(0, 5, size=(3, 8)).astype(np.int64)
    a = np.full((3, 8), 4, dtype=np.int64)
    if mode >= 2:
        a[rs.randint(3), :rs.randint(1, 9)] = rs.randint(4)
    return a


def compare_state(tag, eng, rec, o):
    """CUDA env record vs oracle env; raises AssertionError naming what differs."""
    st = eng.decode_state(rec)
    h, e = st["header"], o.e
    cells = e.L * e.L
    bad = []
    if float(h["cost_def"]).hex() != float(e.cost_def).hex():
        bad.append("cost_def %r != %r" % (float(h["cost_def"]), e.cost_def))
    if float(h["cost_atk"]).hex() != float(e.cost_atk).hex():
        bad.append("cost_atk %r != %r" % (float(h["cost_atk"]), e.cost_atk))
    for name, want in (("base_LP", e.base_LP if e.has_base_LP else -1), ("steps", e.steps),
                       ("defender_cd", e.defender_cd), ("attacker_cd", e.attacker_cd),
                       ("n_towers", e.n_towers), ("n_enemies", e.n_enemies)):
        if int(h[name]) != int(want):
            bad.append("%s %d != %d" % (name, int(h[name]), int(want)))
    if not bad:
        for i in range(e.n_towers):
            t, r = e.towers[i], st["towers"][i]
            got = (int(r["loc"]), int(r["type_lv"]) & 3, int(r["type_lv"]) >> 2, float(r["cd"]).hex())
            want = (t.loc, t.type, t.lv, float(t.cd).hex())
            if got != want:
                bad.append("tower %d %r != %r" % (i, got, want))
        for i in range(e.n_enemies):
            x, r = e.enemies[i], st["enemies"][i]
            got = (int(r["loc"]), int(r["type_lv"]) & 3, float(r["LP"]).hex(), float(r["margin"]).hex(),
                   int(r["slowdown"]))
            want = (x.loc, x.type, float(x.LP).hex(), float(x.margin).hex(), x.slowdown)
            if got != want:
                bad.append("enemy %d %r != %r" % (i, got, want))
        if not np.array_equal(st["map6"], np.ctypeslib.as_array(e.map6)[:cells]):
            bad.append("map6")
    if bad:
        raise AssertionError("%s: state mismatch: %s" % (tag, "; ".join(bad[:6])))


# ------------------------------------------------------------------------------------------------
# Constructed states: a board reached through the oracle's own API, then written into a CUDA env record

BIG_PURSE = float("inf")          # no cost check fails while the lists are built


def road_cells(o):
    """Road cells of the oracle env other than the end cell, where an enemy can stand (r-major order)."""
    e = o.e
    cells = e.L * e.L
    road = np.ctypeslib.as_array(e.road)[:cells] & 1
    return [c for c in np.flatnonzero(road).tolist() if c != e.end]


def free_cells(o):
    """Cells where a tower can be built now (map6 == 0, r-major order)."""
    e = o.e
    return np.flatnonzero(np.ctypeslib.as_array(e.map6)[:e.L * e.L] == 0).tolist()


def construct_state(o, towers=(), enemies=(), **header):
    """Bring oracle env `o` (fresh from oracle_env_from_map) to a constructed state.

    towers: (type, lv, loc, cd) in list order; tower_build, then tower_lvup for level 1, so the upgraded tower keeps
    the reference's swapped constants (TDElements.py:163-169) and map6 its diamond counts; then cd is written.
    cd None keeps the fresh tower's 0.
    enemies: (type, lv, loc, margin, LP, slowdown) in list order; summon_enemy at the level `progress` selects,
    then loc (a road cell, dist = dist[loc]), margin in [0, 1), LP in (0, maxLP] (None: maxLP) and slowdown written.
    header: cost_def, cost_atk, steps, defender_cd, attacker_cd, base_LP -- written last.
    Purses are large while the lists are built.  Ends with refresh() (progress, enemy statistics).  The enemies'
    levels, which the oracle does not store, are kept in o.enemy_lv (list order)."""
    e = o.e
    cells = e.L * e.L
    road = np.ctypeslib.as_array(e.road)[:cells] & 1
    for t, lv, loc, cd in towers:
        assert not road[loc], "tower on a road cell"
        e.cost_def = BIG_PURSE
        assert o.tower_build(t, loc), "tower_build(%d, %d) failed (fail code %d)" % (t, loc, e.fail_code)
        if lv:
            assert o.tower_lvup(loc)
        if cd is not None:
            e.towers[e.n_towers - 1].cd = cd
    levels = []
    upgrade_at = e.cfg.enemy_upgrade_at
    for t, lv, loc, margin, LP, slowdown in enemies:
        assert road[loc] and loc != e.end, "enemy off the road"
        assert 0.0 <= margin < 1.0 and 0 <= slowdown <= 255
        e.cost_atk = BIG_PURSE
        e.progress = 1e300 if lv else -1e300
        assert (e.progress >= upgrade_at) == bool(lv), "enemy_upgrade_at %r leaves no level-%d summon" % (upgrade_at, lv)
        assert o.summon_enemy(t, 0)
        x = e.enemies[e.n_enemies - 1]
        x.loc, x.dist, x.margin, x.slowdown = loc, e.dist[loc], margin, slowdown
        if LP is not None:
            assert 0.0 < LP <= x.maxLP, "LP %r outside (0, maxLP]" % (LP,)
            x.LP = LP
        levels.append(int(lv))
    h = dict(cost_def=e.cfg.defender_init_cost, cost_atk=e.cfg.attacker_init_cost)
    h.update(header)
    for k, v in h.items():
        if k == "base_LP":
            assert e.has_base_LP, "base_LP of a config without a base"
        setattr(e, k, v)
    o.enemy_lv = levels
    o.refresh()
    return o


def encode_record(eng, row, o, ep=None):
    """Write oracle env `o` into the CUDA env record `row` (a row of eng.get_state_raw() of the same env, which keeps
    its static map, generator word cache and rng_pos): the inverse of compare_state.  Enemy levels come from
    o.enemy_lv (construct_state).  ep: optional (ep_return, ep_kills, ep_leaks) of the running episode."""
    e, lay = o.e, eng.layout
    cells = e.L * e.L
    assert e.n_towers <= E.CAP_TOWERS and e.n_enemies <= E.CAP_ENEMIES
    h = row[:64].view(E.HEADER_DTYPE)
    h["cost_def"], h["cost_atk"] = e.cost_def, e.cost_atk
    h["base_LP"] = e.base_LP if e.has_base_LP else -1
    h["steps"], h["defender_cd"], h["attacker_cd"] = e.steps, e.defender_cd, e.attacker_cd
    h["n_towers"], h["n_enemies"] = e.n_towers, e.n_enemies
    if ep is not None:
        h["ep_return"] = ep[0]
        h["ep_kills"], h["ep_kills_hi"] = ep[1] & 0xffff, ep[1] >> 16
        h["ep_leaks"], h["ep_leaks_hi"] = ep[2] & 0xffff, ep[2] >> 16
    tw = row[lay.off_towers:lay.off_towers + 16 * E.CAP_TOWERS].view(E.TOWER_DTYPE)
    for i in range(e.n_towers):
        t = e.towers[i]
        tw[i]["cd"], tw[i]["loc"], tw[i]["type_lv"] = t.cd, t.loc, t.type | (t.lv << 2)
    en = row[lay.off_enemies:lay.off_enemies + 24 * E.CAP_ENEMIES].view(E.ENEMY_DTYPE)
    assert len(o.enemy_lv) == e.n_enemies
    for i in range(e.n_enemies):
        x = e.enemies[i]
        en[i]["LP"], en[i]["margin"], en[i]["loc"] = x.LP, x.margin, x.loc
        en[i]["type_lv"], en[i]["slowdown"] = x.type | (o.enemy_lv[i] << 2), x.slowdown
    row[lay.off_map6:lay.off_map6 + cells] = np.ctypeslib.as_array(e.map6)[:cells].astype(np.uint8)
    return row


def run_parity(kind, L, n_envs, steps, seed=0, multi=False, opponent="device", difficulty=1, cfg_overrides=None,
               check_state_every=1, device=0, use_host_api=False, multi_mode="sparse", incremental=False,
               past_done=0, overflow="forbid", generic_kernels=False, auto_reset=False, prepare=None, inspect=None,
               obs_offset=0, atk_policy=None):
    """Step `n_envs` instances on the GPU and in the oracle; compare everything each step.

    opponent: "device" (on-device CPython-compatible generator), "stream" (host-resolved type/road
    bytes, DEF only) or "none".  Returns the number of env-steps compared.

    past_done: steps every env keeps taking after its episode ended (auto-reset is off, and the reference has no
    done latch), with fresh actions, still compared with its oracle twin, which keeps stepping too.

    overflow: "forbid" -- no env may overflow its tower / enemy capacity; "expect" -- the header flags are read
    after every step, an env's overflow flag must rise on exactly the step where the oracle's tower list first
    exceeds 32 or its enemy list first exceeds enemy_capacity(L) (at any point inside the step), and the env is
    compared bit for bit until then and dropped from that step on.

    auto_reset: the step kernel restarts a finished env on its map (map_stride = n_envs) inside the step; the oracle
    twin is rebuilt on the same map and keeps its opponent stream.

    The episode statistics of the handle (td_get_stats) are checked against the oracle run at the end: every
    episode counts once, on the step where it ends.

    prepare: fn(i, oracle, rs) called for every env after the reset; it brings oracle env i to a constructed state
    (construct_state) and may return (ep_return, ep_kills, ep_leaks) of the running episode.  Every env is then
    written into its CUDA record (encode_record, td_set_state), td_observe must match get_states() bit for bit, and
    the steps start from there.  inspect: fn(eng, oracles) called right after that check, before the first step.

    obs_offset: the observation buffer starts this many float32 elements after a 256-byte aligned allocation
    (1: 4 bytes off the 16-byte boundary, the scalar store path).

    atk_policy: fn(rs) -> (3, 8) attacker action, in place of attacker_action.
    """
    import torch
    assert overflow in ("forbid", "expect") and not (auto_reset and past_done)
    dev = torch.device("cuda", device)
    LAST_MAX.update(towers=0, enemies=0)
    LAST_RUN.clear()
    LAST_RUN.update(post_done_steps=0, overflows=0, episodes=0, max_ep_kills=0, max_ep_leaks=0)
    rs = np.random.RandomState(seed)
    cfg = make_config(**(cfg_overrides or {}))
    ocfg = oracle_config_from_engine(cfg)
    eng = E.Engine(kind, L, n_envs, device=device, cfg=cfg)
    if generic_kernels:
        eng.set_option("generic_kernels", 1)
    ecap = enemy_capacity(L)
    seeds = (np.arange(n_envs, dtype=np.uint32) * 7 + 1000 * seed + 11).astype(np.uint32)
    maps, seeds, _ = mapgen.generate_batch(seeds, L)
    eng.upload_maps(maps)
    oracles = [oracle_env_from_map(maps[i], ocfg) for i in range(n_envs)]
    cells = L * L
    if opponent == "device" and kind != "2p":
        states = np.zeros((n_envs, 625), dtype=np.uint32)
        for i in range(n_envs):
            st = random.Random(int(seeds[i])).getstate()
            states[i] = np.asarray(st[1], dtype=np.uint64).astype(np.uint32)
            oracles[i].set_pyrand(st)
        eng.seed_opponent(states)
        eng.set_difficulty(difficulty)

    obs_buf = torch.empty(n_envs * 45 * cells + obs_offset, dtype=torch.float32, device=dev)
    obs = obs_buf[obs_offset:].view(n_envs, 45, L, L)
    eng.reset(obs=obs)
    torch.cuda.synchronize()
    obs_h = obs.cpu().numpy()
    for i, o in enumerate(oracles):
        assert np.array_equal(obs_h[i].view(np.uint32), o.get_states().view(np.uint32)), "obs0 env %d" % i
    ep0 = [(0.0, 0, 0)] * n_envs
    if prepare is not None:
        recs = eng.get_state_raw()
        for i, o in enumerate(oracles):
            ep0[i] = prepare(i, o, rs) or ep0[i]
            encode_record(eng, recs[i], o, ep0[i])
        eng.set_state_raw(recs)
        eng.observe(obs)
        torch.cuda.synchronize()
        obs_h = obs.cpu().numpy()
        for i, o in enumerate(oracles):
            oo = o.get_states()
            if not np.array_equal(obs_h[i].view(np.uint32), oo.view(np.uint32)):
                ch = sorted(set(np.argwhere(obs_h[i].view(np.uint32) != oo.view(np.uint32))[:, 0].tolist()))
                raise AssertionError("%s L=%d env=%d constructed state: td_observe differs in channels %s" % (kind, L, i, ch))
            compare_state("%s L=%d env=%d constructed state" % (kind, L, i), eng, eng.get_state_raw(i, 1)[0], o)
        if inspect is not None:
            inspect(eng, oracles)
            eng.observe(obs)                     # the step's in-place update trusts the buffer written last

    t = dict(
        reward=torch.zeros(n_envs, dtype=torch.float64, device=dev),
        done=torch.zeros(n_envs, dtype=torch.uint8, device=dev),
        win=torch.zeros(n_envs, dtype=torch.int8, device=dev),
        allow_next=torch.zeros(n_envs, dtype=torch.uint8, device=dev),
        fail_def=torch.zeros(n_envs, dtype=torch.int32, device=dev),
        fail_atk=torch.zeros((n_envs, 4), dtype=torch.int32, device=dev),
        real_atk=torch.zeros((n_envs, 3, 8), dtype=torch.int64, device=dev),
        real_def=torch.zeros((n_envs, 6, L, L) if multi else (n_envs,), dtype=torch.int64, device=dev),
    )
    def_shape = (n_envs, 6, L, L) if multi else (n_envs,)
    def_act = torch.zeros(def_shape, dtype=torch.int64, device=dev)
    atk_act = torch.zeros((n_envs, 3, 8), dtype=torch.int64, device=dev)
    opp = torch.zeros(n_envs, dtype=torch.uint8, device=dev)
    alive = np.ones(n_envs, dtype=bool)
    extra = np.full(n_envs, past_done, dtype=np.int64)       # steps still to take after done
    ended = np.zeros(n_envs, dtype=bool)
    overflowed = np.zeros(n_envs, dtype=bool)
    episodes = [[] for _ in range(n_envs)]                   # (return, length, win, kills, leaks) per finished episode
    ep_ret, ep_kills, ep_leaks = [list(v) for v in zip(*ep0)]
    compared = 0
    for step in range(1, steps + 1):
        a_def = np.zeros(def_shape, dtype=np.int64)
        a_atk = np.full((n_envs, 3, 8), 4, dtype=np.int64)
        a_opp = np.full(n_envs, 0xFF, dtype=np.uint8)
        for i, o in enumerate(oracles):
            if not alive[i]:
                if not multi and kind != "atk":
                    a_def[i] = 6 * cells
                continue
            if kind != "atk":
                a_def[i] = ((uniform_multi_action(L, rs) if multi_mode == "uniform" else sparse_multi_action(L, rs))
                            if multi else smart_defender_action(o, rs))
            if kind != "def":
                a_atk[i] = (atk_policy or attacker_action)(rs)
            if kind == "def" and opponent == "stream":
                tt, rd = rs.randint(4), rs.randint(o.e.num_roads)
                a_opp[i] = tt | (rd << 4)
        def_act.copy_(torch.from_numpy(a_def))
        atk_act.copy_(torch.from_numpy(a_atk))
        opp.copy_(torch.from_numpy(a_opp))
        io = E.Engine.make_io(def_action=def_act if kind != "atk" else None,
                              atk_action=atk_act if kind != "def" else None,
                              opponent=opp if (kind == "def" and opponent == "stream") else None,
                              multi_action=multi, auto_reset=auto_reset, obs=obs, reward=t["reward"], done=t["done"],
                              win=t["win"], allow_next=t["allow_next"], real_def=t["real_def"],
                              real_atk=t["real_atk"], fail_def=t["fail_def"], fail_atk=t["fail_atk"],
                              obs_incremental=incremental)
        # snapshot the records of finished envs: they must not be stepped in the comparison below
        eng.step(io, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        host = {k: v.cpu().numpy() for k, v in t.items()}
        obs_h = obs.cpu().numpy()
        check_state = step % check_state_every == 0 or step == steps
        recs = eng.get_state_raw() if (check_state or overflow == "expect") else None
        for i, o in enumerate(oracles):
            if not alive[i]:
                continue
            tag = "%s L=%d env=%d step=%d%s" % (kind, L, i, step, " (after done)" if ended[i] else "")
            o.e.peak_towers, o.e.peak_enemies = o.e.n_towers, o.e.n_enemies
            real_multi = None
            if kind == "def":
                if multi:
                    if opponent == "stream":
                        out, real_multi = _def_multi_stream(o, a_def[i], a_opp[i])
                    else:
                        out, real_multi = o.def_step_multi(a_def[i], difficulty if opponent == "device" else -1)
                elif opponent == "stream":
                    out = _def_stream(o, int(a_def[i]), a_opp[i])
                else:
                    out = o.def_step(int(a_def[i]), difficulty if opponent == "device" else -1)
            elif kind == "atk":
                out = o.atk_step(a_atk[i], difficulty if opponent == "device" else -1)
            else:
                if multi:
                    out, real_multi = o.multi_step_multi(a_atk[i], a_def[i])
                else:
                    out = o.multi_step(a_atk[i], int(a_def[i]))
            over = o.e.peak_towers > E.CAP_TOWERS or o.e.peak_enemies > ecap
            if overflow == "expect":
                flags = int(eng.decode_state(recs[i])["header"]["flags"])
                assert flags & ~3 == 0, tag + " internal check failed (flags %#x)" % flags
                assert bool(flags) == over, tag + " overflow flag %#x, oracle peak lists %d towers / %d enemies (cap %d / %d)" % (
                    flags, o.e.peak_towers, o.e.peak_enemies, E.CAP_TOWERS, ecap)
                if over:
                    alive[i] = False                 # past its capacity the env is no longer the reference's
                    overflowed[i] = True
                    LAST_RUN["overflows"] += 1
                    continue
            assert not over, tag + " the oracle's lists exceed the capacity (%d towers, %d enemies): use overflow='expect'" % (
                o.e.peak_towers, o.e.peak_enemies)
            assert float(host["reward"][i]).hex() == float(out.reward).hex(), \
                "%s reward %r != %r" % (tag, host["reward"][i], out.reward)
            assert bool(host["done"][i]) == bool(out.done), tag + " done"
            assert int(host["win"][i]) == int(out.win), tag + " win %d != %d" % (host["win"][i], out.win)
            allow = (1 if out.allow_next_def else 0) | (2 if out.allow_next_atk else 0)
            assert int(host["allow_next"][i]) == allow, tag + " allow_next"
            if kind != "atk":
                if multi:
                    assert np.array_equal(host["real_def"][i], real_multi), tag + " real_def (multi)"
                    assert int(host["fail_def"][i]) == 0
                else:
                    assert int(host["real_def"][i]) == int(out.real_def), tag + " real_def"
                    assert int(host["fail_def"][i]) == int(out.fail_def), \
                        tag + " fail_def %d != %d (a=%d)" % (host["fail_def"][i], out.fail_def, a_def[i])
            if kind != "def":
                assert np.array_equal(host["real_atk"][i], np.ctypeslib.as_array(out.real_atk)), tag + " real_atk"
                want = [out.n_fail_atk] + list(out.fail_atk[:out.n_fail_atk])
                got = host["fail_atk"][i].tolist()
                assert got[:1 + out.n_fail_atk] == want, tag + " fail_atk %r != %r" % (got, want)
            if not ended[i]:
                ep_ret[i] += out.reward
                ep_kills[i] += o.e.last_kills
                ep_leaks[i] += o.e.last_leaks
                LAST_RUN["max_ep_kills"] = max(LAST_RUN["max_ep_kills"], ep_kills[i])
                LAST_RUN["max_ep_leaks"] = max(LAST_RUN["max_ep_leaks"], ep_leaks[i])
                if out.done:
                    episodes[i].append((ep_ret[i], o.e.steps, int(out.win), ep_kills[i], ep_leaks[i]))
                    if auto_reset:
                        py = o.e.pyrand
                        oracles[i] = o = oracle_env_from_map(maps[i], ocfg)
                        o.e.pyrand = py
                        ep_ret[i], ep_kills[i], ep_leaks[i] = 0.0, 0, 0
                    else:
                        ended[i] = True
            elif not out.done:
                raise AssertionError(tag + " a finished env must report done on every later step")
            else:
                LAST_RUN["post_done_steps"] += 1
            oo = o.get_states()
            if not np.array_equal(obs_h[i].view(np.uint32), oo.view(np.uint32)):
                ch = sorted(set(np.argwhere(obs_h[i] != oo)[:, 0].tolist()))
                raise AssertionError("%s obs differs in channels %s" % (tag, ch))
            if check_state:
                compare_state(tag, eng, recs[i], o)
            compared += 1
            LAST_MAX["towers"] = max(LAST_MAX["towers"], o.e.n_towers)
            LAST_MAX["enemies"] = max(LAST_MAX["enemies"], o.e.n_enemies)
            if ended[i]:
                if extra[i] == 0:
                    alive[i] = False
                extra[i] -= 1
        if not alive.any():
            break
    st = eng.stats()
    if overflow == "forbid":
        assert st["overflow_envs"] == 0, "capacity overflow flagged"
    else:
        assert st["overflow_envs"] == int(overflowed.sum()), "overflow flagged on %d envs, expected %d" % (
            st["overflow_envs"], overflowed.sum())
    # statistics: envs that overflowed go on with lists the reference does not have; leave them out
    if not overflowed.any():
        eps = [w for per_env in episodes for w in per_env]
        LAST_RUN["episodes"] = len(eps)
        got = (st["episodes"], st["length_sum"], st["wins"], st["kills"], st["leaks"])
        want = (len(eps), sum(w[1] for w in eps), sum(w[2] for w in eps), sum(w[3] for w in eps), sum(w[4] for w in eps))
        assert got == want, "stats (episodes, length, wins, kills, leaks) %r != %r" % (got, want)
        per_env = []
        for ep in episodes:                                  # EnvStats.return_sum: the env's episodes in order
            r = 0.0
            for w in ep:
                r += w[0]
            per_env.append(r)
        want_ret = stats_reduction_order(per_env)
        assert float(st["return_sum"]).hex() == float(want_ret).hex(), "stats return %r != %r" % (st["return_sum"], want_ret)
    eng.close()
    return compared


def _opp_cluster(o, byte):
    if byte == 0xFF or o.e.attacker_cd != 0:
        return
    o.summon_cluster(np.full(8, byte & 3, dtype=np.int64), (byte >> 4) & 3)
    o.e.attacker_cd = o.cfg.attacker_action_interval


def _def_stream(o, action, byte):
    """TDDefense.step with the scripted attacker's (type, road) supplied by the caller."""
    L_ = o.L_
    # decode with no opponent (difficulty -1), but the board step must come after the summon:
    # run the wrapper pieces by hand through the oracle's board API
    e = o.e
    e.attacker_cd = max(e.attacker_cd - 1, 0)
    e.defender_cd = max(e.defender_cd - 1, 0)
    cells = e.L * e.L
    out = o.out
    C.memset(C.byref(out), 0, C.sizeof(out))
    out.win, out.win_attacker = -1, -1
    out.real_def, out.fail_def = 6 * cells, 0
    if e.defender_cd == 0 and action != 6 * cells:
        act, loc = divmod(action, cells)
        ok = o.tower_build(act, loc) if act < 4 else (o.tower_lvup(loc) if act == 4 else o.tower_destruct(loc))
        if ok:
            e.defender_cd = o.cfg.defender_action_interval
            out.real_def = action
        out.fail_def = e.fail_code
    _opp_cluster(o, int(byte))
    out.reward = o.board_step()
    out.done = int(o.done())
    if out.done:
        out.win = 1 if (not e.has_base_LP or e.base_LP > 0) else 0
    out.allow_next_def = int(e.defender_cd <= 1)
    out.allow_next_atk = int(e.attacker_cd <= 1)
    return out


def _def_multi_stream(o, action, byte):
    """TDDefense.step in multi-action mode (TDDefense.py:40-60) with the scripted attacker's (type, road) supplied
    by the caller: the wrapper restated over the oracle's board calls, flagged cells in r-major / c / channel order."""
    e = o.e
    e.attacker_cd = max(e.attacker_cd - 1, 0)
    e.defender_cd = max(e.defender_cd - 1, 0)
    L = e.L
    out = o.out
    C.memset(C.byref(out), 0, C.sizeof(out))
    out.win, out.win_attacker = -1, -1
    real = np.zeros((6, L, L), dtype=np.int64)
    if e.defender_cd == 0:
        flagged = np.argwhere(np.transpose(action, (1, 2, 0)) == 1)          # sorted by (r, c, channel)
        for r, c, ch in flagged:
            loc = int(r) * L + int(c)
            ok = o.tower_build(int(ch), loc) if ch < 4 else (o.tower_lvup(loc) if ch == 4 else o.tower_destruct(loc))
            if ok:
                e.defender_cd = o.cfg.defender_action_interval
                real[ch, r, c] = 1
    _opp_cluster(o, int(byte))
    out.reward = o.board_step()
    out.done = int(o.done())
    if out.done:
        out.win = 1 if (not e.has_base_LP or e.base_LP > 0) else 0
    out.allow_next_def = int(e.defender_cd <= 1)
    out.allow_next_atk = int(e.attacker_cd <= 1)
    return out, real
