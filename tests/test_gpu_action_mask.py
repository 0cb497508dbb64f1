"""Action masks (td_action_mask, TDVecEnv.action_mask) against the oracle, action by action.

The definition the masks are held to is what the next step does:
- defender entry a is 1 exactly when the Discrete action a comes back with RealAction == a, and, in multi-action mode,
  when the Box action whose only flag is (ch, r, c) comes back with real_def[ch, r, c] == 1;
- attacker entry (r, t) is 1 exactly when a cluster whose only non-empty slot is type t on road r summons the enemy.
  RealAction cannot decide that (TD-2p echoes the input), so the oracle's enemy counter (next_uid) does.
Every candidate action is tried on a fresh copy of the env's oracle twin (ctypes copy of oracle.td_oracle.Env,
generator state included), stepped through the same env wrapper the twin follows.
"""
import ctypes as C

import numpy as np
import pytest

from gym_td_b200 import engine as E
from gym_td_b200 import mapgen
from oracle import td_oracle as TO
from tests import parity_util as PU

EMPTY_CLUSTER = np.full((3, 8), 4, dtype=np.int64)


class Twin(object):
    """Scratch copy of an oracle env: load() overwrites it with the env to be tried."""

    def __init__(self, o):
        self.c = TO.OracleEnv.__new__(TO.OracleEnv)
        self.c.L_, self.c.cfg, self.c.out = o.L_, o.cfg, TO.StepOut()
        self.c.e = TO.Env.from_buffer_copy(o.e)

    def load(self, o):
        C.memmove(C.byref(self.c.e), C.byref(o.e), C.sizeof(TO.Env))
        return self.c


def oracle_def_mask(kind, multi, o, difficulty):
    """The defender mask by definition: every Discrete action (or single-flag Box action) on a fresh twin."""
    L = o.e.L
    cells = L * L
    nop = 6 * cells
    tw = Twin(o)
    if not multi:
        want = np.zeros(nop + 1, dtype=bool)
        for a in range(nop + 1):
            c = tw.load(o)
            out = c.def_step(a, difficulty) if kind == "def" else c.multi_step(EMPTY_CLUSTER, a)
            want[a] = int(out.real_def) == a
        return want
    want = np.zeros(nop, dtype=bool)
    box = np.zeros(nop, dtype=np.int64)
    for a in range(nop):
        c = tw.load(o)
        box[a] = 1
        if kind == "def":
            _, real = c.def_step_multi(box.reshape(6, L, L), difficulty)
        else:
            _, real = c.multi_step_multi(EMPTY_CLUSTER, box.reshape(6, L, L))
        box[a] = 0
        real = real.reshape(-1)
        assert real.sum() == real[a], "a single-flag Box action set another RealAction flag"
        want[a] = real[a] == 1
    return want


def oracle_atk_mask(kind, multi, o, difficulty):
    """The attacker mask by definition: every single-slot cluster on a fresh twin; summoned = the enemy counter moved."""
    L = o.e.L
    tw = Twin(o)
    want = np.zeros((3, 4), dtype=bool)
    for r in range(3):
        for t in range(4):
            cluster = EMPTY_CLUSTER.copy()
            cluster[r, 0] = t
            c = tw.load(o)
            before = c.e.next_uid
            if kind == "atk":
                c.atk_step(cluster, difficulty)
            elif multi:
                c.multi_step_multi(cluster, np.zeros((6, L, L), dtype=np.int64))
            else:
                c.multi_step(cluster, 6 * L * L)
            want[r, t] = c.e.next_uid > before
    return want


def check_masks(tag, kind, multi, o, difficulty, dmask, amask):
    """GPU mask rows of one env vs the oracle twin, action by action."""
    L = o.e.L
    if kind != "atk":
        got = dmask.astype(bool)
        assert got.shape == (6 * L * L + 1,)
        assert got[-1], tag + " the no-op must always be legal"
        want = oracle_def_mask(kind, multi, o, difficulty)
        if multi:
            got = got[:-1]
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, "%s defender mask differs at %d actions, first %r (mask %r, step %r)" % (
            tag, bad.size, bad[:8].tolist(), got[bad[:8]].tolist(), want[bad[:8]].tolist())
    if kind != "def":
        got = amask.astype(bool).reshape(3, 4)
        want = oracle_atk_mask(kind, multi, o, difficulty)
        assert np.array_equal(got, want), "%s attacker mask %r != %r" % (tag, got.astype(int).tolist(), want.astype(int).tolist())


def read_masks(eng, kind, n, L, torch, dev):
    d = torch.zeros((n, 6 * L * L + 1), dtype=torch.uint8, device=dev) if kind != "atk" else None
    a = torch.zeros((n, 3, 4), dtype=torch.uint8, device=dev) if kind != "def" else None
    eng.action_mask(d, a, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return (d.cpu().numpy() if d is not None else None), (a.cpu().numpy() if a is not None else None)


def run_masks(kind, L, multi, n_envs, steps, check_at, per_check, seed, auto_reset, cfg_overrides):
    """Random play on the GPU and in the oracle; at the steps in check_at, the masks of `per_check` sampled envs are
    checked action by action.  Returns (checks, checks of envs past the end of an episode or restarted)."""
    import torch
    dev = torch.device("cuda", 0)
    rs = np.random.RandomState(seed)
    cfg = PU.make_config(**cfg_overrides)
    ocfg = PU.oracle_config_from_engine(cfg)
    eng = E.Engine(kind, L, n_envs, cfg=cfg)
    maps, seeds, _ = mapgen.generate_batch((np.arange(n_envs, dtype=np.uint32) * 13 + 100 * seed + 5).astype(np.uint32), L)
    eng.upload_maps(maps)
    oracles = [PU.oracle_env_from_map(maps[i], ocfg) for i in range(n_envs)]
    difficulty = 1
    if kind != "2p":
        import random
        states = np.zeros((n_envs, 625), dtype=np.uint32)
        for i in range(n_envs):
            st = random.Random(int(seeds[i])).getstate()
            states[i] = np.asarray(st[1], dtype=np.uint64).astype(np.uint32)
            oracles[i].set_pyrand(st)
        eng.seed_opponent(states)
        eng.set_difficulty(difficulty)
    cells = L * L
    eng.reset()
    def_shape = (n_envs, 6, L, L) if multi else (n_envs,)
    t = dict(real_def=torch.zeros(def_shape, dtype=torch.int64, device=dev),
             real_atk=torch.zeros((n_envs, 3, 8), dtype=torch.int64, device=dev),
             done=torch.zeros(n_envs, dtype=torch.uint8, device=dev))
    def_act = torch.zeros(def_shape, dtype=torch.int64, device=dev)
    atk_act = torch.zeros((n_envs, 3, 8), dtype=torch.int64, device=dev)
    finished = np.zeros(n_envs, dtype=bool)          # past done (auto-reset off) or restarted (auto-reset on)
    checks = special = 0
    for step in range(steps + 1):
        if step in check_at:
            dm, am = read_masks(eng, kind, n_envs, L, torch, dev)
            recs = eng.get_state_raw()
            pick = rs.choice(n_envs, size=per_check, replace=False)
            # prefer envs past an episode end when there are some
            late = np.flatnonzero(finished)
            if late.size:
                pick[0] = late[rs.randint(late.size)]
            for i in pick:
                tag = "%s L=%d multi=%d env=%d step=%d" % (kind, L, multi, i, step)
                PU.compare_state(tag, eng, recs[i], oracles[i])
                check_masks(tag, kind, multi, oracles[i], difficulty,
                            dm[i] if dm is not None else None, am[i] if am is not None else None)
                checks += 1
                special += int(finished[i])
        if step == steps:
            break
        a_def = np.zeros(def_shape, dtype=np.int64)
        a_atk = np.full((n_envs, 3, 8), 4, dtype=np.int64)
        for i, o in enumerate(oracles):
            if kind != "atk":
                a_def[i] = PU.sparse_multi_action(L, rs, p=0.05) if multi else PU.smart_defender_action(o, rs)
            if kind != "def":
                a_atk[i] = PU.attacker_action(rs)
        def_act.copy_(torch.from_numpy(a_def))
        atk_act.copy_(torch.from_numpy(a_atk))
        io = E.Engine.make_io(def_action=def_act if kind != "atk" else None, atk_action=atk_act if kind != "def" else None,
                              multi_action=multi, auto_reset=auto_reset, done=t["done"], real_def=t["real_def"],
                              real_atk=t["real_atk"])
        eng.step(io, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        done = t["done"].cpu().numpy()
        for i, o in enumerate(oracles):
            if kind == "def":
                out = o.def_step_multi(a_def[i], difficulty)[0] if multi else o.def_step(int(a_def[i]), difficulty)
            elif kind == "atk":
                out = o.atk_step(a_atk[i], difficulty)
            else:
                out = o.multi_step_multi(a_atk[i], a_def[i])[0] if multi else o.multi_step(a_atk[i], int(a_def[i]))
            assert bool(done[i]) == bool(out.done), "%s L=%d env=%d step=%d done" % (kind, L, i, step)
            if out.done:
                finished[i] = True
                if auto_reset:
                    py = o.e.pyrand
                    oracles[i] = PU.oracle_env_from_map(maps[i], ocfg)
                    oracles[i].e.pyrand = py
    assert eng.stats()["overflow_envs"] == 0
    eng.close()
    return checks, special


CASES = [(kind, L, multi) for kind in ("def", "atk", "2p") for L in (10, 20, 30, 13)
         for multi in ((False,) if kind == "atk" else (False, True))]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,L,multi", CASES)
def test_mask_matches_next_step(kind, L, multi):
    # short episodes, so that the checks see envs restarted by the step (auto-reset on 10 / 30) and envs stepped past
    # the end (auto-reset off on 20 / 13); cooldowns of 2 on half the cases make defender_cd / attacker_cd 2 reachable
    auto_reset = L in (10, 30)
    cfg = dict(max_episode_steps=14)
    if multi or L == 20:
        cfg.update(defender_action_interval=2, attacker_action_interval=2)
    per_check = 3 if L < 30 else 2
    checks, special = run_masks(kind, L, multi, n_envs=12, steps=22, check_at=(0, 4, 9, 13, 17, 22), per_check=per_check,
                                seed=L * 7 + (3 if multi else 0) + {"def": 0, "atk": 1, "2p": 2}[kind],
                                auto_reset=auto_reset, cfg_overrides=cfg)
    assert checks == 6 * per_check
    assert special >= 2, "no check saw an env past the end of an episode"


# ------------------------------------------------------------------------------------------------
# Constructed boundary states

def _maps_with_roads(L, roads_per_env, seed):
    out = []
    for k, nr in enumerate(roads_per_env):
        maps, _, _ = mapgen.generate_batch(np.array([seed + 31 * k], dtype=np.uint32), L, num_roads=nr)
        out.append(E.TdMap.from_buffer_copy(maps[0]))
    return out


def run_constructed(kind, L, cfg_overrides, specs, multi=False, seed=0):
    """One env per spec: spec(o, rs) brings oracle env o to a state (construct_state); the states go into the CUDA
    records (encode_record, td_set_state) and the masks are checked action by action.  Returns the mask rows."""
    import torch
    dev = torch.device("cuda", 0)
    rs = np.random.RandomState(seed)
    n = len(specs)
    cfg = PU.make_config(**cfg_overrides)
    ocfg = PU.oracle_config_from_engine(cfg)
    eng = E.Engine(kind, L, n, cfg=cfg)
    maps = _maps_with_roads(L, [1 + i % 3 for i in range(n)], 1000 + seed)
    eng.upload_maps(maps)
    oracles = [PU.oracle_env_from_map(maps[i], ocfg) for i in range(n)]
    eng.reset()
    recs = eng.get_state_raw()
    for i, (o, spec) in enumerate(zip(oracles, specs)):
        spec(o, rs)
        PU.encode_record(eng, recs[i], o)
    eng.set_state_raw(recs)
    dm, am = read_masks(eng, kind, n, L, torch, dev)
    for i, o in enumerate(oracles):
        tag = "%s L=%d constructed env=%d" % (kind, L, i)
        PU.compare_state(tag, eng, eng.get_state_raw(i, 1)[0], o)
        if o.e.n_towers < E.CAP_TOWERS:        # the oracle's list has no such capacity: test_mask_full_tower_list
            check_masks(tag, kind, multi, o, -1, dm[i] if dm is not None else None, am[i] if am is not None else None)
    eng.close()
    return dm, am, oracles


def _down(x):
    return float(np.nextafter(x, -np.inf))


# distinct prices per level, so that the level a summon or an LvUp uses shows in the mask
BOUNDARY_CFG = dict(tower_cost=[[10, 11], [17, 18], [23, 24], [12, 13]], enemy_cost=[[8, 9], [15, 16], [40, 41], [30, 31]],
                    max_episode_steps=100, enemy_upgrade_at=0.75)
UPGRADE_STEP = 75


def _tower_spec(cost_def, lv, **hdr):
    def spec(o, rs):
        loc = PU.free_cells(o)[rs.randint(len(PU.free_cells(o)))]
        PU.construct_state(o, towers=[(0, lv, loc, None)], cost_def=cost_def, **hdr)
    return spec


def _header_spec(**hdr):
    def spec(o, rs):
        PU.construct_state(o, **hdr)
    return spec


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["def", "atk", "2p"])
def test_mask_boundary_states(kind):
    assert E.upgrade_step(100, 0.75) == UPGRADE_STEP
    specs = [
        _header_spec(cost_def=17.0),                          # build type 1 exactly affordable, type 2 not
        _header_spec(cost_def=_down(17.0)),                   # one ulp short of type 1
        _tower_spec(11.0, 0),                                 # LvUp of a type-0 tower exactly affordable
        _tower_spec(_down(11.0), 0),                          # one ulp short
        _tower_spec(1e9, 1),                                  # at max level: LvUp 0, Destruct 1
        _header_spec(cost_def=50.0, defender_cd=0, attacker_cd=0, cost_atk=50.0),
        _header_spec(cost_def=50.0, defender_cd=1, attacker_cd=1, cost_atk=50.0),
        _header_spec(cost_def=50.0, defender_cd=2, attacker_cd=2, cost_atk=50.0),
        _header_spec(cost_atk=15.0, steps=UPGRADE_STEP - 1),  # type 1 at level 0 exactly affordable
        _header_spec(cost_atk=_down(15.0), steps=UPGRADE_STEP - 1),
        _header_spec(cost_atk=16.0, steps=UPGRADE_STEP),      # level 1 prices from the upgrade step on
        _header_spec(cost_atk=_down(16.0), steps=UPGRADE_STEP),
        _header_spec(cost_atk=15.0, steps=UPGRADE_STEP),      # the level-0 price no longer suffices
        _header_spec(cost_def=float("inf"), cost_atk=float("inf")),
        _tower_spec(float("inf"), 0, cost_atk=float("inf"), steps=UPGRADE_STEP + 3),
    ]
    dm, am, oracles = run_constructed(kind, 10, BOUNDARY_CFG, specs)
    cells = 100
    if dm is not None:
        build = dm[:, :4 * cells].reshape(-1, 4, cells)
        assert build[0, 1].any() and not build[0, 2].any() and not build[1, 1].any()
        for i, want in ((2, 1), (3, 0), (4, 0)):
            loc = oracles[i].e.towers[0].loc
            assert dm[i, 4 * cells + loc] == want and dm[i, 5 * cells + loc] == 1
        assert dm[5, :-1].any() and dm[6, :-1].any() and not dm[7, :-1].any()      # defender_cd 0 / 1 act, 2 does not
        assert dm[13, :-1].any()
    if am is not None:
        assert am[5].any() and am[6].any() and not am[7].any()                      # attacker_cd 0 / 1 act, 2 does not
        roads = [1 + i % 3 for i in range(len(specs))]
        assert am[8][:, 1].tolist() == [1 if r < roads[8] else 0 for r in range(3)]
        assert not am[9][:, 1].any() and am[10][:, 1].any() and not am[11][:, 1].any() and not am[12][:, 1].any()
        assert am[13].sum() == 4 * roads[13]


@pytest.mark.gpu
@pytest.mark.parametrize("distance", [0, 8])
def test_mask_tower_distance(distance):
    def spec(o, rs):
        free = PU.free_cells(o)
        PU.construct_state(o, towers=[(1, 0, free[len(free) // 2], None)], cost_def=40.0)
    run_constructed("2p", 10, dict(tower_distance=distance), [spec, spec, spec], seed=distance)


@pytest.mark.gpu
def test_mask_full_tower_list():
    """32 towers: every build is 0 although purse and position allow it, and the step agrees."""
    import torch

    def spec(o, rs):
        free = PU.free_cells(o)
        PU.construct_state(o, towers=[(k % 4, k % 2, free[k], None) for k in range(E.CAP_TOWERS)], cost_def=90.0)
    dm, _, oracles = run_constructed("def", 10, dict(tower_distance=0), [spec, spec], seed=4)
    cells = 100
    for i, o in enumerate(oracles):
        free = PU.free_cells(o)
        assert free and not dm[i, :4 * cells].any()
        for k in range(E.CAP_TOWERS):
            t = o.e.towers[k]
            assert dm[i, 5 * cells + t.loc] == 1 and dm[i, 4 * cells + t.loc] == (1 if t.lv == 0 else 0)
    # the step itself: a build on a free cell comes back as the no-op
    cfg = PU.make_config(tower_distance=0)
    eng = E.Engine("def", 10, 1, cfg=cfg)
    maps = _maps_with_roads(10, [1], 1000 + 4)
    eng.upload_maps(maps)
    eng.reset()
    o = PU.oracle_env_from_map(maps[0], PU.oracle_config_from_engine(cfg))
    spec(o, None)
    rec = eng.get_state_raw()
    PU.encode_record(eng, rec[0], o)
    eng.set_state_raw(rec)
    act = torch.tensor([PU.free_cells(o)[0]], dtype=torch.int64, device="cuda")
    real = torch.zeros(1, dtype=torch.int64, device="cuda")
    eng.step(E.Engine.make_io(def_action=act, real_def=real))
    assert int(real[0]) == 6 * cells
    eng.close()


# ------------------------------------------------------------------------------------------------
# The mask changes nothing

@pytest.mark.gpu
@pytest.mark.parametrize("kind,multi", [("def", False), ("def", True), ("atk", False), ("2p", False), ("2p", True)])
def test_mask_changes_nothing(kind, multi):
    import torch
    from gym_td_b200.vec_env import TDVecEnv
    n, L = 64, 10
    envs = [TDVecEnv(kind, L, n, seed=9, multi_action=multi, cfg=PU.make_config(max_episode_steps=20)) for _ in range(2)]
    rs = np.random.RandomState(1)
    for e in envs:
        e.reset()
    envs[0].action_mask()
    for step in range(45):
        d = torch.from_numpy(rs.randint(0, 3, size=(n, 6, L, L)) * (rs.random_sample((n, 6, L, L)) < 0.02)
                             if multi else rs.randint(0, 6 * L * L + 1, size=n)).to("cuda")
        a = torch.from_numpy(np.stack([PU.attacker_action(rs) for _ in range(n)])).to("cuda")
        act = {"def": d, "atk": a, "2p": {"Attacker": a, "Defender": d}}[kind]
        outs = []
        for k, e in enumerate(envs):
            obs, rew, done, info = e.step(act)
            if k == 0:
                e.action_mask()
            torch.cuda.synchronize()
            outs.append((obs.cpu().numpy().copy(), rew.cpu().numpy().copy(), done.cpu().numpy().copy(),
                         e._slab.cpu().numpy().copy(), e.engine.get_state_raw()))
        for x, y in zip(outs[0], outs[1]):
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), "step %d" % step
    assert envs[0].stats() == envs[1].stats()


# ------------------------------------------------------------------------------------------------
# Buffers and API

@pytest.mark.gpu
@pytest.mark.parametrize("kind,L,n", [("2p", 10, 7), ("2p", 13, 5), ("def", 30, 3), ("atk", 20, 6)])
def test_mask_unaligned_buffers(kind, L, n):
    """Output pointers 1 byte past an aligned address, batch sizes that are not a multiple of 4: the same bytes, and
    nothing outside the rows is written."""
    import torch
    from gym_td_b200.vec_env import TDVecEnv
    env = TDVecEnv(kind, L, n, seed=3)
    env.reset()
    rs = np.random.RandomState(2)
    for _ in range(15):
        d = torch.from_numpy(rs.randint(0, 6 * L * L + 1, size=n)).to("cuda")
        a = torch.from_numpy(np.stack([PU.attacker_action(rs) for _ in range(n)])).to("cuda")
        env.step({"def": d, "atk": a, "2p": {"Attacker": a, "Defender": d}}[kind])
    m = env.action_mask()
    ref = {"def": (m, None), "atk": (None, m), "2p": (m.get("Defender"), m.get("Attacker")) if kind == "2p" else None}[kind]
    ref_d, ref_a = [x.to(torch.uint8).cpu().numpy().reshape(n, -1) if x is not None else None for x in ref]
    R = 6 * L * L + 1
    for off in (1, 3, 8, 15):
        bd = torch.full((n * R + 64,), 0xAB, dtype=torch.uint8, device="cuda")
        ba = torch.full((n * 12 + 64,), 0xAB, dtype=torch.uint8, device="cuda")
        env.engine.action_mask(bd.data_ptr() + off if ref_d is not None else None,
                               ba.data_ptr() + off if ref_a is not None else None,
                               torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        for buf, want, w in ((bd, ref_d, R), (ba, ref_a, 12)):
            h = buf.cpu().numpy()
            if want is None:
                assert (h == 0xAB).all()
                continue
            assert np.array_equal(h[off:off + n * w].reshape(n, w), want), "offset %d" % off
            assert (h[:off] == 0xAB).all() and (h[off + n * w:] == 0xAB).all(), "offset %d: bytes outside the rows" % off


@pytest.mark.gpu
def test_mask_facades_match_vec_env():
    import torch
    from gym_td_b200 import envs as G
    from gym_td_b200 import params
    from gym_td_b200.vec_env import TDVecEnv

    def compare(f, kind, multi):
        vec = TDVecEnv(kind, f.map_size, 1, seed=0, multi_action=multi)
        vec.engine.set_state_raw(f._engine.get_state_raw())
        got, want = f.action_mask(), vec.action_mask()
        torch.cuda.synchronize()
        if kind == "2p":
            for side in ("Attacker", "Defender"):
                assert np.array_equal(got[side], want[side][0].cpu().numpy())
        else:
            assert np.array_equal(got, want[0].cpu().numpy())
        assert got is not None
        vec.close()

    rs = np.random.RandomState(5)
    for cls, kind in ((G.TDDefense, "def"), (G.TDAttack, "atk"), (G.TDMulti, "2p")):
        f = cls(10, seed=3)
        for _ in range(12):
            compare(f, kind, False)
            f.step(f.action_space.sample() if kind != "2p" else {"Attacker": PU.attacker_action(rs),
                                                                 "Defender": int(rs.randint(601))})
        f.close()
    # the hyper parameters refuse assignment (as the reference's do); the multi-action façade is set up behind that
    old = params.hyper_parameters.allow_multiple_actions
    object.__setattr__(params.hyper_parameters, "allow_multiple_actions", True)
    try:
        f = G.TDDefense(10, seed=4)
        for _ in range(8):
            m = f.action_mask()
            assert m.shape == (6, 10, 10) and m.dtype == bool
            compare(f, "def", True)
            f.step(PU.sparse_multi_action(10, rs, p=0.05))
        f.close()
    finally:
        object.__setattr__(params.hyper_parameters, "allow_multiple_actions", old)


@pytest.mark.gpu
def test_mask_api_errors():
    import torch
    buf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    eng = E.Engine("def", 10, 4)
    with pytest.raises(E.TdError) as ei:                      # before any map was uploaded and the envs reset
        eng.action_mask(def_mask=buf)
    assert ei.value.code == -4
    eng.upload_maps(mapgen.generate_batch(np.arange(4, dtype=np.uint32), 10)[0])
    eng.reset()
    for kw in (dict(atk_mask=buf), dict(def_mask=buf, atk_mask=buf), dict()):
        with pytest.raises(E.TdError) as ei:
            eng.action_mask(**kw)
        assert ei.value.code == -1
    eng.action_mask(def_mask=buf)
    eng.close()
    eng = E.Engine("atk", 10, 4)
    eng.upload_maps(mapgen.generate_batch(np.arange(4, dtype=np.uint32), 10)[0])
    eng.reset()
    with pytest.raises(E.TdError) as ei:
        eng.action_mask(def_mask=buf)
    assert ei.value.code == -1
    eng.action_mask(atk_mask=buf)
    eng.close()


def test_mask_no_cpu_fallback():
    """Without a CUDA device there is no handle to mask: creating one fails with TD_E_CUDA, and the entry point
    itself refuses a missing handle."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert hasattr(E.lib(), "td_action_mask") and "td_action_mask" in E.EXPORTS
    assert E.lib().td_action_mask(None, None, None, None) == -1
    with pytest.raises(E.TdError) as ei:
        E.Engine("2p", 10, 4)
    assert ei.value.code == -2 and "no CPU fallback" in str(ei.value)
    from gym_td_b200.vec_env import TDVecEnv
    with pytest.raises(E.TdError) as ei:
        TDVecEnv("def", 10, 4).action_mask()
    assert ei.value.code == -2
