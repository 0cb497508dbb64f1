"""GPU: the observation writer and the step from constructed board states.

Play almost never reaches the states where the observation writer and the list paths are easiest to get wrong:
crowded (cell, type) groups whose members have distinct LP ratios, list lengths at the edges of the speculative
prefetch, equal sort keys, exact boundaries of the scalar planes, plane values that overflow float32.  Each family
below builds such states through the oracle's own API (tests/parity_util.py: construct_state), writes them into
the CUDA env records (encode_record, td_set_state) and checks, bit for bit against the oracle:
- td_observe (float32) into the step's buffer and into one 4 bytes off the 16-byte boundary (the scalar stores);
- td_observe_as bfloat16 / uint8 against an independent NumPy conversion of the oracle's float32 planes;
- td_observe_snapshot of a td_snapshot taken from the same state, for a record count that is not a multiple of 4;
- 40 steps from the state through run_parity: the fused kernel's observation, rules, record and statistics.

Every family runs over LEGS: boards 10 / 20 / 30 and the run-time sizes 13 / 15, the three env kinds, Discrete and
multi-action defenders, full and in-place (incremental) observations, aligned and misaligned step buffers.
"""
import math

import numpy as np
import pytest

from gym_td_b200 import engine as E
from gym_td_b200 import mapgen
from tests import parity_util as PU

pytestmark = pytest.mark.gpu

STEPS = 40
T4 = lambda a, b=None: [[a, a if b is None else b]] * 4          # noqa: E731 -- one value for every (type, lv)
DPR, DPC = (0, 0, 1, -1), (1, -1, 0, 0)                          # movement by direction code (TDBoard.py:319-346)

# (kind, L, multi-action, incremental observation, obs_offset in float32 elements)
LEGS = [
    ("def", 10, False, False, 0),
    ("atk", 10, False, True, 0),
    ("2p", 10, True, False, 1),        # step kernel writing a misaligned buffer: scalar stores at L = 10
    ("def", 20, True, True, 0),
    ("2p", 20, False, False, 0),
    ("atk", 30, False, True, 1),       # in-place update asked for on a misaligned buffer: full write, scalar stores
    ("def", 30, True, False, 0),
    ("atk", 13, False, False, 0),      # run-time board size
    ("2p", 15, True, False, 0),        # odd board size: L * L not a multiple of 4
    ("def", 15, False, False, 1),
]


def _leg_id(leg):
    kind, L, multi, inc, off = leg
    return "%s-L%d%s%s%s" % (kind, L, "-multi" if multi else "", "-inc" if inc else "", "-off4" if off else "")


# ------------------------------------------------------------------------------------------------ state helpers

def _max_lp(o, t, lv):
    return o.e.cfg.enemy_LP[t][lv]


def _ratio32(o, t, lv, LP):
    return np.float32(LP / _max_lp(o, t, lv))


def _tower_cells(o, n, near=None, rs=None):
    """n cells for towers built in this order: off the road and outside the diamonds (tower_distance) of the ones
    before; nearest to `near` (Chebyshev) first, or shuffled by rs."""
    e = o.e
    L, D = e.L, e.cfg.tower_distance
    blocked = np.ctypeslib.as_array(e.map6)[:L * L] > 0
    cand = np.flatnonzero(~blocked).tolist()
    if near is not None:
        nr, nc = divmod(near, L)
        cand.sort(key=lambda c: (max(abs(c // L - nr), abs(c % L - nc)), c))
    elif rs is not None:
        rs.shuffle(cand)
    out = []
    for c in cand:
        if blocked[c]:
            continue
        out.append(c)
        r0, c0 = divmod(c, L)
        for i in range(-D, D + 1):
            for j in range(-D, D + 1):
                if abs(i) + abs(j) <= D and 0 <= r0 + i < L and 0 <= c0 + j < L:
                    blocked[(r0 + i) * L + c0 + j] = True
        if len(out) == n:
            return out
    raise AssertionError("the map has room for %d towers, %d wanted" % (len(out), n))


def _group_order_matters(ratios32):
    """True when summing the float32 ratios in list order gives another mean than in reverse or sorted order."""
    def mean(seq):
        s = np.float32(0)
        for r in seq:
            s = np.float32(s + r)
        return np.float32(s / np.float32(len(seq)))
    m = mean(ratios32)
    return m != mean(ratios32[::-1]) and m != mean(sorted(ratios32))


def _crowd_ratios(rs, size):
    """Distinct non-dyadic ratios in (0, 1) per group; groups of 3+ members get ratios whose float32 mean depends
    on the summation order."""
    while True:
        r = [np.float32(x) for x in rs.uniform(0.01, 1.0, size)]
        if len(set(r)) == size and (size < 3 or _group_order_matters(r)):
            return r


def _next_to_end(o):
    """A road cell whose next step (its direction) is the end cell."""
    e = o.e
    L = e.L
    for c in PU.road_cells(o):
        d = e.dir[c]
        if (c // L + DPR[d]) * L + c % L + DPC[d] == e.end:
            return c
    raise AssertionError("no road cell leads to the end")


# ------------------------------------------------------------------------------------------------ families
# A family: (config overrides, n_envs, build(o, i, rs) -> (towers, enemies, header, ep), coverage check)

def crowd_sizes(L):
    # 8 / 32: the one-warp __match_any_sync fold (L = 10 holds at most 32); 33 / 64: the multi-pass fold (L >= 20)
    return (8, 32) if L == 10 else (8, 32, 33, 64)


def build_crowd(o, i, rs):
    """One road cell holding 8 / 32 / 33 / 64 enemies: the four types and both levels interleaved in the list, every
    (cell, type) group with distinct non-dyadic LP ratios whose float32 mean depends on the summation order
    (obs_sparse_enemies, both folds).  Four towers next to it, one of each type, splash and freeze included."""
    L = o.e.L
    sizes = crowd_sizes(L)
    n = sizes[i % len(sizes)]
    rc = PU.road_cells(o)
    cell = rc[len(rc) // 2]
    per_type = [[k for k in range(n) if k % 4 == t] for t in range(4)]
    enemies = [None] * n
    for t in range(4):
        ratios = _crowd_ratios(rs, len(per_type[t]))
        for j, k in enumerate(per_type[t]):
            lv = (k // 4) % 2
            LP = float(ratios[j]) * _max_lp(o, t, lv)
            enemies[k] = (t, lv, cell, float(rs.choice([0.0, 0.25, 0.5])), LP, int(rs.randint(0, 3)))
    towers = [(t, t % 2, c, None) for t, c in enumerate(_tower_cells(o, 4, near=cell))]
    return towers, enemies, dict(cost_def=30.0), None


def check_crowd(built, L):
    ne = sorted(set(b["n_enemies"] for b in built))
    assert ne == list(crowd_sizes(L)), ne
    assert max(b["max_group"] for b in built) == max(crowd_sizes(L)) // 4 + (1 if max(crowd_sizes(L)) % 4 else 0)
    assert any(b["order_sensitive_groups"] for b in built)


def build_towers32(o, i, rs):
    """32 towers, every (type, lv), cd 0 / fractional / equal to the interval (the tower list at its capacity:
    the speculative prefix plus the second fetch, the tower one-hots, the firing loop), six enemies in range."""
    cells = _tower_cells(o, 32, rs=rs)
    towers = []
    for k, c in enumerate(cells):
        cd = (0.0, 0.37 + 0.01 * k, "intv")[k % 3]
        towers.append((k % 4, (k // 4) % 2, c, cd))
    rc = PU.road_cells(o)
    enemies = [(int(rs.randint(4)), int(rs.randint(2)), rc[int(rs.randint(len(rc)))], float(rs.uniform(0, 1)),
                None, 0) for _ in range(6)]
    return towers, enemies, dict(cost_def=0.0), None


def check_towers32(built, L):
    assert all(b["n_towers"] == 32 for b in built)
    assert {b["tower_kinds"] for b in built} == {8}


PREFETCH = [(12, 8), (13, 9), (16, 8), (17, 9), (12, 9), (13, 8), (16, 9), (17, 8)]


def build_prefetch(o, i, rs):
    """List lengths at the edges of the speculative prefetch (12 towers / 8 enemies in the first round trip): one
    element more on either list sends the env through the second fetch (finish_env_load)."""
    nt, ne = PREFETCH[i % len(PREFETCH)]
    towers = [(int(rs.randint(4)), int(rs.randint(2)), c, float(rs.uniform(0, 3))) for c in _tower_cells(o, nt, rs=rs)]
    rc = PU.road_cells(o)
    enemies = []
    for _ in range(ne):
        t, lv = int(rs.randint(4)), int(rs.randint(2))
        enemies.append((t, lv, rc[int(rs.randint(len(rc)))], float(rs.uniform(0, 1)),
                        float(rs.uniform(0.01, 1)) * _max_lp(o, t, lv), int(rs.randint(0, 3))))
    return towers, enemies, dict(cost_def=15.0, cost_atk=20.0), None


def check_prefetch(built, L):
    assert {(b["n_towers"], b["n_enemies"]) for b in built} == set(PREFETCH)


def build_ties(o, i, rs):
    """Equal sort keys (dist - margin) in scrambled list order: five enemies on one cell with one margin, and pairs
    on different cells of equal dist.  The stable sort keeps list order among them and the single-target towers
    next to the cell hit the first one (the sort in board_step, the targeting scan)."""
    e = o.e
    rc = PU.road_cells(o)
    cell = rc[len(rc) // 3]
    same = [(int(t), int(rs.randint(2)), cell, 0.5) for t in rs.permutation([0, 1, 2, 3, 1])]
    by_dist = {}
    for c in rc:
        by_dist.setdefault(e.dist[c], []).append(c)
    pairs = [cs[:2] for cs in by_dist.values() if len(cs) >= 2][:2]
    more = [(int(rs.randint(4)), int(rs.randint(2)), c, 0.25) for cs in pairs for c in cs]
    spec = same + more
    order = rs.permutation(len(spec))
    enemies = []
    for k in order:
        t, lv, c, m = spec[k]
        enemies.append((t, lv, c, m, float(rs.uniform(0.3, 1)) * _max_lp(o, t, lv), 0))
    towers = [(t, 0, c, 0.0) for t, c in zip((0, 1, 3), _tower_cells(o, 3, near=cell))]
    return towers, enemies, dict(cost_def=12.0, cost_atk=10.0), None


def check_ties(built, L):
    assert all(b["max_group"] >= 2 and b["n_enemies"] >= 5 for b in built)


def build_scalars(o, i, rs):
    """Exact boundaries of the broadcast planes and the header scalars (obs_prepare, the cooldown / AllowNextMove
    bits, the summon level, the episode end, the leak that ends it, margins and LP at their extremes)."""
    e, cfg = o.e, o.e.cfg
    v = i % 10
    rc = PU.road_cells(o)
    towers = [(0, 0, c, 0.0) for c in _tower_cells(o, 2, rs=rs)]
    enemies = [(1, 0, rc[len(rc) // 2], 0.5, None, 0)]
    h = dict(cost_def=20.0, cost_atk=50.0)
    if v == 0:
        h["cost_def"] = cfg.tower_cost[0][0]                                  # buildable plane 21: the >= holds
    elif v == 1:
        h["cost_def"] = math.nextafter(cfg.tower_cost[1][0], -math.inf)       # ... one ulp below: it does not
    elif v == 2:
        h["cost_def"] = h["cost_atk"] = cfg.max_cost                          # planes 11 / 12 at exactly 1
    elif v == 3:
        h["steps"] = E.upgrade_step(cfg.max_episode_steps, cfg.enemy_upgrade_at) - 1   # next summons: level 0, then 1
    elif v == 4:
        h["steps"] = cfg.max_episode_steps - 1                                # the next step ends the episode
    elif v == 5:
        h.update(defender_cd=0, attacker_cd=1)
    elif v == 6:
        h.update(defender_cd=2, attacker_cd=2)
    elif v == 7:
        h.update(defender_cd=1, attacker_cd=0)
    elif v == 8:
        # the last base point and an enemy one cell from the end, one ulp short of moving: it leaks on the next step
        enemies = [(0, 0, _next_to_end(o), math.nextafter(1.0, 0.0), None, 0)]
        h["base_LP"] = 1
    else:
        # margin one ulp below 1.0, LP one ulp above 0 (ratio 0 in float32) and LP = maxLP, slowdowns 0 / 1 / frozen
        c = rc[len(rc) // 2]
        enemies = [(2, 0, c, math.nextafter(1.0, 0.0), 5e-324, cfg.frozen_time),
                   (2, 1, c, 0.0, None, 1), (2, 0, c, math.nextafter(1.0, 0.0), None, 0),
                   (3, 1, rc[0], math.nextafter(1.0, 0.0), math.nextafter(0.0, 1.0), 0)]
    return towers, enemies, h, None


def check_scalars(built, L):
    assert len(built) == 10


def build_divisors(o, i, rs):
    """A few towers and enemies under the divisor edge configs: planes 11-12 / 41-44 that overflow float32 to inf,
    underflow to 0 or land on large finite values (the f64 quotient rounded once, u8 / bf16 saturation)."""
    rc = PU.road_cells(o)
    towers = [(int(rs.randint(4)), 0, c, 0.0) for c in _tower_cells(o, 3, rs=rs)]
    enemies = [(int(rs.randint(4)), 0, rc[int(rs.randint(len(rc)))], 0.0, None, 0) for _ in range(4)]
    return towers, enemies, dict(cost_def=10.0, cost_atk=3.0), None


def check_divisors(built, L):
    assert any(b["inf_planes"] for b in built)


# max_cost down to the smallest subnormal and up to the largest double; enemy costs from 1e-300 to 1e300
DIVISOR_TINY = dict(max_cost=5e-324, enemy_cost=[[1e-9, 1e-9], [1e-300, 1e-300], [1e300, 1e300], [2.5, 2.5]])
DIVISOR_HUGE = dict(max_cost=1.7976931348623157e308, defender_init_cost=1e308,
                    enemy_cost=[[1e-300, 8], [3.0, 15], [1e-9, 40], [7.0, 30]])

# no summon ever succeeds (no income, empty purse): the crowded lists are the ones compared, step after step
NO_INCOME = dict(attacker_init_cost=0.0, attacker_cost_init_rate=0.0, attacker_cost_final_rate=0.0)

FAMILIES = {
    "crowd": (dict(NO_INCOME, tower_distance=1), 8, build_crowd, check_crowd),
    "towers32": (dict(tower_distance=0), 6, build_towers32, check_towers32),
    "prefetch": (dict(tower_distance=0), 8, build_prefetch, check_prefetch),
    "ties": (dict(tower_distance=1), 6, build_ties, check_ties),
    "scalars": (dict(max_episode_steps=120, enemy_upgrade_at=0.5), 10, build_scalars, check_scalars),
    "divisor_tiny": (DIVISOR_TINY, 5, build_divisors, check_divisors),
    "divisor_huge": (DIVISOR_HUGE, 5, build_divisors, check_divisors),
}


# ------------------------------------------------------------------------------------------------ independent references

def bf16_reference(f32):
    """float32 -> bfloat16 bits, round to nearest even on the uint32 bits (no NaN reaches the observation)."""
    assert not np.isnan(f32).any()
    u = f32.view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def u8_reference(f32):
    """obs_u8: rint(min(255 v, 255)) in float32; inf -> 255, NaN -> 255 (fminf), negative values -> 0."""
    v = (f32.astype(np.float32) * np.float32(255)).astype(np.float32)
    v = np.where(np.isnan(v), np.float32(255), np.minimum(v, np.float32(255)))
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


def check_views(eng, oracles, L):
    """The constructed states through every other observation path, against the oracle."""
    import torch
    n = len(oracles)
    want = np.stack([o.get_states() for o in oracles])
    stream = torch.cuda.current_stream().cuda_stream
    buf = torch.empty(n * 45 * L * L + 1, dtype=torch.float32, device="cuda")
    mis = buf[1:].view(n, 45, L, L)
    assert mis.data_ptr() % 16 == 4
    eng.observe(mis, stream)
    torch.cuda.synchronize()
    got = mis.cpu().numpy()
    for i in range(n):
        assert np.array_equal(got[i].view(np.uint32), want[i].view(np.uint32)), "misaligned td_observe env %d" % i
    if L in (10, 20, 30):
        bf = torch.empty((n, 45, L, L), dtype=torch.bfloat16, device="cuda")
        u8 = torch.empty((n, 45, L, L), dtype=torch.uint8, device="cuda")
        eng.observe(bf, stream, "bf16")
        eng.observe(u8, stream, "u8")
        torch.cuda.synchronize()
        got_bf = bf.view(torch.int16).cpu().numpy().view(np.uint16)
        got_u8 = u8.cpu().numpy()
        for i in range(n):
            bad = np.argwhere(got_bf[i] != bf16_reference(want[i]))
            assert not len(bad), "bf16 env %d differs at (plane, r, c) %s" % (i, bad[:4].tolist())
            bad = np.argwhere(got_u8[i] != u8_reference(want[i]))
            assert not len(bad), "u8 env %d differs at (plane, r, c) %s" % (i, bad[:4].tolist())
    rb = eng.layout.record_bytes
    recs = torch.empty((n, rb), dtype=torch.uint8, device="cuda")
    eng._check(eng._lib.td_snapshot(eng._h, recs.data_ptr(), stream))
    k = n - 1 if (n - 1) % 4 else n - 2                     # not a multiple of 4
    out = torch.empty((k, 45, L, L), dtype=torch.float32, device="cuda")
    eng._check(eng._lib.td_observe_snapshot(eng._h, recs.data_ptr(), k, out.data_ptr(), stream))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    for i in range(k):
        assert np.array_equal(got[i].view(np.uint32), want[i].view(np.uint32)), "td_observe_snapshot env %d" % i


def _summary(o, towers):
    e = o.e
    groups = {}
    for x in e.enemies[:e.n_enemies]:
        groups.setdefault((x.loc, x.type), []).append(x)
    sensitive = 0
    for (loc, t), xs in groups.items():
        if len(xs) >= 3:
            lvs = [o.enemy_lv[k] for k in range(e.n_enemies) if (e.enemies[k].loc, e.enemies[k].type) == (loc, t)]
            r = [_ratio32(o, t, lv, x.LP) for x, lv in zip(xs, lvs)]
            sensitive += _group_order_matters(r)
    st = o.get_states()
    return dict(n_towers=e.n_towers, n_enemies=e.n_enemies, max_group=max((len(v) for v in groups.values()), default=0),
                order_sensitive_groups=sensitive, tower_kinds=len({(t, lv) for t, lv, _, _ in towers}),
                inf_planes=int(np.isinf(st).any()))


def run_family(name, leg):
    ov, n_envs, build, check = FAMILIES[name]
    kind, L, multi, inc, off = leg
    built = []

    def prepare(i, o, rs):
        towers, enemies, header, ep = build(o, i, rs)
        if any(cd == "intv" for _, _, _, cd in towers):
            tw = [(t, lv, c, None if cd == "intv" else cd) for t, lv, c, cd in towers]
            PU.construct_state(o, tw, enemies, **header)
            for k, (_, _, _, cd) in enumerate(towers):
                if cd == "intv":
                    o.e.towers[k].cd = o.e.towers[k].intv
        else:
            PU.construct_state(o, towers, enemies, **header)
        built.append(_summary(o, towers))
        return ep

    n = PU.run_parity(kind, L, n_envs, STEPS, seed=sum(map(ord, name)) + L, multi=multi,
                      opponent="none" if kind == "2p" else "device", cfg_overrides=ov, incremental=inc,
                      obs_offset=off, past_done=STEPS, overflow="expect", prepare=prepare,
                      inspect=lambda eng, oracles: check_views(eng, oracles, L))
    assert len(built) == n_envs
    check(built, L)
    assert n >= n_envs * 5, n
    return built


@pytest.mark.parametrize("leg", LEGS, ids=_leg_id)
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_constructed_state(name, leg):
    run_family(name, leg)


# ------------------------------------------------------------------------------------------------ records the kernels cannot run

def _engine_with_record(L, kind="def"):
    import torch
    cfg = PU.make_config()
    eng = E.Engine(kind, L, 2, cfg=cfg)
    seeds = np.array([3, 4], dtype=np.uint32)
    maps, _, _ = mapgen.generate_batch(seeds, L)
    eng.upload_maps(maps)
    obs = torch.empty((2, 45, L, L), dtype=torch.float32, device="cuda")
    eng.reset(obs=obs)
    torch.cuda.synchronize()
    return eng, maps, PU.oracle_config_from_engine(cfg), obs


def test_set_state_rejects_records_the_step_kernels_cannot_run():
    """td_set_state refuses what no step could hold or walk: more enemies than the step kernel of the board holds
    (32 at L = 10), an enemy off the road or on the end cell, a tower on the road.  The refused record is not
    written; no step is launched on it.  The same lists inside the limits are accepted and observed exactly."""
    import torch
    for L in (10, 20):
        eng, maps, ocfg, obs = _engine_with_record(L)
        base = eng.get_state_raw()

        def record(n_enemies, o=None):
            o = o or PU.oracle_env_from_map(maps[0], ocfg)
            rc = PU.road_cells(o)
            PU.construct_state(o, [(0, 0, _tower_cells(o, 1, rs=np.random.RandomState(1))[0], 0.0)],
                               [(k % 4, 0, rc[k % len(rc)], 0.0, None, 0) for k in range(n_enemies)])
            rec = base.copy()
            PU.encode_record(eng, rec[0], o)
            return rec, o

        def refused(rec):
            before = eng.get_state_raw()
            with pytest.raises(E.TdError) as ei:
                eng.set_state_raw(rec)
            assert ei.value.code == -1
            assert np.array_equal(eng.get_state_raw(), before), "a refused record was written"

        cap = PU.enemy_capacity(L)
        rec, o = record(cap)
        eng.set_state_raw(rec)                                   # at the capacity: accepted, observed exactly
        eng.observe(obs)
        torch.cuda.synchronize()
        assert np.array_equal(obs[0].cpu().numpy().view(np.uint32), o.get_states().view(np.uint32))
        if L == 10:
            refused(record(33)[0])                               # one more than the 10x10 step kernel holds
        else:
            assert cap == 64
        lay = eng.layout
        rec, o = record(4)
        en = rec[0][lay.off_enemies:lay.off_enemies + 24 * 4].view(E.ENEMY_DTYPE)
        road = np.ctypeslib.as_array(o.e.road)[:L * L] & 1
        off_road = int(np.flatnonzero(road == 0)[0])
        bad = rec.copy()
        bad[0][lay.off_enemies:lay.off_enemies + 24 * 4].view(E.ENEMY_DTYPE)[2]["loc"] = off_road
        refused(bad)
        bad = rec.copy()
        bad[0][lay.off_enemies:lay.off_enemies + 24 * 4].view(E.ENEMY_DTYPE)[0]["loc"] = o.e.end
        refused(bad)
        bad = rec.copy()
        bad[0][lay.off_towers:lay.off_towers + 16].view(E.TOWER_DTYPE)[0]["loc"] = int(en[1]["loc"])
        refused(bad)
        eng.set_state_raw(rec)                                   # the unpatched record is fine
        eng.close()


# ------------------------------------------------------------------------------------------------ episode counters

# every attacker slot summons, enemies cost next to nothing and outrun any road: each summoned enemy leaks within
# its step (24 a step on a three-road map), and nothing ends the episode but its length
LEAKY = dict(base_LP=None, enemy_cost=T4(1e-9), enemy_speed=T4(128.0))


def _all_slots(rs):
    return np.zeros((3, 8), dtype=np.int64)


def test_episode_counters_cross_16_bits_from_a_constructed_header():
    """ep_kills / ep_leaks of a record just below 65,536 stepped past it: td_get_stats keeps counting (32-bit header).
    Enemies of 1 LP and four towers at the first start cell make the kills; the rest leak."""
    def prepare(i, o, rs):
        cells = _tower_cells(o, 4, near=o.e.start[0])
        PU.construct_state(o, [(t, 0, c, 0.0) for t, c in zip((0, 2, 1, 2), cells)])
        return (0.0, 65533, 65530)

    PU.run_parity("atk", 10, 4, 40, seed=5, cfg_overrides=dict(LEAKY, max_episode_steps=40, enemy_LP=T4(1.0)),
                  prepare=prepare, atk_policy=_all_slots, overflow="expect")
    assert PU.LAST_RUN["episodes"] == 4, PU.LAST_RUN
    assert PU.LAST_RUN["max_ep_leaks"] > 65535 and PU.LAST_RUN["max_ep_kills"] > 65535, PU.LAST_RUN


def test_episode_counters_of_a_long_episode():
    """One episode that really leaks more than 65,535 enemies (3,000 steps; seed 5 gives two maps with three roads,
    24 leaks a step): td_get_stats matches the oracle's count.  The enemies' LP is out of reach of the scripted
    defender's towers."""
    PU.run_parity("atk", 10, 4, 3000, seed=5, cfg_overrides=dict(LEAKY, max_episode_steps=3000, enemy_LP=T4(1e9)),
                  atk_policy=_all_slots, overflow="expect", check_state_every=50)
    assert PU.LAST_RUN["episodes"] == 4 and PU.LAST_RUN["max_ep_leaks"] > 65535, PU.LAST_RUN


# ------------------------------------------------------------------------------------------------ zero divisors

@pytest.mark.parametrize("ov", [dict(max_cost=0.0), dict(max_cost=-5.0), dict(max_cost=float("nan")),
                                dict(enemy_cost=[[8, 8], [15, 15], [0.0, 40], [30, 30]]),
                                dict(enemy_cost=[[8, 8], [15, 15], [40, 40], [float("nan"), 30]])],
                         ids=["max_cost_0", "max_cost_negative", "max_cost_nan", "enemy_cost_0", "enemy_cost_nan"])
def test_configs_with_zero_divisors_are_rejected(ov):
    """Planes 11-12 divide by max_cost and 41-44 by enemy_cost[t][0]; the reference raises ZeroDivisionError there,
    so td_create and td_set_config refuse such configs (TD_E_INVALID) instead of writing NaN planes."""
    with pytest.raises(E.TdError) as ei:
        E.Engine("def", 10, 2, cfg=PU.make_config(**ov))
    assert ei.value.code == -1
    eng = E.Engine("def", 10, 2, cfg=PU.make_config())
    with pytest.raises(E.TdError):
        eng.set_config(PU.make_config(**ov))
    eng.close()


def test_level_one_enemy_cost_of_zero_is_accepted():
    """Only the level-0 cost divides (planes 41-44); a free level-1 enemy is a config the reference runs."""
    n = PU.run_parity("def", 10, 4, 30, seed=2, cfg_overrides=dict(enemy_cost=[[8, 0], [15, 0], [40, 0], [30, 0]],
                                                                   enemy_upgrade_at=0.0), overflow="expect")
    assert n > 0
