"""Drive the UNMODIFIED reference (gym_TD) for parity checks and golden-vector generation.

TEST INFRASTRUCTURE ONLY.  Restates only the ~20 wrapper lines the reference cannot
execute itself (SURVEY.md 9.6-9.8); everything else calls the reference's own code.
"""
import random

import numpy as np

from . import ref_loader

MAPGEN_BUDGET = 100000  # randint calls per reset; beyond it the seed is "invalid" (SURVEY 9.8)


def _seeding():
    ref_loader.load()
    from gym.utils import seeding
    return seeding


def set_multiple_actions(flag):
    """hyper_parameters is frozen (TDParam.py:112-113); poke __dict__ as SURVEY 9.6 describes."""
    ref_loader.load()
    from gym_TD.envs.TDParam import hyper_parameters
    hyper_parameters.__dict__["allow_multiple_actions"] = bool(flag)


def set_max_episode_steps(n):
    """hyper_parameters.max_episode_steps, poked like allow_multiple_actions; returns the previous value."""
    ref_loader.load()
    from gym_TD.envs.TDParam import hyper_parameters
    old = hyper_parameters.__dict__["max_episode_steps"]
    hyper_parameters.__dict__["max_episode_steps"] = int(n)
    return old


def ref_config():
    ref_loader.load()
    from gym_TD.envs.TDParam import config
    return config


class ref_config_override(object):
    """with ref_config_override(base_LP=None): ...  restores the reference config on exit."""

    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        cfg = ref_config()
        self.saved = {k: getattr(cfg, k) for k in self.kw}
        for k, v in self.kw.items():
            setattr(cfg, k, v)
        return cfg

    def __exit__(self, *a):
        cfg = ref_config()
        for k, v in self.saved.items():
            setattr(cfg, k, v)


def make_env(kind, map_size, seed, difficulty=1, random_agent=True):
    """Construct a reference env; returns None if `seed` is invalid under the seed-skip rule."""
    ref_loader.load()
    from gym_TD.envs import TDDefense, TDAttack, TDMulti
    seeding = _seeding()
    seeding.DRAW_BUDGET = MAPGEN_BUDGET
    try:
        if kind == "def":
            env = TDDefense(map_size, difficulty=difficulty, seed=seed, random_agent=random_agent)
        elif kind == "atk":
            env = TDAttack(map_size, difficulty=difficulty, seed=seed, random_agent=random_agent)
        else:
            env = TDMulti(map_size, seed=seed, random_agent=random_agent)
    except (ValueError, IndexError, seeding.BudgetExceeded):
        return None
    finally:
        seeding.DRAW_BUDGET = None
    env.np_random.budget = None
    return env


def first_valid_seed(kind, map_size, seed, **kw):
    while True:
        env = make_env(kind, map_size, seed, **kw)
        if env is not None:
            return seed, env
        seed += 1


def generate_roads(map_size, seed, num_roads=None):
    """Reference map for RandomState(seed): (num_roads, roads) or None if the seed is invalid.

    num_roads=None draws it first from the same stream, exactly like TDGymBasic.reset (:42).
    """
    ref_loader.load()
    from gym_TD.envs import TDRoadGen
    seeding = _seeding()
    rng = seeding.CountingRandomState(seed)
    rng.budget = MAPGEN_BUDGET
    try:
        if num_roads is None:
            num_roads = int(rng.randint(low=1, high=4))
        roads = TDRoadGen.create_road(rng, map_size, num_roads)
        for rd in roads:   # TDBoard.__init__ would raise IndexError on an empty road
            rd[0], rd[-1]
    except (ValueError, IndexError, seeding.BudgetExceeded):
        return None
    return num_roads, roads


def board_roads(board):
    """Recover the planes the product needs from a reference board."""
    m = board.map
    L = board.map_size
    road_bits = (m[0] | (m[1] << 1) | (m[2] << 2) | (m[3] << 3)).astype(np.uint8)
    return dict(map_size=L, num_roads=len(board.start),
                start=[s[0] * L + s[1] for s in board.start], end=board.end[0] * L + board.end[1],
                road=road_bits.reshape(-1), dist=m[4].reshape(-1).astype(np.int32),
                dir=m[5].reshape(-1).astype(np.int32))


def board_state(env_or_board, env=None):
    """Dynamic state of a reference board in the format of OracleEnv.state_dict()."""
    b = env_or_board._board if hasattr(env_or_board, "_board") else env_or_board
    e = env_or_board if hasattr(env_or_board, "_board") else env
    L = b.map_size
    return dict(
        cost_def=float(b.cost_def), cost_atk=float(b.cost_atk), base_LP=b.base_LP, steps=b.steps,
        attacker_cd=(e.attacker_cd if e is not None else 0),
        defender_cd=(e.defender_cd if e is not None else 0),
        map6=b.map[6].reshape(-1).astype(np.int32).copy(),
        towers=[(int(t.loc[0]) * L + int(t.loc[1]), int(t.type), int(t.lv), float(t.cd), float(t.atk), int(t.rge),
                 int(t.dmgrge), float(t.intv), float(t.cost)) for t in b.towers],
        enemies=[(int(x.loc[0]) * L + int(x.loc[1]), int(x.type), float(x.LP), float(x.maxLP), float(x.margin),
                  int(x.dist), int(x.slowdown), float(x.speed), float(x.defense)) for x in b.enemies],
    )


def states_equal(a, b):
    """Exact comparison (floats by repr) of two state dicts; returns list of differing keys."""
    bad = []
    for k in a:
        if k == "map6":
            if not np.array_equal(a[k], b[k]):
                bad.append(k)
        elif k in ("towers", "enemies"):
            if len(a[k]) != len(b[k]) or any(repr(tuple(x)) != repr(tuple(y)) for x, y in zip(a[k], b[k])):
                bad.append(k)
        elif repr(a[k]) != repr(b[k]):
            bad.append(k)
    return bad


# ---------------------------------------------------------------------------------------------
# Multi-action wrappers: the reference's step() raises UnboundLocalError in this mode (9.6), so
# these restate TDDefense.py:38-60,79-86 / TDMulti.py:50-84,117-125 around the real board calls.

def def_step_multi(env, action):
    from gym_TD.envs.TDParam import config
    env.attacker_cd = max(env.attacker_cd - 1, 0)
    env.defender_cd = max(env.defender_cd - 1, 0)
    b = env._board
    L = b.map_size
    real_act = np.zeros((6, L, L), dtype=np.int64)
    if env.defender_cd == 0:
        for r in range(L):
            for c in range(L):
                for t in range(4):
                    if action[t][r][c] == 1 and b.tower_build(t, [r, c]):
                        env.defender_cd = config.defender_action_interval
                        real_act[t, r, c] = 1
                if action[4][r][c] == 1 and b.tower_lvup([r, c]):
                    env.defender_cd = config.defender_action_interval
                    real_act[4, r, c] = 1
                if action[5][r][c] == 1 and b.tower_destruct([r, c]):
                    env.defender_cd = config.defender_action_interval
                    real_act[5, r, c] = 1
    getattr(env, "random_enemy_lv{}".format(env.difficulty))()
    reward = b.step()
    done = b.done()
    states = b.get_states()
    win = None
    if done:
        win = b.base_LP is None or b.base_LP > 0
    return states, reward, done, {"RealAction": real_act, "Win": win,
                                  "AllowNextMove": env.defender_cd <= 1, "FailCode": 0}


def multi_step_multi(env, action):
    from gym_TD.envs.TDParam import config
    env.attacker_cd = max(env.attacker_cd - 1, 0)
    env.defender_cd = max(env.defender_cd - 1, 0)
    b = env._board
    L = b.map_size
    atk_act, def_act = action["Attacker"], action["Defender"]
    real = {"Attacker": np.copy(atk_act)}
    if env.attacker_cd == 0:
        for i in range(env.num_roads):
            if b.summon_cluster(atk_act[i], i):
                env.attacker_cd = config.attacker_action_interval
            else:
                real["Attacker"][i] = 4
    real["Defender"] = np.zeros((6, L, L), dtype=np.int64)
    if env.defender_cd == 0:
        for r in range(L):
            for c in range(L):
                for t in range(4):
                    if def_act[t][r][c] == 1 and b.tower_build(t, [r, c]):
                        env.defender_cd = config.defender_action_interval
                        real["Defender"][t, r, c] = 1
                if def_act[4][r][c] == 1 and b.tower_lvup([r, c]):
                    env.defender_cd = config.defender_action_interval
                    real["Defender"][4, r, c] = 1
                if def_act[5][r][c] == 1 and b.tower_destruct([r, c]):
                    env.defender_cd = config.defender_action_interval
                    real["Defender"][5, r, c] = 1
    reward = b.step()
    done = b.done()
    states = b.get_states()
    win = None
    if done:
        win = {"Defender": b.base_LP is None or b.base_LP > 0,
               "Attacker": b.base_LP is None or b.base_LP <= 0}
    return states, reward, done, {"RealAction": real, "Win": win,
                                  "AllowNextMove": {"Attacker": env.attacker_cd <= 1,
                                                    "Defender": env.defender_cd <= 1},
                                  "FailCode": {"Attacker": [], "Defender": 0}}


# ---------------------------------------------------------------------------------------------
# Action generators that actually exercise build / LvUp / destruct (uniform actions mostly fail)

def smart_defender_action(board, rs, p_nop=0.3, p_uniform=0.2):
    L = board.map_size
    nop = 6 * L * L
    u = rs.random_sample()
    if u < p_nop:
        return nop
    if u < p_nop + p_uniform:
        return int(rs.randint(nop + 1))
    kind = rs.randint(10)
    if kind < 6 or not board.towers:       # build on a (probably) free cell
        free = np.argwhere(board.map[6] == 0)
        if len(free) == 0:
            return nop
        # bias toward cells close to the road so towers have targets
        r, c = free[rs.randint(len(free))]
        for _ in range(6):
            rr, cc = free[rs.randint(len(free))]
            if board.map[0, max(rr - 2, 0):rr + 3, max(cc - 2, 0):cc + 3].any():
                r, c = rr, cc
                break
        t = int(rs.randint(4))
        return int(t * L * L + r * L + c)
    tw = board.towers[rs.randint(len(board.towers))]
    act = 4 if kind < 9 else 5
    return int(act * L * L + tw.loc[0] * L + tw.loc[1])


def sparse_multi_action(board, rs, p=0.01):
    L = board.map_size
    a = (rs.random_sample((6, L, L)) < p).astype(np.int64)
    a[rs.random_sample((6, L, L)) < p] = 2   # the value 2 is legal and inert (TDDefense.py:22,46)
    return a


def seed_python_random(seed):
    random.seed(seed)
    return random.getstate()
