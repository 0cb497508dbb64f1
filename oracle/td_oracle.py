"""ctypes binding of the CPU oracle (oracle/td_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py -- never by gym_td_b200.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libtd_oracle.so")

MAX_CELLS = 64 * 64
CAP_TOWERS = 1024
CAP_ENEMIES = 2048
NT = 4
NLV = 2
CLUSTER = 8
ROADS = 3

CONFIG_TABLES = ["enemy_LP", "enemy_speed", "enemy_defense", "enemy_cost", "tower_attack",
                 "tower_cost", "tower_attack_interval"]


class Config(C.Structure):
    _fields_ = (
        [(n, (C.c_double * NLV) * NT) for n in CONFIG_TABLES]
        + [("tower_range", (C.c_int32 * NLV) * NT), ("tower_splash_range", (C.c_int32 * NLV) * NT)]
        + [(n, C.c_double) for n in (
            "tower_destruct_return", "frozen_ratio", "attacker_init_cost", "defender_init_cost",
            "max_cost", "reward_kill", "penalty_leak", "reward_time", "attacker_cost_init_rate",
            "attacker_cost_final_rate", "defender_cost_rate", "enemy_upgrade_at")]
        + [(n, C.c_int32) for n in (
            "frozen_time", "base_LP", "tower_distance", "attacker_action_interval",
            "defender_action_interval", "max_episode_steps", "max_tower_lv", "pad_")]
    )


class Enemy(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("maxLP", "LP", "speed", "defense", "cost", "margin")] + \
               [(n, C.c_int32) for n in ("loc", "dist", "slowdown", "type", "uid", "hit")]


class Tower(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("atk", "intv", "cost", "cd")] + \
               [(n, C.c_int32) for n in ("rge", "dmgrge", "loc", "lv", "type", "pad_")]


class MT(C.Structure):
    _fields_ = [("mt", C.c_uint32 * 624), ("pos", C.c_int32), ("pad_", C.c_int32)]


class Env(C.Structure):
    _fields_ = [
        ("cfg", Config),
        ("L", C.c_int32), ("num_roads", C.c_int32),
        ("start", C.c_int32 * ROADS), ("end", C.c_int32),
        ("road", C.c_uint8 * MAX_CELLS),
        ("dist", C.c_int32 * MAX_CELLS),
        ("dir", C.c_int32 * MAX_CELLS),
        ("map6", C.c_int32 * MAX_CELLS),
        ("cost_def", C.c_double), ("cost_atk", C.c_double), ("max_cost", C.c_double),
        ("progress", C.c_double),
        ("base_LP", C.c_int32), ("max_base_LP", C.c_int32), ("has_base_LP", C.c_int32),
        ("steps", C.c_int32), ("fail_code", C.c_int32),
        ("attacker_cd", C.c_int32), ("defender_cd", C.c_int32),
        ("n_towers", C.c_int32), ("n_enemies", C.c_int32), ("next_uid", C.c_int32),
        ("towers", Tower * CAP_TOWERS),
        ("enemies", Enemy * CAP_ENEMIES),
        ("enemy_LP", ((C.c_float * MAX_CELLS) * NT) * 4),
        ("pyrand", MT), ("nprand", MT),
        ("last_kills", C.c_int32), ("last_leaks", C.c_int32),
        ("peak_towers", C.c_int32), ("peak_enemies", C.c_int32),
    ]


class StepOut(C.Structure):
    _fields_ = [
        ("reward", C.c_double),
        ("done", C.c_int32), ("win", C.c_int32), ("win_attacker", C.c_int32),
        ("allow_next_def", C.c_int32), ("allow_next_atk", C.c_int32),
        ("real_def", C.c_int64),
        ("fail_def", C.c_int32), ("n_fail_atk", C.c_int32),
        ("fail_atk", C.c_int32 * ROADS),
        ("real_is_def_only", C.c_int32),
        ("real_atk", (C.c_int64 * CLUSTER) * ROADS),
    ]


_lib = None


def build(force=False):
    if force or not os.path.exists(_SO) or \
            os.path.getmtime(_SO) < max(os.path.getmtime(os.path.join(_HERE, f))
                                        for f in ("td_oracle.c", "td_oracle.h")):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        assert L.tdo_sizeof_env() == C.sizeof(Env), (L.tdo_sizeof_env(), C.sizeof(Env))
        assert L.tdo_sizeof_config() == C.sizeof(Config)
        L.tdo_board_step.restype = C.c_double
        L.tdo_py_random.restype = C.c_double
        L.tdo_np_randint.restype = C.c_int64
        L.tdo_np_randint.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
        L.tdo_mt_next.restype = C.c_uint32
        L.tdo_py_randbelow.restype = C.c_uint32
        L.tdo_def_step.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]
        L.tdo_bench_def.restype = C.c_double
        L.tdo_bench_def.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_void_p]
        L.tdo_multi_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        _lib = L
    return _lib


def default_config():
    c = Config()
    lib().tdo_default_config(C.byref(c))
    return c


def config_from_dict(d, hyper=None):
    """Build a Config from a reference-style config dict (TDParam.getConfig())."""
    c = default_config()
    for name in CONFIG_TABLES + ["tower_range", "tower_splash_range"]:
        if name in d:
            for t in range(NT):
                for l in range(NLV):
                    getattr(c, name)[t][l] = d[name][t][l]
    for name, _ in Config._fields_:
        if name in d and name not in CONFIG_TABLES + ["tower_range", "tower_splash_range", "base_LP"]:
            setattr(c, name, d[name])
    if "base_LP" in d:
        c.base_LP = -1 if d["base_LP"] is None else int(d["base_LP"])
    if hyper and "max_episode_steps" in hyper:
        c.max_episode_steps = hyper["max_episode_steps"]
    return c


def mt_from_python_random(state):
    """random.getstate() -> MT"""
    m = MT()
    words = state[1]
    m.mt[:] = words[:624]
    m.pos = words[624]
    return m


def mt_from_numpy(rs):
    """np.random.RandomState -> MT"""
    st = rs.get_state()
    m = MT()
    m.mt[:] = [int(x) for x in st[1]]
    m.pos = int(st[2])
    return m


class OracleEnv(object):
    """One game instance driven through the C restatement."""

    def __init__(self, cfg=None):
        self.L_ = lib()
        self.e = Env()
        self.cfg = cfg if cfg is not None else default_config()
        self.out = StepOut()

    # -- construction -----------------------------------------------------
    def init_from_roads(self, map_size, roads):
        """roads: list (per road) of [r, c] cells from start to end (TDRoadGen output)."""
        flat = np.asarray([p[0] * map_size + p[1] for rd in roads for p in rd], dtype=np.int32)
        lens = np.asarray([len(rd) for rd in roads], dtype=np.int32)
        self.L_.tdo_board_init(C.byref(self.e), C.byref(self.cfg), map_size, len(roads),
                               flat.ctypes.data_as(C.c_void_p), lens.ctypes.data_as(C.c_void_p))
        return self

    def init_from_planes(self, map_size, num_roads, start, end, road, dist, dirs):
        start = np.asarray(list(start) + [0] * (3 - len(start)), dtype=np.int32)
        road = np.ascontiguousarray(road, dtype=np.uint8).ravel()
        dist = np.ascontiguousarray(dist, dtype=np.int32).ravel()
        dirs = np.ascontiguousarray(dirs, dtype=np.int32).ravel()
        self.L_.tdo_board_init_planes(C.byref(self.e), C.byref(self.cfg), map_size, num_roads,
                                      start.ctypes.data_as(C.c_void_p), int(end),
                                      road.ctypes.data_as(C.c_void_p), dist.ctypes.data_as(C.c_void_p),
                                      dirs.ctypes.data_as(C.c_void_p))
        return self

    def set_pyrand(self, state):
        self.e.pyrand = mt_from_python_random(state)

    def set_nprand(self, rs):
        self.e.nprand = mt_from_numpy(rs)

    # -- board API ----------------------------------------------------------
    def tower_build(self, t, loc):
        return bool(self.L_.tdo_tower_build(C.byref(self.e), int(t), int(loc)))

    def tower_lvup(self, loc):
        return bool(self.L_.tdo_tower_lvup(C.byref(self.e), int(loc)))

    def tower_destruct(self, loc):
        return bool(self.L_.tdo_tower_destruct(C.byref(self.e), int(loc)))

    def summon_enemy(self, t, start_id):
        return bool(self.L_.tdo_summon_enemy(C.byref(self.e), int(t), int(start_id)))

    def summon_cluster(self, types, start_id):
        types = np.ascontiguousarray(types, dtype=np.int64)
        real = np.zeros(CLUSTER, dtype=np.int64)
        ok = self.L_.tdo_summon_cluster(C.byref(self.e), types.ctypes.data_as(C.c_void_p), int(start_id),
                                        real.ctypes.data_as(C.c_void_p))
        return bool(ok), real

    def board_step(self):
        return float(self.L_.tdo_board_step(C.byref(self.e)))

    def done(self):
        return bool(self.L_.tdo_done(C.byref(self.e)))

    def refresh(self):
        """Bring the derived fields in line with a state written field by field: progress (steps / max_episode_steps
        in f64, as tdo_board_step computes it) and the enemy-statistics planes of the current lists (tdo_enemy_stats)."""
        self.e.progress = float(self.e.steps) / float(self.e.cfg.max_episode_steps)
        self.L_.tdo_enemy_stats(C.byref(self.e))

    def get_states(self):
        L = self.e.L
        out = np.empty((45, L, L), dtype=np.float32)
        self.L_.tdo_get_states(C.byref(self.e), out.ctypes.data_as(C.c_void_p))
        return out

    # -- env wrappers ---------------------------------------------------------
    def def_step(self, action, difficulty=1, use_np=False):
        self.L_.tdo_def_step(C.byref(self.e), int(action), int(difficulty), int(use_np), C.byref(self.out))
        return self.out

    def def_step_multi(self, action, difficulty=1, use_np=False):
        a = np.ascontiguousarray(action, dtype=np.int64)
        real = np.zeros_like(a)
        self.L_.tdo_def_step_multi(C.byref(self.e), a.ctypes.data_as(C.c_void_p),
                                   real.ctypes.data_as(C.c_void_p), int(difficulty), int(use_np),
                                   C.byref(self.out))
        return self.out, real

    def atk_step(self, action, difficulty=1, use_np=False):
        a = np.ascontiguousarray(action, dtype=np.int64)
        self.L_.tdo_atk_step(C.byref(self.e), a.ctypes.data_as(C.c_void_p), int(difficulty), int(use_np),
                             C.byref(self.out))
        return self.out

    def multi_step(self, atk_action, def_action):
        a = np.ascontiguousarray(atk_action, dtype=np.int64)
        self.L_.tdo_multi_step(C.byref(self.e), a.ctypes.data_as(C.c_void_p), int(def_action),
                               C.byref(self.out))
        return self.out

    def multi_step_multi(self, atk_action, def_action):
        a = np.ascontiguousarray(atk_action, dtype=np.int64)
        d = np.ascontiguousarray(def_action, dtype=np.int64)
        real = np.zeros_like(d)
        self.L_.tdo_multi_step_multi(C.byref(self.e), a.ctypes.data_as(C.c_void_p),
                                     d.ctypes.data_as(C.c_void_p), real.ctypes.data_as(C.c_void_p),
                                     C.byref(self.out))
        return self.out, real

    # -- state inspection -------------------------------------------------------
    def state_dict(self):
        """Full dynamic board state in list order (the comparison key for parity tests)."""
        e = self.e
        cells = e.L * e.L
        return dict(
            cost_def=e.cost_def, cost_atk=e.cost_atk,
            base_LP=(e.base_LP if e.has_base_LP else None), steps=e.steps,
            attacker_cd=e.attacker_cd, defender_cd=e.defender_cd,
            map6=np.ctypeslib.as_array(e.map6)[:cells].copy(),
            towers=[(t.loc, t.type, t.lv, t.cd, t.atk, t.rge, t.dmgrge, t.intv, t.cost)
                    for t in e.towers[:e.n_towers]],
            enemies=[(x.loc, x.type, x.LP, x.maxLP, x.margin, x.dist, x.slowdown, x.speed, x.defense)
                     for x in e.enemies[:e.n_enemies]],
        )
