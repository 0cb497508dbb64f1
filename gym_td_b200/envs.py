"""Single-instance gym-style environments: drop-in counterparts of the reference's
TDDefense / TDAttack / TDMulti (gym_TD/envs/TDDefense.py:13-87, TDAttack.py:12-56, TDMulti.py:10-139,
base class TDGymBasic.py:12-55), implemented as n = 1 façades over the batched CUDA engine.

Same constructor arguments, attributes (`observation_space`, `action_space`, `name`, `num_roads`,
`map_size`, `difficulty`, `np_random`), old-gym 4-tuple `step`, `reset() -> obs`, `seed(s) -> [s]`,
`empty_action()`, `info` keys and value types -- including the reference's quirks (TDMulti's
RealAction collapsing to an int on defender success, TDMulti.py:114).

Randomness contract (SURVEY.md 8c): `seed(s)` installs numpy.random.RandomState(s) as `np_random`; the map
is generated from that live stream (`num_roads` first), so repeated `reset()` calls walk the stream exactly
like the reference.  With `random_agent=True` (default) the scripted opponent consumes Python's global
`random` module, as in the reference: the façade hands the module's generator state to the device before a
step and installs the advanced state afterwards, so `random.seed(s)` replays bit for bit.

Deviations (documented, SURVEY.md 9.6-9.8): an invalid map draw (the reference raises or hangs) is retried
from the same stream; multi-action mode returns FailCode 0 / [] where the reference raises;
`random_agent=False` (the scripted opponent on the env's own `np_random`) covers what the reference can run:
TDDefense at difficulty 0 and 1, TDAttack at difficulty 0 (its lv1/lv2 np_random paths raise in the reference the
first time the destruct gate opens, TDGymBasic.py:191,287); the draws are made on the host from the live
`np_random` object and handed to the step as resolved opponent words.  `render` is out of scope.
"""
import random

import numpy as np
import torch

from . import engine as E
from . import mapgen, params, spaces
from .params import config, hyper_parameters


class Tower(object):
    __slots__ = ("loc", "type", "lv", "cd")


class Enemy(object):
    __slots__ = ("loc", "type", "lv", "LP", "maxLP", "margin", "slowdown")


class BoardView(object):
    """Read-only snapshot of the device-side board, shaped like the reference's TDBoard attributes."""

    def __init__(self, env):
        eng, L = env._engine, env.map_size
        st = eng.decode_state(eng.get_state_raw(0, 1)[0])
        h = st["header"]
        self.map_size = L
        self.cost_def, self.cost_atk = float(h["cost_def"]), float(h["cost_atk"])
        self.max_cost = config.max_cost
        self.base_LP = None if config.base_LP is None else int(h["base_LP"])
        self.max_base_LP = config.base_LP
        self.steps = int(h["steps"])
        self.progress = self.steps / hyper_parameters.max_episode_steps
        p = mapgen.planes(env._map)
        self.start = [[s // L, s % L] for s in p["start"]]
        self.end = [p["end"] // L, p["end"] % L]
        self.map = np.zeros((7, L, L), dtype=np.int32)
        self.map[0:4], self.map[4], self.map[5] = p["road"], p["dist"], p["dir"]
        self.map[6] = st["map6"].reshape(L, L)
        self.towers, self.enemies = [], []
        for r in st["towers"]:
            t = Tower()
            t.loc, t.type, t.lv, t.cd = [int(r["loc"]) // L, int(r["loc"]) % L], int(r["type_lv"]) & 3, \
                int(r["type_lv"]) >> 2, float(r["cd"])
            self.towers.append(t)
        for r in st["enemies"]:
            e = Enemy()
            e.loc, e.type, e.lv = [int(r["loc"]) // L, int(r["loc"]) % L], int(r["type_lv"]) & 3, int(r["type_lv"]) >> 2
            e.LP, e.margin, e.slowdown = float(r["LP"]), float(r["margin"]), int(r["slowdown"])
            e.maxLP = config.enemy_LP[e.type][e.lv]
            self.enemies.append(e)
        self._env = env

    def get_states(self):
        return self._env._observe()

    def done(self):
        return (self.base_LP is not None and self.base_LP <= 0) or self.steps >= hyper_parameters.max_episode_steps

    @staticmethod
    def n_channels():
        return params.n_channels()

    @property
    def state_shape(self):
        return (params.n_channels(), self.map_size, self.map_size)


class TDGymBasic(object):
    metadata = {"render.modes": ["human", "rgb_array"],
                "video.frames_per_second": hyper_parameters.video_frames_per_second}
    _kind = None

    def __init__(self, map_size, seed, fixed_seed=False, random_agent=True, device=0):
        self.observation_space = spaces.Box(low=0., high=1., shape=(params.n_channels(), map_size, map_size),
                                            dtype=np.float32)
        self.map_size = map_size
        self.fixed_seed = fixed_seed
        self.input_seed = seed
        self.random_agent = random_agent
        self._device = torch.device("cuda", device)
        self._engine = E.Engine(self._kind, map_size, 1, device=device)   # raises when CUDA / the library is missing
        L = map_size
        dev = self._device
        self._obs = torch.empty((1, E.NCH, L, L), dtype=torch.float32, device=dev)
        self._out = dict(reward=torch.zeros(1, dtype=torch.float64, device=dev),
                         done=torch.zeros(1, dtype=torch.uint8, device=dev),
                         win=torch.zeros(1, dtype=torch.int8, device=dev),
                         allow=torch.zeros(1, dtype=torch.uint8, device=dev),
                         fail_def=torch.zeros(1, dtype=torch.int32, device=dev),
                         fail_atk=torch.zeros((1, 4), dtype=torch.int32, device=dev),
                         real_atk=torch.zeros((1, 3, 8), dtype=torch.int64, device=dev))
        self._map = None
        self.seed(seed)
        self.reset()

    # -- gym API --------------------------------------------------------------------------------------
    def seed(self, seed=None):
        self.np_random = np.random.RandomState(seed)
        return [seed]

    def reset(self):
        if self.fixed_seed:
            self.seed(self.input_seed)
        m = None
        while m is None:                      # the reference raises / hangs on these draws (SURVEY 9.8)
            m = mapgen.generate_from_stream(self.np_random, self.map_size)
        self._map = m
        self.num_roads = m.num_roads
        self._engine.set_config(config)       # `config` is read afresh, like TDGymBasic.reset does
        self._engine.upload_maps([m])
        self._engine.reset(obs=self._obs, stream=self._stream())
        self.attacker_cd = 0
        self.defender_cd = 0
        return self._obs_numpy()

    def step(self, action):
        raise NotImplementedError()

    def action_mask(self):
        """Which actions the next step() would carry out (TDVecEnv.action_mask for this one env), as numpy bool
        arrays: TDDefense the Discrete mask [6*L*L + 1] or, with allow_multiple_actions, the single-flag Box mask
        (6, L, L); TDAttack (3, 4) per (road, enemy type); TDMulti {"Attacker": ..., "Defender": ...}."""
        L = self.map_size
        d = torch.zeros((1, 6 * L * L + 1), dtype=torch.uint8, device=self._device) if self._kind != "atk" else None
        a = torch.zeros((1, E.ROADS, E.NT), dtype=torch.uint8, device=self._device) if self._kind != "def" else None
        self._engine.action_mask(d, a, self._stream())
        if d is not None:
            d = d[0].cpu().numpy().astype(bool)
            if self._multi():
                d = d[:-1].reshape(6, L, L)
        if a is not None:
            a = a[0].cpu().numpy().astype(bool)
        return {"def": d, "atk": a, "2p": {"Attacker": a, "Defender": d}}[self._kind]

    def render(self, mode="human"):
        raise NotImplementedError("rendering (pyglet viewer, TDBoard.py:387-664) is outside the B200 hot path")

    def close(self):
        self._engine.close()

    # -- helpers --------------------------------------------------------------------------------------
    @property
    def _board(self):
        return BoardView(self)

    def _stream(self):
        return torch.cuda.current_stream(self._device).cuda_stream

    def _obs_numpy(self):
        return self._obs[0].cpu().numpy()

    def _observe(self):
        self._engine.observe(self._obs, self._stream())
        return self._obs_numpy()

    def _multi(self):
        return bool(hyper_parameters.allow_multiple_actions)

    def _launch(self, def_action=None, atk_action=None, opponent=None, real_def=None, scripted=False,
                opponent_cluster=None):
        """One device step.  `scripted`: the on-device opponent runs on Python's global `random` stream."""
        if scripted:
            st = random.getstate()
            self._engine.seed_opponent(np.asarray(st[1], dtype=np.uint64).astype(np.uint32).reshape(1, 625))
        o = self._out
        io = E.Engine.make_io(def_action=def_action, atk_action=atk_action, opponent=opponent,
                              opponent_cluster=opponent_cluster, multi_action=self._multi() and self._kind != "atk", auto_reset=False, obs=self._obs,
                              reward=o["reward"], done=o["done"], win=o["win"], allow_next=o["allow"],
                              real_def=real_def, real_atk=o["real_atk"], fail_def=o["fail_def"],
                              fail_atk=o["fail_atk"])
        self._engine.step(io, self._stream())
        torch.cuda.synchronize(self._device)
        if scripted:
            words = self._engine.get_opponent(0, 1)[0]
            random.setstate((st[0], tuple(int(x) for x in words), st[2]))

    def _sync_cds(self):
        h = self._engine.decode_state(self._engine.get_state_raw(0, 1)[0])["header"]
        self.attacker_cd, self.defender_cd = int(h["attacker_cd"]), int(h["defender_cd"])
        if int(h["flags"]):
            # more live enemies / towers than the device lists hold (only reachable through paramConfig overrides):
            # entries were dropped, the trajectory no longer follows the reference -- never silently
            raise E.TdError(-5, "tower / enemy capacity exceeded (flags=%d): the episode is invalid" % int(h["flags"]))

    def _win(self):
        w = int(self._out["win"][0])
        return None if w < 0 else bool(w)


def _as_device_action(a, shape, device):
    t = torch.as_tensor(np.ascontiguousarray(a, dtype=np.int64).reshape(shape))
    return t.to(device)


class TDDefense(TDGymBasic):
    _kind = "def"

    def __init__(self, map_size, difficulty=1, seed=None, fixed_seed=False, random_agent=True, device=0):
        super(TDDefense, self).__init__(map_size, seed, fixed_seed, random_agent, device)
        if hyper_parameters.allow_multiple_actions:
            self.action_space = spaces.Box(low=0., high=2., shape=(config.tower_types + 2, map_size, map_size),
                                           dtype=np.int64)
        else:
            self.action_space = spaces.Discrete(map_size * map_size * (config.tower_types + 2) + 1)
        if difficulty not in (0, 1):
            raise AttributeError("'TDDefense' object has no attribute 'random_enemy_lv%s'" % (difficulty,))
        self.difficulty = difficulty
        self.name = "TDDefense"

    def empty_action(self):
        L = self.map_size
        if hyper_parameters.allow_multiple_actions:
            return np.zeros((config.tower_types + 2, L, L), dtype=np.int64)
        return L * L * (config.tower_types + 2)

    def step(self, action):
        err_msg = "%r (%s) invalid" % (action, type(action))
        assert self.action_space.contains(action), err_msg
        L, dev = self.map_size, self._device
        multi = self._multi()
        if multi:
            d = _as_device_action(action, (1, 6, L, L), dev)
            real = torch.zeros_like(d)
        else:
            d = torch.tensor([int(action)], dtype=torch.int64, device=dev)
            real = torch.zeros(1, dtype=torch.int64, device=dev)
        opponent = None
        if self.random_agent:
            self._engine.set_difficulty(self.difficulty)
            self._launch(def_action=d, real_def=real, scripted=True)
        elif self.difficulty == 1:
            byte = 0xFF
            if max(self.attacker_cd - 1, 0) == 0:                      # TDGymBasic.py:96,102-103
                t = int(self.np_random.randint(0, config.enemy_types))
                road = int(self.np_random.randint(self.num_roads))
                byte = t | (road << 4)
            opponent = torch.tensor([byte], dtype=torch.uint8, device=dev)
            self._launch(def_action=d, real_def=real, opponent=opponent)
        else:
            word = 0xFFFFFFFF
            if max(self.attacker_cd - 1, 0) == 0:                      # TDGymBasic.py:82,87-89
                cluster = self.np_random.randint(0, config.enemy_types, [hyper_parameters.max_cluster_length],
                                                 dtype=np.int64)
                road = int(self.np_random.randint(self.num_roads))
                word = sum(int(c) << (2 * k) for k, c in enumerate(cluster)) | (road << 16)
            cl = torch.tensor([word], dtype=torch.int64, device=dev).to(torch.uint32)
            self._launch(def_action=d, real_def=real, opponent_cluster=cl)
        self._sync_cds()
        o = self._out
        done = bool(o["done"][0])
        if multi:
            real_act, fail = real[0].cpu().numpy(), 0
        else:
            real_act, fail = int(real[0]), int(o["fail_def"][0])
        return self._obs_numpy(), float(o["reward"][0]), done, {
            "RealAction": real_act, "Win": self._win(), "AllowNextMove": self.defender_cd <= 1, "FailCode": fail}


class TDAttack(TDGymBasic):
    _kind = "atk"

    def __init__(self, map_size, difficulty=1, seed=None, fixed_seed=False, random_agent=True, device=0):
        super(TDAttack, self).__init__(map_size, seed, fixed_seed, random_agent, device)
        self.action_space = spaces.Box(low=0, high=config.enemy_types,
                                       shape=(hyper_parameters.max_num_of_roads, hyper_parameters.max_cluster_length),
                                       dtype=np.int64)
        if difficulty not in (0, 1, 2):
            raise AttributeError("'TDAttack' object has no attribute 'random_tower_lv%s'" % (difficulty,))
        if not random_agent and difficulty != 0:
            raise NotImplementedError("TDAttack(random_agent=False) at difficulty 1 / 2 raises in the reference "
                                      "(TDGymBasic.py:191,287); use random_agent=True and random.seed()")
        self.difficulty = difficulty
        self.name = "TDAttack"

    def empty_action(self):
        return np.full((hyper_parameters.max_num_of_roads, hyper_parameters.max_cluster_length), config.enemy_types)

    def step(self, action):
        err_msg = "%r (%s) invalid" % (action, type(action))
        assert self.action_space.contains(action), err_msg
        a = _as_device_action(action, (1, 3, 8), self._device)
        if self.random_agent:
            self._engine.set_difficulty(self.difficulty)
            self._launch(atk_action=a, scripted=True)
        else:
            build = -1
            if max(self.defender_cd - 1, 0) == 0:                      # TDGymBasic.py:112,118-119
                r, c = self.np_random.randint(0, self.map_size, [2, ])
                t = int(self.np_random.randint(0, config.tower_types))
                build = t * self.map_size * self.map_size + int(r) * self.map_size + int(c)
            b = torch.tensor([build], dtype=torch.int64, device=self._device)
            self._launch(atk_action=a, def_action=b)
        self._sync_cds()
        o = self._out
        fa = o["fail_atk"][0].tolist()
        return self._obs_numpy(), float(o["reward"][0]), bool(o["done"][0]), {
            "RealAction": o["real_atk"][0].cpu().numpy(), "Win": self._win(),
            "AllowNextMove": self.attacker_cd <= 1, "FailCode": fa[1:1 + fa[0]]}


class TDMulti(TDGymBasic):
    _kind = "2p"

    def __init__(self, map_size, seed=None, fixed_seed=False, random_agent=True, device=0):
        super(TDMulti, self).__init__(map_size, seed, fixed_seed, random_agent, device)
        atk = spaces.Box(low=0, high=4, shape=(hyper_parameters.max_num_of_roads, hyper_parameters.max_cluster_length),
                         dtype=np.int64)
        if hyper_parameters.allow_multiple_actions:
            self.action_space = spaces.Dict({"Attacker": atk, "Defender": spaces.Box(
                low=0., high=2., shape=(6, map_size, map_size), dtype=np.int64)})
        else:
            self.action_space = spaces.Dict({"Attacker": atk, "Defender": spaces.Discrete(map_size * map_size * 6 + 1)})
        self.name = "TDMulti"

    def empty_action(self):
        L = self.map_size
        atk = np.full((hyper_parameters.max_num_of_roads, hyper_parameters.max_cluster_length), 4, dtype=np.int64)
        if hyper_parameters.allow_multiple_actions:
            return {"Attacker": atk, "Defender": np.zeros((6, L, L), dtype=np.int64)}
        return {"Attacker": atk, "Defender": L * L * 6}

    @property
    def board(self):
        return self._board

    def step(self, action):
        err_msg = "%r (%s) invalid" % (action, type(action))
        assert self.action_space.contains(action), err_msg
        L, dev = self.map_size, self._device
        multi = self._multi()
        a = _as_device_action(action["Attacker"], (1, 3, 8), dev)
        if multi:
            d = _as_device_action(action["Defender"], (1, 6, L, L), dev)
            real = torch.zeros_like(d)
        else:
            d = torch.tensor([int(action["Defender"])], dtype=torch.int64, device=dev)
            real = torch.zeros(1, dtype=torch.int64, device=dev)
        self._launch(def_action=d, atk_action=a, real_def=real)
        self._sync_cds()
        o = self._out
        done = bool(o["done"][0])
        fa = o["fail_atk"][0].tolist()
        if multi:
            real_act = {"Attacker": o["real_atk"][0].cpu().numpy(), "Defender": real[0].cpu().numpy()}
            fail = {"Attacker": [], "Defender": 0}
        else:
            nop = L * L * 6
            rd = int(real[0])
            if rd != nop:
                real_act = rd                                       # TDMulti.py:114: the dict is replaced by the int
            else:
                real_act = {"Attacker": o["real_atk"][0].cpu().numpy(), "Defender": nop}
            fail = {"Attacker": fa[1:1 + fa[0]], "Defender": int(o["fail_def"][0])}
        win = None
        if done:
            w = bool(int(o["win"][0]))
            win = {"Defender": w, "Attacker": (config.base_LP is None) or (not w)}
        return self._obs_numpy(), float(o["reward"][0]), done, {
            "RealAction": real_act, "Win": win,
            "AllowNextMove": {"Attacker": self.attacker_cd <= 1, "Defender": self.defender_cd <= 1},
            "FailCode": fail}
