"""ctypes binding of the C ABI in include/td_b200.h (libtd_b200.so, built in-tree by build.py).

This is the only place Python touches the native library.  There is no CPU fallback and no
alternative implementation: if the shared library is missing, importing this module raises.
"""
import ctypes as C
import os

import numpy as np

from . import params

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TD_B200_LIB") or os.path.join(_HERE, "libtd_b200.so")   # override: kernel experiments

NT, NLV, CLUSTER, ROADS, NCH, MAX_L = 4, 2, 8, 3, 45, 64
CAP_TOWERS, CAP_ENEMIES = 32, 64
KIND_DEF, KIND_ATK, KIND_2P = 0, 1, 2
KINDS = {"def": KIND_DEF, "atk": KIND_ATK, "2p": KIND_2P}
OBS_FORMATS = {"f32": 0, "bf16": 1, "u8": 2}
OPTIONS = {"host_chunks": 1, "host_graph": 2, "generic_kernels": 5, "host_chain": 6, "host_first_chunk": 7, "host_zero_copy": 8}

_TABLES_F64 = ["enemy_LP", "enemy_speed", "enemy_defense", "enemy_cost", "tower_attack", "tower_cost",
               "tower_attack_interval"]
_TABLES_I32 = ["tower_range", "tower_splash_range"]
_SCALARS_F64 = ["tower_destruct_return", "frozen_ratio", "attacker_init_cost", "defender_init_cost", "max_cost",
                "reward_kill", "penalty_leak", "reward_time", "attacker_cost_init_rate",
                "attacker_cost_final_rate", "defender_cost_rate", "enemy_upgrade_at"]
_SCALARS_I32 = ["frozen_time", "base_LP", "tower_distance", "attacker_action_interval",
                "defender_action_interval", "max_episode_steps", "max_tower_lv", "pad_"]


class TdConfig(C.Structure):
    _fields_ = ([(n, (C.c_double * NLV) * NT) for n in _TABLES_F64]
                + [(n, (C.c_int32 * NLV) * NT) for n in _TABLES_I32]
                + [(n, C.c_double) for n in _SCALARS_F64]
                + [(n, C.c_int32) for n in _SCALARS_I32])


class TdMap(C.Structure):
    _fields_ = [("map_size", C.c_int32), ("num_roads", C.c_int32), ("start", C.c_int32 * ROADS),
                ("end", C.c_int32), ("max_dist", C.c_int32), ("n_randint", C.c_int32),
                ("cells", C.c_uint8 * (MAX_L * MAX_L)), ("dist", C.c_uint8 * (MAX_L * MAX_L))]


class TdStepIO(C.Structure):
    _fields_ = [("def_action_dev", C.c_void_p), ("atk_action_dev", C.c_void_p), ("opponent_dev", C.c_void_p),
                ("multi_action", C.c_int32), ("auto_reset", C.c_int32),
                ("obs_dev", C.c_void_p), ("reward_dev", C.c_void_p), ("done_dev", C.c_void_p),
                ("win_dev", C.c_void_p), ("allow_next_dev", C.c_void_p), ("real_def_dev", C.c_void_p),
                ("real_atk_dev", C.c_void_p), ("fail_def_dev", C.c_void_p), ("fail_atk_dev", C.c_void_p),
                ("obs_incremental", C.c_int32), ("obs_format", C.c_int32), ("opponent_cluster_dev", C.c_void_p),
                ("packed_out_dev", C.c_void_p)]


class TdHostIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "def_action_host", "atk_action_host", "opponent_host", "obs_host", "reward_host", "done_host",
        "win_host", "allow_next_host", "real_def_host", "real_atk_host", "fail_def_host", "fail_atk_host",
        "opponent_cluster_host", "packed_host")]


class TdLayout(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "record_bytes", "off_header", "off_towers", "off_enemies", "off_map6", "tower_stride", "enemy_stride",
        "cap_towers", "cap_enemies", "map_record_bytes", "mt_words", "pad_")]


class TdStats(C.Structure):
    _fields_ = [("return_sum", C.c_double)] + [(n, C.c_int64) for n in (
        "episodes", "length_sum", "wins", "kills", "leaks", "overflow_envs", "steps")]


HEADER_DTYPE = np.dtype([
    ("cost_def", "<f8"), ("cost_atk", "<f8"), ("ep_return", "<f8"), ("base_LP", "<i4"), ("steps", "<i4"),
    ("map_id", "<i4"), ("episode", "<i4"), ("defender_cd", "<i2"), ("attacker_cd", "<i2"),
    ("n_towers", "u1"), ("n_enemies", "u1"), ("flags", "u1"), ("pad0", "u1"), ("ep_kills", "<u2"),
    ("ep_leaks", "<u2"), ("rng_pos", "<i4"), ("pad1", "<i4"), ("ep_kills_hi", "<u2"), ("ep_leaks_hi", "<u2")])
TOWER_DTYPE = np.dtype([("cd", "<f8"), ("loc", "<u2"), ("type_lv", "u1"), ("scratch", "u1", (5,))])
ENEMY_DTYPE = np.dtype([("LP", "<f8"), ("margin", "<f8"), ("loc", "<u2"), ("type_lv", "u1"),
                        ("slowdown", "u1"), ("scratch", "u1", (4,))])
assert HEADER_DTYPE.itemsize == 64 and TOWER_DTYPE.itemsize == 16 and ENEMY_DTYPE.itemsize == 24


class TdError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("td_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None

EXPORTS = ["td_abi_version", "td_last_error", "td_default_config", "td_mapgen", "td_mapgen_stream",
           "td_mapgen_batch", "td_seed_opponent_python", "td_create",
           "td_destroy", "td_set_config", "td_get_layout", "td_upload_maps", "td_set_map_stride", "td_reset",
           "td_seed_opponent", "td_set_difficulty", "td_step", "td_observe", "td_step_host", "td_get_state",
           "td_set_state", "td_get_opponent", "td_get_stats", "td_reset_stats", "td_rollout_mask", "td_rollout_record",
           "td_gae", "td_snapshot", "td_observe_snapshot", "td_set_option", "td_packed_stride", "td_invalidate_obs", "td_observe_as",
           "td_alloc_compressible", "td_free_compressible", "td_upgrade_step", "td_action_mask"]


def lib():
    """Load libtd_b200.so (fails loudly when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not found: build it with `python -m gym_td_b200.build` "
                              "(nvcc, sm_100a); there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.td_last_error.restype = C.c_char_p
        L.td_last_error.argtypes = [C.c_void_p]
        L.td_default_config.restype = None
        L.td_mapgen.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.td_mapgen_stream.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.td_seed_opponent_python.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.td_mapgen_batch.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p]
        L.td_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        for name in ("td_destroy", "td_get_layout", "td_set_config"):
            getattr(L, name).argtypes = [C.c_void_p] + ([C.c_void_p] if name != "td_destroy" else [])
        L.td_upload_maps.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.td_set_map_stride.argtypes = [C.c_void_p, C.c_int]
        L.td_set_difficulty.argtypes = [C.c_void_p, C.c_int]
        L.td_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_seed_opponent.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.td_get_opponent.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.td_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_observe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_step_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_get_state.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.td_set_state.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.td_get_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_reset_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.td_snapshot.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_observe_snapshot.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.td_rollout_mask.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_rollout_record.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_gae.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                             C.c_void_p, C.c_void_p, C.c_void_p]
        L.td_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.td_invalidate_obs.argtypes = [C.c_void_p]
        L.td_observe_as.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.td_alloc_compressible.argtypes = [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p]
        L.td_free_compressible.argtypes = [C.c_void_p]
        L.td_upgrade_step.argtypes = [C.c_int, C.c_double]
        L.td_action_mask.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        if L.td_abi_version() != 3:
            raise ImportError("libtd_b200.so ABI version mismatch")
        _lib = L
    return _lib


class CompressibleBuffer:
    """Device memory from td_alloc_compressible (a compressible CUDA virtual-memory allocation, zero-filled), exposed
    through __cuda_array_interface__ so that torch.as_tensor() wraps it without a copy; freed when the last tensor
    over it is gone.  `compressed` tells whether the driver granted compression."""

    def __init__(self, nbytes, device=0):
        ptr, granted = C.c_void_p(), C.c_int(0)
        rc = lib().td_alloc_compressible(int(device), int(nbytes), C.byref(ptr), C.byref(granted))
        if rc != 0:
            raise TdError(rc, (lib().td_last_error(None) or b"").decode())
        self.ptr, self.nbytes, self.device, self.compressed = ptr.value, int(nbytes), int(device), bool(granted.value)
        self.__cuda_array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 2,
                                         "strides": None}

    def tensor(self, shape, dtype):
        """A torch tensor of `shape` / `dtype` over the buffer (keeps the buffer alive)."""
        import torch
        flat = torch.as_tensor(self, device="cuda:%d" % self.device)
        return flat.view(dtype).view(shape)

    def __del__(self):
        ptr, self.ptr = getattr(self, "ptr", None), None
        if ptr and _lib is not None:
            _lib.td_free_compressible(C.c_void_p(ptr))


def _base_lp(v):
    """base_LP -> the td_config field (-1: no base).  The reference compares the live count with `<= 0`, so a
    fraction would add a leak (5.5 ends after 6 leaks) and a negative count would end every step: both rejected."""
    if v is None:
        return -1
    try:
        iv = int(v)
    except (TypeError, ValueError, OverflowError):
        raise ValueError("base_LP must be None or a non-negative integer, got %r" % (v,))
    if iv != v or iv < 0:
        raise ValueError("base_LP must be None or a non-negative integer, got %r" % (v,))
    return iv


def upgrade_step(max_episode_steps, enemy_upgrade_at):
    """First step count from which summoned enemies are level 1 (td_upgrade_step; 2**31 - 1: never)."""
    return lib().td_upgrade_step(int(max_episode_steps), float(enemy_upgrade_at))


def config_struct(cfg=None, hyper=None):
    """Snapshot a reference-style config object / dict into a td_config."""
    cfg = params.config if cfg is None else cfg
    d = cfg if isinstance(cfg, dict) else cfg.__dict__
    hyper = params.hyper_parameters.__dict__ if hyper is None else hyper
    for key, want in (("enemy_types", NT), ("tower_types", NT), ("max_enemy_lv", 1), ("max_tower_lv", 1)):
        if d.get(key, want) != want:
            raise ValueError("this build supports %s == %d only" % (key, want))
    if hyper.get("max_cluster_length", CLUSTER) != CLUSTER or hyper.get("max_num_of_roads", ROADS) != ROADS:
        raise ValueError("max_cluster_length / max_num_of_roads are fixed at 8 / 3")
    c = TdConfig()
    lib().td_default_config(C.byref(c))
    for name in _TABLES_F64 + _TABLES_I32:
        if name in d:
            for t in range(NT):
                for l in range(NLV):
                    getattr(c, name)[t][l] = d[name][t][l]
    for name in _SCALARS_F64 + _SCALARS_I32:
        if name in d and name not in ("base_LP", "pad_"):
            setattr(c, name, d[name])
    if "base_LP" in d:
        c.base_LP = _base_lp(d["base_LP"])
    # the observation divides by these (TDBoard.py:118,123-125,142); the reference raises ZeroDivisionError there
    if not c.max_cost > 0:
        raise ValueError("max_cost must be > 0 (and not NaN), got %r" % (c.max_cost,))
    if any(c.enemy_cost[t][0] == 0 or c.enemy_cost[t][0] != c.enemy_cost[t][0] for t in range(NT)):
        raise ValueError("enemy_cost[t][0] must not be 0 or NaN, got %r" % ([c.enemy_cost[t][0] for t in range(NT)],))
    c.max_episode_steps = int(hyper.get("max_episode_steps", 1200))
    return c


def _ptr(x):
    """Device/host pointer of a torch tensor / numpy array / int / None."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        assert x.flags["C_CONTIGUOUS"]
        return x.ctypes.data
    assert x.is_contiguous(), "tensor must be contiguous"
    return x.data_ptr()


def map_from_planes(map_size, num_roads, start, end, road_bits, dist, dirs):
    """Build a TdMap from reference-style planes (road bits map[0..3], map[4], map[5])."""
    m = TdMap()
    cells = map_size * map_size
    m.map_size, m.num_roads, m.end = int(map_size), int(num_roads), int(end)
    for i in range(ROADS):
        m.start[i] = int(start[i]) if i < num_roads else 0
    road_bits = np.asarray(road_bits, dtype=np.uint8).reshape(-1)
    dist = np.asarray(dist).reshape(-1)
    dirs = np.asarray(dirs, dtype=np.uint8).reshape(-1)
    packed = (road_bits & 15) | ((dirs & 3) << 4)
    C.memmove(m.cells, packed.astype(np.uint8).ctypes.data, cells)
    C.memmove(m.dist, dist.astype(np.uint8).ctypes.data, cells)
    m.max_dist = int(dist.max())
    return m


class Engine(object):
    """One td_handle: n_envs game instances of one kind / map size on one CUDA device."""

    def __init__(self, kind, map_size, n_envs, device=0, cfg=None):
        self._lib = lib()
        self._h = C.c_void_p()
        self.kind = KINDS[kind] if isinstance(kind, str) else int(kind)
        self.map_size, self.n_envs, self.device = int(map_size), int(n_envs), int(device)
        self.cells = self.map_size * self.map_size
        c = cfg if isinstance(cfg, TdConfig) else config_struct(cfg)
        rc = self._lib.td_create(C.byref(c), self.kind, self.map_size, self.n_envs, self.device, C.byref(self._h))
        if rc != 0:
            raise TdError(rc, self._lib.td_last_error(None).decode())
        lay = TdLayout()
        self._check(self._lib.td_get_layout(self._h, C.byref(lay)))
        self.layout = lay
        self.n_maps = 0

    def _check(self, rc):
        if rc != 0:
            raise TdError(rc, self._lib.td_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.td_destroy(self._h)
            self._h = None

    __del__ = close

    # -- configuration / maps ---------------------------------------------------------------
    def set_config(self, cfg=None):
        c = cfg if isinstance(cfg, TdConfig) else config_struct(cfg)
        self._check(self._lib.td_set_config(self._h, C.byref(c)))

    def upload_maps(self, maps):
        """maps: ctypes array of TdMap or a list of TdMap."""
        if isinstance(maps, (list, tuple)):
            arr = (TdMap * len(maps))()
            for i, m in enumerate(maps):
                C.memmove(C.byref(arr, i * C.sizeof(TdMap)), C.byref(m), C.sizeof(TdMap))
            maps = arr
        self._check(self._lib.td_upload_maps(self._h, maps, len(maps)))
        self.n_maps = len(maps)

    def set_map_stride(self, stride):
        self._check(self._lib.td_set_map_stride(self._h, int(stride)))

    def set_option(self, option, value):
        """Tuning knobs of the handle (TD_OPT_* of td_b200.h): "host_chunks", "host_graph", "generic_kernels", "host_chain", "host_first_chunk", "host_zero_copy"."""
        self._check(self._lib.td_set_option(self._h, OPTIONS[option] if isinstance(option, str) else int(option), int(value)))

    def set_difficulty(self, difficulty):
        self._check(self._lib.td_set_difficulty(self._h, int(difficulty)))

    def seed_opponent(self, states, first_env=0):
        """states: uint32 array [n, 625] = random.Random(s).getstate()[1] per env."""
        states = np.ascontiguousarray(states, dtype=np.uint32)
        assert states.ndim == 2 and states.shape[1] == 625
        self._check(self._lib.td_seed_opponent(self._h, states.ctypes.data, int(first_env), states.shape[0]))

    def seed_opponent_python(self, seeds, first_env=0):
        """Env i gets the generator state of CPython's random.seed(int(seeds[i]))."""
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32).reshape(-1)
        self._check(self._lib.td_seed_opponent_python(self._h, seeds.ctypes.data, int(first_env), seeds.shape[0]))

    def get_opponent(self, first_env=0, n=None):
        n = self.n_envs - first_env if n is None else n
        out = np.zeros((n, 625), dtype=np.uint32)
        self._check(self._lib.td_get_opponent(self._h, int(first_env), int(n), out.ctypes.data))
        return out

    # -- stepping -----------------------------------------------------------------------------
    def reset(self, mask=None, map_ids=None, obs=None, stream=0):
        self._check(self._lib.td_reset(self._h, _ptr(mask), _ptr(map_ids), _ptr(obs), stream))

    @staticmethod
    def make_io(def_action=None, atk_action=None, opponent=None, multi_action=False, auto_reset=False, obs=None,
                reward=None, done=None, win=None, allow_next=None, real_def=None, real_atk=None, fail_def=None,
                fail_atk=None, obs_incremental=False, opponent_cluster=None, packed_out=None, obs_format="f32"):
        io = TdStepIO()
        io.obs_format = OBS_FORMATS[obs_format] if isinstance(obs_format, str) else int(obs_format)
        io.packed_out_dev = _ptr(packed_out)
        io.opponent_cluster_dev = _ptr(opponent_cluster)
        io.obs_incremental = int(bool(obs_incremental))
        io.def_action_dev, io.atk_action_dev, io.opponent_dev = _ptr(def_action), _ptr(atk_action), _ptr(opponent)
        io.multi_action, io.auto_reset = int(bool(multi_action)), int(bool(auto_reset))
        io.obs_dev, io.reward_dev, io.done_dev, io.win_dev = _ptr(obs), _ptr(reward), _ptr(done), _ptr(win)
        io.allow_next_dev, io.real_def_dev, io.real_atk_dev = _ptr(allow_next), _ptr(real_def), _ptr(real_atk)
        io.fail_def_dev, io.fail_atk_dev = _ptr(fail_def), _ptr(fail_atk)
        return io

    def step(self, io, stream=0):
        self._check(self._lib.td_step(self._h, C.byref(io), stream))

    def step_host(self, io, host_io, stream=0):
        self._check(self._lib.td_step_host(self._h, C.byref(io), C.byref(host_io), stream))

    def invalidate_obs(self):
        self._check(self._lib.td_invalidate_obs(self._h))

    def observe(self, obs, stream=0, obs_format="f32"):
        fmt = OBS_FORMATS[obs_format] if isinstance(obs_format, str) else int(obs_format)
        self._check(self._lib.td_observe_as(self._h, fmt, _ptr(obs), stream))

    def action_mask(self, def_mask=None, atk_mask=None, stream=0):
        """td_action_mask: which actions the next step would carry out, from the current env records.  def_mask:
        uint8 [n, 6*L*L + 1] (TD-def, TD-2p), atk_mask: uint8 [n, 3, 4] (TD-atk, TD-2p); device buffers, either
        may be None, not both."""
        self._check(self._lib.td_action_mask(self._h, _ptr(def_mask), _ptr(atk_mask), stream))

    # -- state / statistics ---------------------------------------------------------------------
    def get_state_raw(self, first_env=0, n=None):
        n = self.n_envs - first_env if n is None else n
        blob = np.zeros((n, self.layout.record_bytes), dtype=np.uint8)
        self._check(self._lib.td_get_state(self._h, int(first_env), int(n), blob.ctypes.data))
        return blob

    def set_state_raw(self, blob, first_env=0):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self._check(self._lib.td_set_state(self._h, int(first_env), blob.shape[0], blob.ctypes.data))

    def decode_state(self, blob_row):
        """One env record -> dict in the format of the oracle's state_dict()."""
        lay = self.layout
        hdr = blob_row[:64].view(HEADER_DTYPE)[0]
        nt, ne = int(hdr["n_towers"]), int(hdr["n_enemies"])
        tw = blob_row[lay.off_towers:lay.off_towers + 16 * nt].view(TOWER_DTYPE)
        en = blob_row[lay.off_enemies:lay.off_enemies + 24 * ne].view(ENEMY_DTYPE)
        return dict(header=hdr, towers=tw, enemies=en,
                    map6=blob_row[lay.off_map6:lay.off_map6 + self.cells].astype(np.int32))

    def stats(self, stream=0):
        s = TdStats()
        self._check(self._lib.td_get_stats(self._h, C.byref(s), stream))
        return {n: getattr(s, n) for n, _ in TdStats._fields_}

    def reset_stats(self, stream=0):
        self._check(self._lib.td_reset_stats(self._h, stream))
