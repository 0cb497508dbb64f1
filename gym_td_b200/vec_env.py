"""TDVecEnv: N independent gym-TD instances advanced in lockstep on one B200.

The batched counterpart of the reference's `gym.vector.AsyncVectorEnv([make_fn] * n)` use
(train/main.py:345): same per-env semantics as TDDefense / TDAttack / TDMulti.step, a leading
env dimension on every tensor, finished envs restarted in place on the next map of the pool.
All tensors live on the GPU; `step()` launches one fused kernel and returns views of
pre-allocated output tensors (valid until the next step).

Seeding contract (SURVEY.md 8d): env with global index g = env_offset + i uses the first valid
map seed >= seed + g (numpy RandomState stream, num_roads drawn first) and a scripted-opponent
generator in the state of CPython's random.seed(seed + g), which keeps running across episodes
like the reference's global `random` module does.
"""

import numpy as np
import torch

from . import engine as E
from . import mapgen, params


class _Info(dict):
    """Lazy info dict: RealAction / Win / FailCode are tensor views, AllowNextMove is computed on access."""

    def __init__(self, env):
        super().__init__()
        k = env.kind
        self._allow = env._allow
        self._kind = k
        self["Win"] = env.win
        if k == "def":
            self["RealAction"], self["FailCode"] = env.real_def, env.fail_def
        elif k == "atk":
            self["RealAction"], self["FailCode"] = env.real_atk, env.fail_atk
        else:
            self["RealAction"] = {"Attacker": env.real_atk, "Defender": env.real_def}
            self["FailCode"] = {"Attacker": env.fail_atk, "Defender": env.fail_def}
        self["AllowNextMoveBits"] = env._allow          # bit0 defender, bit1 attacker

    def __missing__(self, key):
        if key != "AllowNextMove":
            raise KeyError(key)
        a = self._allow
        if self._kind == "def":
            v = (a & 1).bool()
        elif self._kind == "atk":
            v = (a & 2).bool()
        else:
            v = {"Attacker": (a & 2).bool(), "Defender": (a & 1).bool()}
        self[key] = v
        return v

    def __contains__(self, key):
        return key == "AllowNextMove" or dict.__contains__(self, key)


class TDVecEnv(object):
    def __init__(self, kind, map_size, num_envs, seed=0, device=0, difficulty=1, auto_reset=True, env_offset=0,
                 n_maps=None, scripted_opponent=True, multi_action=None, cfg=None, mapgen_threads=None,
                 incremental_obs=False, obs_format="f32", obs_memory="auto"):
        if kind not in E.KINDS:
            raise ValueError("kind must be one of %r" % (sorted(E.KINDS),))
        self.kind, self.map_size, self.num_envs = kind, int(map_size), int(num_envs)
        self.device = torch.device("cuda", device)
        self.auto_reset = bool(auto_reset)
        # incremental_obs: `self.obs` is only ever written by this env, so the step may update it in place instead
        # of rewriting all 45 planes (td_step_io.obs_incremental; the tensor is bit-identical either way).  Leave
        # it off if you write into `env.obs` yourself.
        self.incremental_obs = bool(incremental_obs)
        self.multi_action = params.hyper_parameters.allow_multiple_actions if multi_action is None else bool(multi_action)
        if kind == "atk":
            self.multi_action = False
        self.engine = E.Engine(kind, map_size, num_envs, device=device, cfg=cfg)
        n_maps = self.num_envs if n_maps is None else int(n_maps)
        base = (int(seed) + int(env_offset)) & 0xFFFFFFFF
        seeds = (np.arange(n_maps, dtype=np.uint64) + base).astype(np.uint32)
        maps, self.map_seeds, _ = mapgen.generate_batch(seeds, map_size, threads=mapgen_threads)
        self.engine.upload_maps(maps)
        self.engine.set_map_stride(1)
        self.num_roads = np.array([maps[i].num_roads for i in range(n_maps)], dtype=np.int32)
        self.scripted = bool(scripted_opponent and kind != "2p")
        self.difficulty = int(difficulty)
        if self.scripted:
            self.engine.set_difficulty(difficulty)
            self.engine.seed_opponent_python((np.arange(num_envs, dtype=np.uint64) + base).astype(np.uint32))
        N, L, dev = self.num_envs, self.map_size, self.device
        # obs_format: "f32" is the reference's tensor; "bf16" / "u8" are the opt-in reduced-precision planes (SURVEY 8(f)
        # f4): same (N, 45, L, L) layout, the float32 value rounded to bfloat16 / quantised to rint(min(255 v, 255))
        if obs_format not in E.OBS_FORMATS:
            raise ValueError("obs_format must be one of %r" % (sorted(E.OBS_FORMATS),))
        if obs_format != "f32" and (self.multi_action or L not in (10, 20, 30) or incremental_obs):
            raise ValueError("reduced-precision observations: boards 10 / 20 / 30, Discrete actions, full writes")
        self.obs_format = obs_format
        self._obs_dtype = {"f32": torch.float32, "bf16": torch.bfloat16, "u8": torch.uint8}[obs_format]
        self._obs = self._alloc_obs((N, E.NCH, L, L), dev, obs_memory)
        # the small per-step outputs live in one slab (mirrored by one pinned host slab in step_host, so that
        # td_step_host moves them with a single device->host copy)
        self._layout, off = {}, 0
        fields = [("reward", (N,), torch.float64)]
        if kind != "atk":
            fields += [("real_def", (N, 6, L, L) if self.multi_action else (N,), torch.int64), ("fail_def", (N,), torch.int32)]
        if kind != "def":
            fields += [("real_atk", (N, E.ROADS, E.CLUSTER), torch.int64), ("fail_atk", (N, 4), torch.int32)]
        fields += [("done", (N,), torch.uint8), ("win", (N,), torch.int8), ("allow", (N,), torch.uint8)]
        for name, shape, dtype in fields:
            nbytes = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
            self._layout[name] = (off, nbytes, shape, dtype)
            off += (nbytes + 255) & ~255
        # (the Box RealAction of a multi-action batch is hundreds of MB of 0 / 1 int64: it compresses like the observation)
        self._slab, self.slab_memory = self._alloc_bytes(off, dev, obs_memory if obs_memory != "auto" or off >= (32 << 20) else "plain")
        view = lambda slab, k: slab[self._layout[k][0]:self._layout[k][0] + self._layout[k][1]].view(
            self._layout[k][3]).view(self._layout[k][2])
        self._view = view
        opt = lambda k: view(self._slab, k) if k in self._layout else None
        self.reward, self.real_def, self.real_atk = view(self._slab, "reward"), opt("real_def"), opt("real_atk")
        self.fail_atk, self.fail_def = opt("fail_atk"), opt("fail_def")
        self._done, self.win, self._allow = view(self._slab, "done"), view(self._slab, "win"), view(self._slab, "allow")
        self._allow.fill_(3)                                                 # AllowNextMove starts True (train/main.py:87)
        self._host = None
        self._io_cache = None
        self._hio_cache = None
        self._host_io = None
        self._host_sig = None
        self._masks = None

    @staticmethod
    def _alloc_bytes(nbytes, dev, mode):
        """(zero-filled uint8 tensor of nbytes, what it lives in).  mode "compressible" / "auto": a compressible
        allocation when the device grants one (td_alloc_compressible), else -- "auto" only -- ordinary torch memory."""
        if mode in ("compressible", "auto"):
            try:
                buf = E.CompressibleBuffer(nbytes, dev.index if dev.index is not None else 0)
                if buf.compressed or mode == "compressible":
                    return buf.tensor((nbytes,), torch.uint8), "compressible" if buf.compressed else "plain (compression not granted)"
            except E.TdError:
                if mode == "compressible":
                    raise
        return torch.zeros(nbytes, dtype=torch.uint8, device=dev), "plain"

    def _alloc_obs(self, shape, dev, obs_memory):
        """The observation tensor.  obs_memory = "compressible": device memory from a compressible allocation
        (td_alloc_compressible: B200 compresses the mostly-zero / broadcast planes in L2 on their way to HBM, lossless
        and invisible to readers; the step writes it 11 - 23 % faster and a reader streams it 22 % faster, DESIGN.md
        7.2h); "plain": an ordinary torch allocation; "auto": compressible for batches of 32 MB and more when the
        device grants it, else plain -- and plain for in-place updates on 10x10 boards, the one case that measures
        slower on compressed lines (0.167 -> 0.175 ms; every other board size and mode gains or ties).
        `self.obs_memory` says what was used."""
        if obs_memory not in ("auto", "compressible", "plain"):
            raise ValueError('obs_memory must be "auto", "compressible" or "plain"')
        nbytes = int(np.prod(shape)) * torch.empty((), dtype=self._obs_dtype).element_size()
        small_inplace = self.incremental_obs and self.map_size <= 10
        mode = obs_memory if obs_memory != "auto" else ("auto" if nbytes >= (32 << 20) and not small_inplace else "plain")
        flat, self.obs_memory = self._alloc_bytes(nbytes, dev, mode)
        return flat.view(self._obs_dtype).view(shape)

    # `obs` is the tensor every step writes.  Rebinding it (env.obs = other) is allowed; the in-place observation
    # update (incremental_obs) then starts over with a full write, also when the new tensor reuses the old address.
    @property
    def obs(self):
        return self._obs

    @obs.setter
    def obs(self, t):
        N, L = self.num_envs, self.map_size
        if tuple(t.shape) != (N, E.NCH, L, L) or t.dtype != self._obs_dtype or not t.is_cuda or not t.is_contiguous():
            raise ValueError("obs must be a contiguous CUDA %s tensor of shape %r" % (self._obs_dtype, (N, E.NCH, L, L)))
        self._obs = t
        self.engine.invalidate_obs()

    def invalidate_obs(self):
        """Call after writing into `env.obs` yourself while incremental_obs is on."""
        self.engine.invalidate_obs()

    # -- spaces-like metadata -------------------------------------------------------------------
    @property
    def observation_shape(self):
        return (self.num_envs, E.NCH, self.map_size, self.map_size)

    def empty_action(self):
        """Batched TD*.empty_action() (TDDefense.py:28-32, TDAttack.py:24-25, TDMulti.py:30-40)."""
        N, L = self.num_envs, self.map_size
        d = (torch.zeros((N, 6, L, L), dtype=torch.int64, device=self.device) if self.multi_action
             else torch.full((N,), 6 * L * L, dtype=torch.int64, device=self.device))
        a = torch.full((N, E.ROADS, E.CLUSTER), E.NT, dtype=torch.int64, device=self.device)
        return {"def": d, "atk": a, "2p": {"Attacker": a, "Defender": d}}[self.kind]

    # -- core -----------------------------------------------------------------------------------
    def reset(self, mask=None, map_ids=None):
        s = torch.cuda.current_stream(self.device).cuda_stream
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if map_ids is not None:
            map_ids = map_ids.to(device=self.device, dtype=torch.int32).contiguous()
        if self.obs_format == "f32":
            self.engine.reset(mask=mask, map_ids=map_ids, obs=self.obs, stream=s)
        else:                                   # td_reset writes float32: restart, then one observation pass
            self.engine.reset(mask=mask, map_ids=map_ids, obs=None, stream=s)
            self.engine.observe(self.obs, s, self.obs_format)
        return self.obs

    def _split(self, action):
        if self.kind == "def":
            return action, None
        if self.kind == "atk":
            return None, action
        return action["Defender"], action["Attacker"]

    def _io(self, d, a, opponent=None):
        """The td_step_io of this env: output pointers are fixed, only the action pointers change per call."""
        io = self._io_cache
        if io is None:
            io = self._io_cache = E.Engine.make_io(
                multi_action=self.multi_action, auto_reset=self.auto_reset, obs=self.obs, reward=self.reward,
                done=self._done, win=self.win, allow_next=self._allow, real_def=self.real_def,
                real_atk=self.real_atk, fail_def=self.fail_def, fail_atk=self.fail_atk)
        io.auto_reset = int(self.auto_reset)
        io.obs_incremental = int(self.incremental_obs)
        io.obs_format = E.OBS_FORMATS[self.obs_format]
        io.obs_dev = E._ptr(self.obs)
        io.def_action_dev = d.data_ptr() if d is not None else None
        io.atk_action_dev = a.data_ptr() if a is not None else None
        io.opponent_dev = opponent.data_ptr() if opponent is not None else None
        return io

    def _check(self, d, a):
        N, L = self.num_envs, self.map_size
        if d is not None:
            want = (N, 6, L, L) if self.multi_action else (N,)
            if tuple(d.shape) != want or d.dtype != torch.int64 or not d.is_cuda or not d.is_contiguous():
                raise AssertionError("defender action must be a contiguous CUDA int64 tensor of shape %r" % (want,))
        if a is not None:
            want = (N, E.ROADS, E.CLUSTER)
            if tuple(a.shape) != want or a.dtype != torch.int64 or not a.is_cuda or not a.is_contiguous():
                raise AssertionError("attacker action must be a contiguous CUDA int64 tensor of shape %r" % (want,))

    def step(self, action, opponent=None):
        """One lockstep step.  Returns (obs, reward, done, info) -- tensors with a leading env dim."""
        d, a = self._split(action)
        self._check(d, a)
        self.engine.step(self._io(d, a, opponent), torch.cuda.current_stream(self.device).cuda_stream)
        return self.obs, self.reward, self._done.view(torch.bool), self.info()

    def info(self):
        """info dict of the last step.  Values are views of the output tensors; the AllowNextMove masks are
        derived from the packed bits only when they are read (no extra kernels on the step path)."""
        return _Info(self)

    def action_mask(self):
        """Which actions the next step() would carry out, computed on the current stream from the current state
        (td_action_mask; nothing runs unless this is called).  TD-def: a bool [N, 6*L*L + 1] mask of the Discrete
        actions, entry a = the action would come back as RealAction a (the no-op is always True); in multi-action mode
        the [N, 6, L, L] view of its first 6*L*L entries, entry (ch, r, c) = a Box action whose only flag is (ch, r, c)
        would succeed.  TD-atk: bool [N, 3, 4], entry (road, type) = a cluster whose only slot is that enemy type on
        that road would summon it (each slot alone: later slots of one cluster see a smaller purse).  TD-2p:
        {"Attacker": ..., "Defender": ...}.  Views of buffers allocated on the first call, valid until the next call."""
        N, L = self.num_envs, self.map_size
        if self._masks is None:
            self._masks = (torch.zeros((N, 6 * L * L + 1), dtype=torch.uint8, device=self.device) if self.kind != "atk" else None,
                           torch.zeros((N, E.ROADS, E.NT), dtype=torch.uint8, device=self.device) if self.kind != "def" else None)
        d, a = self._masks
        self.engine.action_mask(d, a, torch.cuda.current_stream(self.device).cuda_stream)
        if d is not None:
            d = d.view(torch.bool)
            if self.multi_action:
                d = d[:, :-1].view(N, 6, L, L)
        if a is not None:
            a = a.view(torch.bool)
        return {"def": d, "atk": a, "2p": {"Attacker": a, "Defender": d}}[self.kind]

    # -- host-buffer path (what a numpy-facing gym caller uses) ------------------------------------
    def _host_buffers(self):
        """Page-locked host side of step_host.  The small outputs arrive as one packed record per env
        (td_step_packed, 32 B for TD-def, 256 B otherwise) that the step kernel stores straight into this
        buffer -- no device->host copy; the dict exposes the fields as (strided) views of it."""
        if self._host is None:
            N = self.num_envs
            stride = 32 if self.kind == "def" else 256
            packed = torch.zeros((N, stride), dtype=torch.uint8).pin_memory()
            f = lambda lo, hi, dt: packed[:, lo:hi].view(dt)
            h = dict(packed=packed, reward=f(0, 8, torch.float64)[:, 0], done=packed[:, 20], win=f(21, 22, torch.int8)[:, 0],
                     allow=packed[:, 22], real_def=None, fail_def=None, real_atk=None, fail_atk=None, obs=None)
            if self.kind != "atk":
                h["fail_def"] = f(16, 20, torch.int32)[:, 0]
                if not self.multi_action:
                    h["real_def"] = f(8, 16, torch.int64)[:, 0]
                else:                                  # [N, 6, L, L]: too large for the record, copied on request
                    h["real_def"] = torch.empty(self.real_def.shape, dtype=torch.int64).pin_memory()
            if self.kind != "def":
                h["fail_atk"] = f(32, 48, torch.int32)
                h["real_atk"] = f(64, 256, torch.int64).view(N, E.ROADS, E.CLUSTER)
            h["def_dev"] = torch.zeros_like(self.real_def) if self.real_def is not None else None
            h["atk_dev"] = torch.zeros_like(self.real_atk) if self.real_atk is not None else None
            self._host = h
        return self._host

    def step_host(self, action, want_obs=False):
        """Host in, host out through td_step_host: `action` are pinned CPU int64 tensors; the small outputs land
        in pinned host memory while the kernel runs (and the observation is copied when want_obs); the stream
        is synchronised before the call returns.  Returns a dict of host tensors (views, valid until the next call)."""
        h = self._host_buffers()
        d, a = self._split(action)
        if want_obs and h["obs"] is None:
            h["obs"] = torch.empty(self.obs.shape, dtype=self._obs_dtype).pin_memory()
        # the device side of the call never changes between calls (the actions land in the env's own staging tensors):
        # the td_step_io is rebuilt only when the observation tensor or a mode flag changed (4-6 us of Python per call
        # were 2 % of a 65,536-env step)
        sig = (self.obs.data_ptr(), self.auto_reset, self.incremental_obs, self.obs_format)
        if sig != self._host_sig:
            src = self._io(h["def_dev"] if d is not None else None, h["atk_dev"] if a is not None else None)
            self._host_io = E.TdStepIO.from_buffer_copy(src)
            self._host_sig = sig
        io = self._host_io
        hio = self._hio_cache
        if hio is None:
            hio = self._hio_cache = E.TdHostIO()
            hio.packed_host = h["packed"].data_ptr()
            if self.kind != "atk" and self.multi_action:
                hio.real_def_host = h["real_def"].data_ptr()
        if d is not None:
            hio.def_action_host = d.data_ptr()
        if a is not None:
            hio.atk_action_host = a.data_ptr()
        hio.obs_host = h["obs"].data_ptr() if want_obs else None
        self.engine.step_host(io, hio, torch.cuda.current_stream(self.device).cuda_stream)
        return h

    def host_bytes_per_step(self, want_obs=False):
        N, L = self.num_envs, self.map_size
        h2d = 0
        if self.kind != "atk":
            h2d += self.real_def.numel() * 8
        if self.kind != "def":
            h2d += N * 24 * 8
        d2h = N * (32 if self.kind == "def" else 256)          # packed records, written by the kernel itself
        if self.kind != "atk" and self.multi_action:
            d2h += self.real_def.numel() * 8
        if want_obs:
            d2h += N * E.NCH * L * L * self.obs.element_size()
        return h2d, d2h

    # -- statistics -------------------------------------------------------------------------------
    def stats(self):
        s = self.engine.stats(torch.cuda.current_stream(self.device).cuda_stream)
        if s["overflow_envs"]:
            raise E.TdError(-5, "%d env(s) exceeded the tower/enemy capacity; their results are invalid"
                            % s["overflow_envs"])
        return s

    def allreduce_stats(self):
        """Episode statistics summed over all ranks (NCCL all_reduce when torch.distributed is up)."""
        from . import dist
        return dist.reduce_stats(self.stats(), self.device)

    # -- compact observations (SURVEY.md 8(f) f4) ----------------------------------------------------------------
    def snapshot(self, out=None):
        """Copy the current env records (record_bytes per env, ~2.5 KB at L=10 instead of the 18 KB observation)
        into `out` ([num_envs, record_bytes] uint8 CUDA tensor, allocated when None).  The observation can be
        rebuilt from a record at any time with observe_snapshot()."""
        rb = self.engine.layout.record_bytes
        if out is None:
            out = torch.empty((self.num_envs, rb), dtype=torch.uint8, device=self.device)
        assert out.is_cuda and out.is_contiguous() and out.numel() == self.num_envs * rb
        eng = self.engine
        eng._check(eng._lib.td_snapshot(eng._h, out.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream))
        return out

    def observe_snapshot(self, records, out=None):
        """(n, 45, L, L) float32 observations of `records` ([n, record_bytes] uint8 CUDA tensor of stored records)."""
        rb = self.engine.layout.record_bytes
        records = records.view(-1, rb)
        n, L = records.shape[0], self.map_size
        assert records.is_cuda and records.is_contiguous() and records.dtype == torch.uint8
        if out is None:
            out = torch.empty((n, E.NCH, L, L), dtype=torch.float32, device=self.device)
        eng = self.engine
        eng._check(eng._lib.td_observe_snapshot(eng._h, records.data_ptr(), n, out.data_ptr(),
                                                torch.cuda.current_stream(self.device).cuda_stream))
        return out

    # -- checkpoint / resume (SURVEY.md section 5: the reference has no env-state checkpoint) ------------------
    def state_dict(self):
        """Everything needed to continue bit-identically: env records, opponent generators, last AllowNextMove bits.
        (The map pool and config are construction arguments and are not part of the snapshot.)"""
        torch.cuda.synchronize(self.device)
        d = {"kind": self.kind, "map_size": self.map_size, "num_envs": self.num_envs,
             "records": torch.from_numpy(self.engine.get_state_raw()), "allow": self._allow.cpu().clone()}
        try:
            d["opponent"] = torch.from_numpy(self.engine.get_opponent().astype(np.int64))
        except E.TdError:
            d["opponent"] = None
        return d

    def load_state_dict(self, d):
        if (d["kind"], d["map_size"], d["num_envs"]) != (self.kind, self.map_size, self.num_envs):
            raise ValueError("snapshot is for a different env batch")
        torch.cuda.synchronize(self.device)
        self.engine.set_state_raw(d["records"].numpy())
        if d.get("opponent") is not None:
            # seed_opponent resets the cached-word count of every record, which is what a restore needs:
            # the cached words are re-read from the restored generator state on the first draw
            self.engine.seed_opponent(d["opponent"].numpy().astype(np.uint32))
        self._allow.copy_(d["allow"].to(self.device))
        self.engine.observe(self.obs, torch.cuda.current_stream(self.device).cuda_stream, self.obs_format)
        return self.obs

    def close(self):
        self.engine.close()
