"""Kernel choice of the engine (td_engine.cu, step_kernel): every step kernel the table can pick -- each env kind,
board 10 / 20 / 30 / 13, Discrete and multi-action, float32 full write, float32 in-place update, bfloat16 and uint8
observations, opponent-specialised and generic kernels -- computes the same step as the generic full-write float32
kernel of a twin handle on the same maps and seeds, across auto-resets.  The retired tuning options 3 and 4 are
refused."""
import numpy as np
import pytest

from gym_td_b200 import engine as E
from gym_td_b200 import mapgen
from tests import parity_util as PU
from tests.test_gpu_constructed_states import bf16_reference, u8_reference

pytestmark = pytest.mark.gpu

N, STEPS = 12, 40
CFG = dict(max_episode_steps=15)          # every env restarts (auto-reset) at least twice within the run


def _legs(kind, L):
    """(multi, observation, opponent) of every table entry the handle can reach."""
    for multi in ((False,) if kind == "atk" else (False, True)):
        for obs in ("f32", "in_place") + (("bf16", "u8") if L in (10, 20, 30) and not multi else ()):
            for opp in (("generic",) if kind == "2p" else ("specialised", "generic")):
                yield multi, obs, opp


class _Run:
    """One handle with its own output buffers.  `generic`: never the opponent-specialised kernels."""

    def __init__(self, kind, L, maps, seeds, multi, obs, generic):
        import torch
        self.kind, self.L, self.multi, self.fmt = kind, L, multi, obs
        self.eng = E.Engine(kind, L, N, cfg=PU.make_config(**CFG))
        self.eng.upload_maps(maps)
        if kind != "2p":
            self.eng.seed_opponent_python(seeds)          # difficulty 1: the scripted opponent on the device generator
        if generic:
            self.eng.set_option("generic_kernels", 1)
        dt = {"bf16": torch.bfloat16, "u8": torch.uint8}.get(obs, torch.float32)
        self.obs = torch.empty((N, 45, L, L), dtype=dt, device="cuda")
        self.out = dict(
            reward=torch.zeros(N, dtype=torch.float64, device="cuda"),
            done=torch.zeros(N, dtype=torch.uint8, device="cuda"),
            win=torch.zeros(N, dtype=torch.int8, device="cuda"),
            allow_next=torch.zeros(N, dtype=torch.uint8, device="cuda"),
            real_def=torch.zeros((N, 6, L, L) if multi else (N,), dtype=torch.int64, device="cuda"),
            real_atk=torch.zeros((N, 3, 8), dtype=torch.int64, device="cuda"),
            fail_def=torch.zeros(N, dtype=torch.int32, device="cuda"),
            fail_atk=torch.zeros((N, 4), dtype=torch.int32, device="cuda"),
        )
        self.eng.reset(obs=self.obs if dt == torch.float32 else None)

    def step(self, def_act, atk_act):
        import torch
        io = E.Engine.make_io(def_action=def_act if self.kind != "atk" else None,
                              atk_action=atk_act if self.kind != "def" else None, multi_action=self.multi,
                              auto_reset=True, obs=self.obs, obs_incremental=self.fmt == "in_place",
                              obs_format=self.fmt if self.fmt in ("bf16", "u8") else "f32", **self.out)
        self.eng.step(io, torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize("L", [10, 20, 30, 13])
@pytest.mark.parametrize("kind", ["def", "atk", "2p"])
def test_every_step_kernel_matches_the_generic_full_write(kind, L):
    import torch
    seeds = (np.arange(N, dtype=np.uint32) * 13 + 7 * L + 3).astype(np.uint32)
    maps, seeds, _ = mapgen.generate_batch(seeds, L)
    legs = list(_legs(kind, L))
    for multi in sorted({m for m, _, _ in legs}):
        twin = _Run(kind, L, maps, seeds, multi, "f32", generic=True)
        runs = {(o, p): _Run(kind, L, maps, seeds, multi, o, generic=p == "generic") for m, o, p in legs if m == multi}
        rs = np.random.RandomState(L + 100 * multi)
        restarts = 0
        for step in range(STEPS):
            if multi:
                d = (rs.rand(N, 6, L, L) < 0.02).astype(np.int64)
            else:
                d = rs.randint(0, 6 * L * L + 1, size=N).astype(np.int64)
            def_act = torch.from_numpy(d).cuda()
            atk_act = torch.from_numpy(rs.randint(0, 5, size=(N, 3, 8)).astype(np.int64)).cuda()
            twin.step(def_act, atk_act)
            for r in runs.values():
                r.step(def_act, atk_act)
            torch.cuda.synchronize()
            want = twin.obs.cpu().numpy()
            restarts += int(twin.out["done"].sum())
            for (obs, opp), r in runs.items():
                tag = (kind, L, multi, obs, opp, step)
                for name, t in twin.out.items():
                    assert torch.equal(r.out[name], t), tag + (name,)
                got = r.obs.cpu()
                if obs == "bf16":
                    assert np.array_equal(got.view(torch.int16).numpy().view(np.uint16), bf16_reference(want)), tag
                elif obs == "u8":
                    assert np.array_equal(got.numpy(), u8_reference(want)), tag
                else:
                    assert np.array_equal(got.numpy().view(np.uint32), want.view(np.uint32)), tag
        assert restarts >= 2 * N, restarts
        records, stats = twin.eng.get_state_raw(), twin.eng.stats()
        for (obs, opp), r in runs.items():
            assert np.array_equal(r.eng.get_state_raw(), records), (kind, L, multi, obs, opp)
            assert r.eng.stats() == stats, (kind, L, multi, obs, opp)
            r.eng.close()
        twin.eng.close()


def test_retired_options_are_refused():
    """TD_OPT 3 and 4 (shared-memory experiments) are gone: td_set_option rejects them like any unknown option."""
    eng = E.Engine("def", 10, 4)
    for option in (3, 4):
        assert eng._lib.td_set_option(eng._h, option, 64) == -1            # TD_E_INVALID
        with pytest.raises(E.TdError):
            eng.set_option(option, 64)
    for name in ("step_smem_kb", "obs_smem_kb"):
        with pytest.raises(KeyError):
            eng.set_option(name, 64)
    eng.set_option("host_chunks", 2)                                         # the other options still apply
    eng.close()
