"""Live differential test: the C oracle against the unmodified reference, step by step (any checkout
that has the reference, see oracle/ref_loader.py; skipped elsewhere -- the golden fixtures cover those)."""
import numpy as np
import pytest

from oracle import ref_loader

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason=ref_loader.MISSING)


def test_reference_self_test_passes_under_the_stub():
    """python -m gym_TD.envs.TDBoard: the reference's own golden check (TDBoard.py:674-756)."""
    import runpy
    import warnings
    ref_loader.load()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        runpy.run_module("gym_TD.envs.TDBoard", run_name="__main__")     # asserts inside, prints 'passed'


def test_oracle_equals_reference_on_fresh_trajectories():
    from oracle import ref_harness as RH
    from oracle import validate_oracle as V
    ref_loader.load()
    np.seterr(all="ignore")
    rs = np.random.RandomState(2024)
    n = 0
    n += V.run_def(10, 7001, rs, 1, True, max_steps=500)
    n += V.run_def(20, 7002, rs, 0, False, max_steps=300)
    n += V.run_atk(10, 7003, rs, 1, max_steps=500)
    n += V.run_atk(30, 7004, rs, 2, max_steps=200)
    n += V.run_multi(20, 7005, rs, max_steps=300)
    RH.set_multiple_actions(True)
    try:
        n += V.run_def(20, 7006, rs, 1, True, max_steps=200, multi=True)
        n += V.run_multi(10, 7007, rs, max_steps=200, multi=True)
    finally:
        RH.set_multiple_actions(False)
    with RH.ref_config_override(base_LP=None, defender_action_interval=3, attacker_action_interval=2):
        n += V.run_def(10, 7008, rs, 1, True, max_steps=400)
        n += V.run_atk(10, 7009, rs, 1, max_steps=400)
    assert n > 1500


def test_oracle_equals_reference_past_the_end_of_an_episode():
    """Corner configs, each env stepped on after `done` without a reset (the reference has no done latch): summon
    levels that change only after the end (enemy_upgrade_at 1.5), an episode that ends on its first step
    (base_LP 0), and long freezes with a refund above the tower's cost."""
    from oracle import ref_harness as RH
    from oracle import validate_oracle as V
    ref_loader.load()
    np.seterr(all="ignore")
    rs = np.random.RandomState(2025)
    n = 0
    old = RH.set_max_episode_steps(20)
    try:
        with RH.ref_config_override(enemy_upgrade_at=1.5):
            n += V.run_def(10, 7101, rs, 1, True, max_steps=120, past_done=90)
            n += V.run_atk(10, 7102, rs, 0, max_steps=120, past_done=90)
            n += V.run_multi(20, 7103, rs, max_steps=120, past_done=90)
        with RH.ref_config_override(base_LP=0):
            n += V.run_def(10, 7104, rs, 0, False, max_steps=60, past_done=50)
        with RH.ref_config_override(base_LP=1, frozen_time=255, tower_destruct_return=1.5):
            n += V.run_atk(20, 7105, rs, 2, max_steps=150, past_done=100)
    finally:
        RH.set_max_episode_steps(old)
    assert n > 400
