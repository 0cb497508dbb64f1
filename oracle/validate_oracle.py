"""Differential check: C oracle (td_oracle.c) vs the unmodified reference, step by step.

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs the reference):
    python -m oracle.validate_oracle [--episodes N]
Compares, after every env step: full board state (f64 by repr, list order), the
(45, L, L) observation bit for bit, reward (f64 repr), done, and the info dict.
"""
import argparse
import random
import sys

import numpy as np

from . import ref_harness as RH
from . import ref_loader
from . import td_oracle as TO


def oracle_from_ref_env(env, cfg=None):
    o = TO.OracleEnv(cfg)
    p = RH.board_roads(env._board)
    o.init_from_planes(p["map_size"], p["num_roads"], p["start"], p["end"], p["road"], p["dist"], p["dir"])
    return o


def current_oracle_config():
    from gym_TD.envs.TDParam import config, hyper_parameters
    return TO.config_from_dict(config.__dict__, hyper_parameters.__dict__)


def check_step(tag, env, o, obs_ref, rew_ref, done_ref, out, rew_or, step):
    bad = RH.states_equal(RH.board_state(env), o.state_dict())
    obs_or = o.get_states()
    if not np.array_equal(obs_ref.view(np.uint32), obs_or.view(np.uint32)):
        ch = sorted(set(np.argwhere(obs_ref != obs_or)[:, 0].tolist()))
        bad.append("obs channels %s" % ch)
    if repr(float(rew_ref)) != repr(float(rew_or)):
        bad.append("reward %r vs %r" % (rew_ref, rew_or))
    if bool(done_ref) != bool(out.done):
        bad.append("done")
    if bad:
        raise AssertionError("%s step %d mismatch: %s" % (tag, step, bad))


def _episode_over(done, left):
    """True where a run stops: at the first `done`, or left[0] steps after it (the reference has no done latch, so a
    finished env keeps stepping).  left = [steps after done, ended]."""
    left[1] = left[1] or bool(done)
    if not left[1]:
        return False
    if left[0] == 0:
        return True
    left[0] -= 1
    return False


def run_def(L, seed, rs, difficulty=1, random_agent=True, max_steps=1200, multi=False, past_done=0):
    seed, env = RH.first_valid_seed("def", L, seed, difficulty=difficulty, random_agent=random_agent)
    o = oracle_from_ref_env(env, current_oracle_config())
    random.seed(seed)
    o.set_pyrand(random.getstate())
    o.set_nprand(env.np_random)
    tag = "def L=%d seed=%d diff=%d ra=%s multi=%s" % (L, seed, difficulty, random_agent, multi)
    assert np.array_equal(env._board.get_states(), o.get_states()), tag + " obs0"
    nop = 6 * L * L
    left = [past_done, False]
    for step in range(1, max_steps + 1):
        if multi:
            a = RH.sparse_multi_action(env._board, rs, p=0.02)
            obs, rew, done, info = RH.def_step_multi(env, a)
            out, real = o.def_step_multi(a, difficulty, not random_agent)
            assert np.array_equal(info["RealAction"], real), tag + " real_act step %d" % step
        else:
            a = RH.smart_defender_action(env._board, rs)
            obs, rew, done, info = env.step(a)
            out = o.def_step(a, difficulty, not random_agent)
            assert info["RealAction"] == out.real_def, (tag, step, info["RealAction"], out.real_def)
            assert info["FailCode"] == out.fail_def, (tag, step, a, info["FailCode"], out.fail_def)
        check_step(tag, env, o, obs, rew, done, out, out.reward, step)
        assert info["AllowNextMove"] == bool(out.allow_next_def)
        assert info["Win"] == (None if out.win < 0 else bool(out.win))
        if _episode_over(done, left):
            break
    return step


def run_atk(L, seed, rs, difficulty=1, max_steps=1200, past_done=0):
    seed, env = RH.first_valid_seed("atk", L, seed, difficulty=difficulty, random_agent=True)
    o = oracle_from_ref_env(env, current_oracle_config())
    random.seed(seed)
    o.set_pyrand(random.getstate())
    tag = "atk L=%d seed=%d diff=%d" % (L, seed, difficulty)
    left = [past_done, False]
    for step in range(1, max_steps + 1):
        mode = rs.randint(4)
        if mode == 0:
            a = rs.randint(0, 5, size=(3, 8)).astype(np.int64)
        elif mode == 1:
            a = np.full((3, 8), 4, dtype=np.int64)
        else:
            a = np.full((3, 8), 4, dtype=np.int64)
            k = rs.randint(1, 9)
            a[rs.randint(3), :k] = rs.randint(4)
        obs, rew, done, info = env.step(a)
        out = o.atk_step(a, difficulty, False)
        check_step(tag, env, o, obs, rew, done, out, out.reward, step)
        assert np.array_equal(info["RealAction"], np.ctypeslib.as_array(out.real_atk)), (tag, step)
        assert list(info["FailCode"]) == list(out.fail_atk[:out.n_fail_atk]), (tag, step)
        assert info["AllowNextMove"] == bool(out.allow_next_atk)
        assert info["Win"] == (None if out.win < 0 else bool(out.win))
        if _episode_over(done, left):
            break
    return step


def run_multi(L, seed, rs, max_steps=1200, multi=False, past_done=0):
    seed, env = RH.first_valid_seed("2p", L, seed)
    o = oracle_from_ref_env(env, current_oracle_config())
    tag = "2p L=%d seed=%d multi=%s" % (L, seed, multi)
    left = [past_done, False]
    for step in range(1, max_steps + 1):
        atk = np.full((3, 8), 4, dtype=np.int64)
        if rs.randint(3) == 0:
            atk = rs.randint(0, 5, size=(3, 8)).astype(np.int64)
        elif rs.randint(2) == 0:
            atk[rs.randint(3), :rs.randint(1, 9)] = rs.randint(4)
        if multi:
            d = RH.sparse_multi_action(env._board, rs, p=0.02)
            obs, rew, done, info = RH.multi_step_multi(env, {"Attacker": atk, "Defender": d})
            out, real = o.multi_step_multi(atk, d)
            assert np.array_equal(info["RealAction"]["Defender"], real), tag
            assert np.array_equal(info["RealAction"]["Attacker"], np.ctypeslib.as_array(out.real_atk)), tag
        else:
            d = RH.smart_defender_action(env._board, rs)
            obs, rew, done, info = env.step({"Attacker": atk, "Defender": d})
            out = o.multi_step(atk, d)
            ra = info["RealAction"]
            if isinstance(ra, dict):
                assert not out.real_is_def_only, (tag, step)
                assert ra["Defender"] == out.real_def and np.array_equal(
                    ra["Attacker"], np.ctypeslib.as_array(out.real_atk)), (tag, step)
            else:
                assert out.real_is_def_only and ra == out.real_def, (tag, step)
            assert list(info["FailCode"]["Attacker"]) == list(out.fail_atk[:out.n_fail_atk]), (tag, step)
            assert info["FailCode"]["Defender"] == out.fail_def, (tag, step)
        check_step(tag, env, o, obs, rew, done, out, out.reward, step)
        assert info["AllowNextMove"] == {"Attacker": bool(out.allow_next_atk),
                                         "Defender": bool(out.allow_next_def)}
        if done:
            assert info["Win"] == {"Defender": bool(out.win), "Attacker": bool(out.win_attacker)}
        if _episode_over(done, left):
            break
    return step


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--episodes", type=int, default=3)
    args = ap.parse_args(argv)
    ref_loader.load()
    rs = np.random.RandomState(12345)
    total = 0
    for ep in range(args.episodes):
        for L in (10, 20, 30):
            s = 1000 * ep + L
            total += run_def(L, s, rs, 1, True)
            total += run_def(L, s + 1, rs, 0, True)
            total += run_def(L, s + 2, rs, 1, False)
            total += run_def(L, s + 3, rs, 0, False)
            total += run_atk(L, s + 4, rs, 1)
            total += run_atk(L, s + 5, rs, 0)
            total += run_atk(L, s + 6, rs, 2)
            total += run_multi(L, s + 7, rs)
            RH.set_multiple_actions(True)
            try:
                total += run_def(L, s + 8, rs, 1, True, multi=True)
                total += run_multi(L, s + 9, rs, multi=True)
            finally:
                RH.set_multiple_actions(False)
            with RH.ref_config_override(base_LP=None, defender_action_interval=3, attacker_action_interval=2):
                total += run_def(L, s + 10, rs, 1, True)
                total += run_atk(L, s + 11, rs, 1)
                total += run_multi(L, s + 12, rs)
            with RH.ref_config_override(defender_init_cost=60, attacker_init_cost=50, defender_cost_rate=.7):
                total += run_def(L, s + 13, rs, 1, True)
                total += run_multi(L, s + 14, rs)
        print("episode set %d ok, %d steps compared so far" % (ep, total), flush=True)
    print("oracle == reference on %d env steps" % total)
    return 0


if __name__ == "__main__":
    sys.exit(main())
