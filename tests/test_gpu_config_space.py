"""GPU parity across the config space the engine accepts, past the end of an episode and at the list capacities.

Every run compares the CUDA engine with the CPU oracle bit for bit after every step (outputs, observation, env
record) and checks the episode statistics at the end (tests/parity_util.py).  Each row keeps stepping its envs
after `done` without a reset, as the reference allows (TDBoard has no done latch).
"""
import random

import numpy as np
import pytest

from tests import parity_util as PU

pytestmark = pytest.mark.gpu

INF_INTERVAL = 0x7fff          # the largest action interval the engine accepts
T4 = lambda a, b=None: [[a, a if b is None else b]] * 4          # noqa: E731 -- one value for every (type, lv)

# name -> (kind, L, run options, config overrides).  Rows use short episodes (max_episode_steps 40 unless the row is
# about it) so that most of the run happens after `done`.
CORNERS = {
    # diamond_add_cells with D = 0 (one cell) and D = 8 (a diamond wider than the 10x10 board)
    "tower_distance_0": ("def", 10, {}, dict(tower_distance=0)),
    "tower_distance_8": ("2p", 10, {}, dict(tower_distance=8)),
    # Frozen towers hit but slow nothing / freeze for the whole run (slowdown is a u8 in the record)
    "frozen_time_0": ("atk", 10, dict(difficulty=2), dict(frozen_time=0, tower_cost=T4(3))),
    "frozen_time_255": ("atk", 20, dict(difficulty=2), dict(frozen_time=255, tower_cost=T4(3))),
    # margin += speed * frozen_ratio: no movement at 0, more than the free speed above 1
    "frozen_ratio_0": ("atk", 10, dict(difficulty=2), dict(frozen_ratio=0.0, frozen_time=5, tower_cost=T4(3))),
    "frozen_ratio_2.5": ("atk", 10, dict(difficulty=2), dict(frozen_ratio=2.5, frozen_time=5, tower_cost=T4(3))),
    # cooldowns: every step, and longer than the episode (the first action is the only one)
    "intervals_0": ("2p", 10, {}, dict(attacker_action_interval=0, defender_action_interval=0)),
    "intervals_longer_than_episode": ("def", 10, {}, dict(attacker_action_interval=INF_INTERVAL,
                                                          defender_action_interval=100)),
    # base_LP: none (plane 5 = 1, only max_episode_steps ends), 0 (done on the first step), 1, the largest
    "base_LP_None": ("atk", 10, {}, dict(base_LP=None, enemy_speed=T4(0.5))),
    "base_LP_0": ("def", 10, {}, dict(base_LP=0)),
    "base_LP_1": ("atk", 10, dict(difficulty=0), dict(base_LP=1, enemy_speed=T4(0.5))),
    "base_LP_32767": ("2p", 20, {}, dict(base_LP=32767)),
    # episodes of 1 / 2 / 7 steps with auto-reset: the restart path runs on almost every step
    "max_steps_1_auto_reset": ("def", 10, dict(auto_reset=True, past_done=0), dict(max_episode_steps=1)),
    "max_steps_2_auto_reset": ("atk", 10, dict(auto_reset=True, past_done=0), dict(max_episode_steps=2)),
    "max_steps_7_auto_reset": ("2p", 10, dict(auto_reset=True, past_done=0, multi=True), dict(max_episode_steps=7)),
    "max_steps_1_past_done": ("def", 20, {}, dict(max_episode_steps=1)),
    # targeting: range 0 (same cell only) and splash 0; range and splash wider than the board
    "range_0_splash_0": ("2p", 10, {}, dict(tower_range=T4(0), tower_splash_range=T4(0), tower_cost=T4(4))),
    "range_2L_splash_L": ("def", 20, {}, dict(tower_range=T4(40), tower_splash_range=T4(20))),
    # several cells a step, leaking in the middle of the walk; speeds whose f64 sums miss 1.0
    "speeds_ge_1": ("atk", 10, {}, dict(enemy_speed=[[1, 1.5], [2, 2], [3.25, 3.25], [1, 7]], base_LP=None)),
    "speeds_inexact": ("def", 10, {}, dict(enemy_speed=[[.1, .1], [.2, .2], [1 / 3, 1 / 3], [.3, .7]])),
    # damage: defense above attack (the 5 % floor) and zero attack (hits that never kill)
    "defense_above_attack": ("2p", 10, {}, dict(enemy_defense=T4(5000), tower_cost=T4(4))),
    "attack_0": ("def", 20, {}, dict(tower_attack=T4(0))),
    # destruct refund (TDBoard.py:273-293 with the lvup argument swap) at 0, 1 and above 1, clamped by max_cost
    "destruct_return_0": ("def", 10, dict(multi=True, multi_mode="uniform", overflow="expect"), dict(tower_destruct_return=0.0)),
    "destruct_return_1": ("2p", 10, {}, dict(tower_destruct_return=1.0, tower_cost=T4(6))),
    # (1.5 pays more than the tower cost: a uniform multi-action sample would fill the tower list within a few
    # steps, so this row uses the Discrete defender, one operation a step, and lives mostly after `done`)
    "destruct_return_1.5": ("def", 20, dict(overflow="expect"), dict(tower_destruct_return=1.5)),
    # economy clamps: purses above max_cost from the start; max_cost below the cheapest tower (no build ever)
    "init_costs_above_max": ("atk", 10, {}, dict(defender_init_cost=500, attacker_init_cost=400)),
    "max_cost_below_cheapest_tower": ("def", 10, {}, dict(max_cost=8)),
    # summon level: from the first step, exactly at max_episode_steps, and only after done (step 1.5 * max)
    "upgrade_at_0": ("atk", 10, {}, dict(enemy_upgrade_at=0.0)),
    "upgrade_at_1": ("def", 10, dict(difficulty=0), dict(enemy_upgrade_at=1.0, max_episode_steps=20)),
    "upgrade_at_1.5": ("def", 10, {}, dict(enemy_upgrade_at=1.5, max_episode_steps=20)),
    "upgrade_at_1.5_atk": ("atk", 20, {}, dict(enemy_upgrade_at=1.5, max_episode_steps=20)),
    # attacker income falling over the episode (progress < 0.5 blends init and final rates)
    "cost_rate_init_above_final": ("atk", 20, {}, dict(attacker_cost_init_rate=3.0, attacker_cost_final_rate=.25)),
    # rewards that are not dyadic fractions, a negative time reward
    "rewards_non_dyadic": ("def", 10, dict(opponent="stream"), dict(reward_kill=0.1, penalty_leak=1 / 3,
                                                                     reward_time=-1 / 3)),
    # free towers / enemies: the lists run into the capacities (checked in overflow="expect" mode).  Enemies cost
    # 1e-9: a level-0 enemy cost of 0 divides by zero in planes 41-44 and is rejected like the reference rejects it
    "free_towers": ("2p", 10, dict(overflow="expect"), dict(tower_cost=T4(0), tower_distance=0, base_LP=None)),
    # 32 towers held while builds keep failing for cost / position: no flag until a 33rd build would succeed
    "towers_at_capacity_cost_bound": ("2p", 10, dict(overflow="expect", steps=400, past_done=0), dict(
        tower_cost=T4(1), tower_distance=0, defender_init_cost=32, defender_cost_rate=0.03, base_LP=None,
        max_episode_steps=400)),
    "nearly_free_enemies_L10": ("atk", 10, dict(overflow="expect"), dict(enemy_cost=T4(1e-9), enemy_speed=T4(.02),
                                                                         base_LP=None)),
    "nearly_free_enemies_L20": ("def", 20, dict(overflow="expect"), dict(enemy_cost=T4(1e-9), enemy_speed=T4(.02),
                                                                         base_LP=None)),
    # the run-time-size kernel (board size not specialised) with a handful of corners at once
    "runtime_size_L13": ("2p", 13, dict(multi=True), dict(tower_distance=0, frozen_time=255, enemy_upgrade_at=1.5,
                                                            max_episode_steps=20)),
    # the specialised (scripted level-1 opponent on the device generator) and the generic def kernel, same corner
    "generic_kernel_upgrade_at_1.5": ("def", 10, dict(generic_kernels=True), dict(enemy_upgrade_at=1.5,
                                                                                  max_episode_steps=20)),
    # the in-place observation update past done and with the summon level changing after done
    "incremental_upgrade_at_1.5": ("atk", 20, dict(incremental=True), dict(enemy_upgrade_at=1.5, max_episode_steps=20)),
    "incremental_def_multi": ("def", 20, dict(incremental=True, multi=True), dict(tower_distance=1)),
}

OPTS = dict(n_envs=16, steps=200, past_done=150)


def _run(kind, L, opts, ov, seed):
    o = dict(OPTS, **opts)
    o.setdefault("opponent", "none" if kind == "2p" else "device")
    ov = dict(ov)
    ov.setdefault("max_episode_steps", 40)
    if o.get("auto_reset"):
        o["steps"] = 60
    return PU.run_parity(kind, L, o.pop("n_envs"), o.pop("steps"), seed=seed, cfg_overrides=ov, **o)


@pytest.mark.parametrize("name", sorted(CORNERS))
def test_corner_config(name):
    kind, L, opts, ov = CORNERS[name]
    n = _run(kind, L, opts, ov, seed=sum(map(ord, name)))
    assert n > 50
    if name == "towers_at_capacity_cost_bound":
        assert PU.LAST_MAX["towers"] == 32, PU.LAST_MAX          # envs held at capacity and compared there
    elif name.startswith(("free_", "nearly_free_")):
        assert PU.LAST_RUN["overflows"] > 0, "the row is meant to reach the capacity"
    elif opts.get("overflow") == "expect":
        assert PU.LAST_RUN["post_done_steps"] > 100, PU.LAST_RUN
    elif opts.get("auto_reset"):
        assert PU.LAST_RUN["episodes"] > 8
    else:
        assert PU.LAST_RUN["post_done_steps"] > 100, PU.LAST_RUN


def random_config(rs, L):
    """A config from the region validate_config accepts (f64 tables drawn from ranges where play stays varied)."""
    def table(lo, hi):
        return rs.uniform(lo, hi, size=(4, 2)).tolist()

    def itable(hi):
        return rs.randint(0, hi + 1, size=(4, 2)).tolist()

    return dict(
        enemy_LP=table(1, 6000), enemy_speed=table(0, 2.5), enemy_defense=table(0, 800), enemy_cost=table(0.5, 40),
        tower_attack=table(0, 900), tower_cost=table(0.5, 30), tower_attack_interval=table(0, 8),
        tower_range=itable(2 * L), tower_splash_range=itable(L),
        tower_destruct_return=rs.uniform(0, 2), frozen_ratio=rs.uniform(0, 2), frozen_time=int(rs.randint(0, 256)),
        attacker_init_cost=rs.uniform(0, 150), defender_init_cost=rs.uniform(0, 150), max_cost=rs.uniform(1, 150),
        reward_kill=rs.uniform(-1, 1), penalty_leak=rs.uniform(-20, 20), reward_time=rs.uniform(-.1, .1),
        attacker_cost_init_rate=rs.uniform(0, 3), attacker_cost_final_rate=rs.uniform(0, 3),
        defender_cost_rate=rs.uniform(0, 3), enemy_upgrade_at=rs.uniform(-.5, 2.5),
        base_LP=None if rs.randint(4) == 0 else int(rs.randint(0, 12)), tower_distance=int(rs.randint(0, 9)),
        attacker_action_interval=int(rs.choice([0, 1, 2, 3, 7, 1000])),
        defender_action_interval=int(rs.choice([0, 1, 2, 3, 7, 1000])),
        max_episode_steps=int(rs.randint(1, 90)))


RANDOM_LEGS = [("def", 10, dict(difficulty=1)), ("atk", 10, dict(difficulty=2)), ("2p", 20, {}),
               ("def", 20, dict(multi=True, difficulty=0)), ("atk", 20, dict(difficulty=0)),
               ("def", 10, dict(opponent="stream")), ("2p", 10, dict(multi=True)), ("def", 13, dict(difficulty=1))]


@pytest.mark.parametrize("seed", range(8))
def test_random_config(seed):
    """Seeded configs: a failure names its seed, and random_config(np.random.RandomState(seed), L) rebuilds it."""
    kind, L, opts = RANDOM_LEGS[seed % len(RANDOM_LEGS)]
    ov = random_config(np.random.RandomState(1000 + seed), L)
    assert _run(kind, L, dict(opts, overflow="expect"), ov, seed=seed) > 50


@pytest.mark.parametrize("kind", ["def", "atk", "2p"])
def test_stats_count_each_episode_once_without_auto_reset(kind):
    """auto_reset off, every env stepped long after its episode ended: td_get_stats holds each episode once, with
    the return, length, win, kills and leaks of the steps up to and including the one that ended it."""
    n = PU.run_parity(kind, 10, 16, 200, seed=7, opponent="none" if kind == "2p" else "device",
                      cfg_overrides=dict(max_episode_steps=30, base_LP=2), past_done=150)
    assert n > 16 * 30 and PU.LAST_RUN["episodes"] == 16 and PU.LAST_RUN["post_done_steps"] > 16 * 100


FACADE = {"def": "TD-def-small-v0", "atk": "TD-atk-small-v0", "2p": "TD-2p-middle-v0"}


@pytest.mark.parametrize("kind", sorted(FACADE))
def test_facade_steps_past_done_like_the_oracle(kind):
    """G.make(...) keeps stepping a finished env (no reset) for 300 steps: observation, reward, done, Win and the
    board stay those of an oracle twin stepped the same way."""
    import gym_td_b200 as G
    from gym_td_b200 import engine as E
    old = G.hyper_parameters.__dict__["max_episode_steps"]
    G.hyper_parameters.__dict__["max_episode_steps"] = 50          # frozen like the reference's; poked the same way
    try:
        seed = 1024
        random.seed(seed)
        env = G.make(FACADE[kind], seed=seed)
        o = PU.oracle_env_from_map(env._map, PU.oracle_config_from_engine(E.config_struct()))
        assert o.cfg.max_episode_steps == 50
        assert np.array_equal(env._board.get_states().view(np.uint32), o.get_states().view(np.uint32))
        o.set_pyrand(random.getstate())
        rs = np.random.RandomState(5)
        after = 0
        ended = False
        for t in range(2000):
            if kind == "atk":
                a = PU.attacker_action(rs)
                out = o.atk_step(a, 1)
            elif kind == "def":
                a = PU.smart_defender_action(o, rs)
                out = o.def_step(a, 1)
            else:
                a = {"Attacker": PU.attacker_action(rs), "Defender": PU.smart_defender_action(o, rs)}
                out = o.multi_step(a["Attacker"], a["Defender"])
            obs, r, d, info = env.step(a)
            tag = "%s step %d" % (kind, t + 1)
            assert np.array_equal(obs.view(np.uint32), o.get_states().view(np.uint32)), tag
            assert float(r).hex() == float(out.reward).hex() and d == bool(out.done), tag
            win = info["Win"]["Defender"] if isinstance(info["Win"], dict) else info["Win"]
            assert win == (None if out.win < 0 else bool(out.win)), tag
            ended = ended or d
            if ended:
                after += 1
                if after > 300:
                    break
        assert after > 300
        env.close()
    finally:
        G.hyper_parameters.__dict__["max_episode_steps"] = old
