"""The forms of the lane path, each against the C oracle through the C ABI: the two-kernel form
(k_lane_logic with its grouped death test, then k_lane_paint2 with two warps per image buffer), the
regime switch between the fused and the two-kernel form in mid-run, the small-shard batches of
16 / 8 / 4 envs per warp, and the two occupancy sources of the scripted policy kernel.
Reference semantics: gym_snake/envs/snake_multiple_test.py:97-232 (via oracle/snake_oracle.c)."""
import numpy as np
import pytest

import helpers
import c_oracle
from test_gpu_parity import _compare_step

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sb():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import snakes_b200
    return snakes_b200


def _scripted_run(sb, N, steps, debug, kw, seed=3, eps=0.05, state_every=40):
    """Fruit-seeking actions (long bodies, respawns every step) on the device, same actions on the oracle."""
    env = sb.SnakeVecEnv(N, debug=debug, **kw)
    co = c_oracle.COracle(N, **kw)
    assert np.array_equal(env.reset().cpu().numpy(), co.reset())
    kernels = set()
    for t in range(steps):
        a = env.gen_scripted_actions(t, seed=seed, eps=eps).cpu().numpy()
        _compare_step(env, co, a, "%s step %d" % (debug, t), check_state=(t % state_every == state_every - 1))
        kernels.add(env.launch_info()["kernel"])
    env.check_errors()
    st = env.stats(False)
    env.close()
    return st, kernels


@pytest.mark.parametrize("S,D", [(2, 19), (1, 19), (3, 10), (4, 12)])
def test_two_kernel_form_long_bodies(sb, S, D):
    """lane=split: k_lane_logic (grouped death test, 7 CTAs per SM for S <= 2) + k_lane_paint2, long bodies."""
    st, _ = _scripted_run(sb, 1000, 260, "lane=split", dict(size=D, n_snakes=S, rules="classic", seed=11))
    assert st["body_cells"] / st["env_steps"] > 2.0 * S  # the policy did grow them


@pytest.mark.parametrize("rules", ["adversarial", "cut"])
def test_two_kernel_form_other_rules(sb, rules):
    N, kw = 777, dict(size=10, n_snakes=3, rules=rules, seed=4)
    env = sb.SnakeVecEnv(N, debug="lane=split", **kw)
    co = c_oracle.COracle(N, **kw)
    assert np.array_equal(env.reset().cpu().numpy(), co.reset())
    for t in range(120):
        a = env.gen_actions(t, 9).cpu().numpy()
        _compare_step(env, co, a, "%s split step %d" % (rules, t), check_state=(t % 30 == 29))
    env.check_errors()
    env.close()


def test_regime_switch_mid_run(sb):
    """adaptive lane path: threshold lowered so that the handle goes fused -> two kernels while the bodies grow and back
    when random actions shorten them again; every step bit-exact, both plans seen."""
    import torch
    N, kw = 4736, dict(size=19, n_snakes=2, rules="classic", seed=21)
    env = sb.SnakeVecEnv(N, debug="alt_hi=6,epw=32", **kw)   # (a shard this small would shrink its batches and not switch forms)
    assert env.launch_info()["adaptive"]
    co = c_oracle.COracle(N, **kw)
    assert np.array_equal(env.reset().cpu().numpy(), co.reset())
    plans = []
    for t in range(330):
        if t < 200:
            a = env.gen_scripted_actions(t, seed=5, eps=0.05).cpu().numpy()
        else:
            a = env.gen_actions(t, 5).cpu().numpy()
        _compare_step(env, co, a, "adaptive step %d" % t, check_state=(t % 50 == 49))
        torch.cuda.synchronize()
        plans.append(env.launch_info()["kernel"])
    env.check_errors()
    env.close()
    assert len(set(plans)) == 2, "the handle never changed its form: %s" % set(plans)
    assert plans[0] == plans[-1] == "k_step_lane" and plans[190] == "k_lane_logic + k_lane_paint2", "expected fused -> two kernels -> fused"


@pytest.mark.parametrize("epw", [16, 8, 4])
def test_small_shard_batches(sb, epw):
    """epw=<n>: the fused kernel steps n envs per warp batch (idle lanes join the painting); ragged last batch."""
    N, kw = 1003, dict(size=10, n_snakes=2, rules="classic", seed=8)
    env = sb.SnakeVecEnv(N, debug="epw=%d" % epw, **kw)
    co = c_oracle.COracle(N, **kw)
    assert np.array_equal(env.reset().cpu().numpy(), co.reset())
    assert env.launch_info()["envs_per_warp_batch"] == epw
    for t in range(150):
        a = env.gen_scripted_actions(t, seed=1, eps=0.2).cpu().numpy() if t % 3 else env.gen_actions(t, 1).cpu().numpy()
        _compare_step(env, co, a, "epw=%d step %d" % (epw, t), check_state=(t % 50 == 49))
    env.check_errors()
    env.close()


def test_small_shard_default_plan(sb):
    """4 096 envs of 2x10x10 (BASELINE configs[1]) are fewer 32-env batches than the GPU holds warps: the planner shrinks
    the batch; 131 072 envs keep 32."""
    small = sb.SnakeVecEnv(4096, size=10, n_snakes=2)
    big = sb.SnakeVecEnv(131072, size=19, n_snakes=2)
    assert small.launch_info()["envs_per_warp_batch"] < 32
    assert big.launch_info()["envs_per_warp_batch"] == 32 and big.launch_info()["adaptive"]
    small.close(); big.close()


def test_scripted_policy_forms_agree(sb):
    """The policy kernel reads occupancy from the observations when they describe the current state, and walks the
    bodies otherwise (after load_state): same actions."""
    N, kw = 2048, dict(size=19, n_snakes=2, rules="classic", seed=6)
    env = sb.SnakeVecEnv(N, **kw)
    env.reset()
    for t in range(150):
        env.step(env.gen_scripted_actions(t, seed=9))
    a_obs = env.gen_scripted_actions(150, seed=9).clone()
    blob = env.dump_state_blob()
    env.load_state_blob(blob)               # the state is the same, the observations are no longer vouched for
    a_walk = env.gen_scripted_actions(150, seed=9).clone()
    assert bool((a_obs == a_walk).all())
    env.close()
