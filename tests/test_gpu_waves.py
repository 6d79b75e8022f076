"""GPU: the ring-family step kernels against the C oracle past their first wave of CTAs.

k_step_tile, k_step_dense and k_step_rows are persistent grid-stride loops over at most n_sm x occupancy CTAs, so a CTA
steps a second env (or tile group) only when the batch holds more work than one wave.  The small-N parity tests never
get there.  Here every case is sized from the device's own plan to more than three full waves and a ragged fourth whose
last tile group is partial, and every env is compared with the oracle: rewards, dones, num_snakes, rewards_all and
Monitor r / l every step, the observations of the envs around each wave boundary every step and of the whole shard
every 10th, the full state and the statistics at the end.  Half way through, long bodies are loaded into both sides;
in one rule-set per kernel a short max_steps makes time-limit resets land in every wave.

A failure names the env and its place in the launch: CTA blockIdx.x and loop iteration (0 = first wave)."""
import math

import numpy as np
import pytest

import c_oracle
import helpers

pytestmark = pytest.mark.gpu

RULES = ("classic", "adversarial", "cut")
STEPS, LOAD_AT, FULL_EVERY = 160, 80, 10
SEED, ENV_ID_BASE, ACTION_SEED = 41, 7000, 13


def _case_table():
    """name -> (constructor kwargs incl. obs_mode, launch_info()["kernel"], ["block"], ["kind"]).  No force_kernel:
    every case reaches its kernel through the planner (snk_api.cu), and a different plan fails the case."""
    c = {}
    short = {("tile256", "adversarial"), ("tile512", "cut"), ("dense", "classic"), ("rows", "adversarial"), ("rowsgrid", "cut")}
    for r in RULES:
        ms = lambda k: dict(max_steps=40) if (k, r) in short else {}
        # E = V*V*3K = 2940 bytes, G = 4: eight warps of 32 threads
        c["tile256_%s_5x12" % r] = (dict(size=12, n_snakes=5, rules=r, **ms("tile256")), "k_step_tile", 256, 1)
        # E = 2025 is odd, so G = 16 envs share a 16-byte period: sixteen warps; 32 * E does not fit the lane path
        c["tile512_%s_3x13" % r] = (dict(size=13, n_snakes=3, rules=r, **ms("tile512")), "k_step_tile", 512, 1)
        # E = 3969: 32 * E is over the tile kernel's 110 KB and not a multiple of 16 for the rows kernel
        c["dense_%s_3x19" % r] = (dict(size=19, n_snakes=3, n_views=3, rules=r, **ms("dense")), "k_step_dense", 256, 2)
        # 16 views of 26x26 (32 448 bytes per env), chunks of R = 6 rows
        c["rows_%s_16x24" % r] = (dict(size=24, n_snakes=16, rules=r, **ms("rows")), "k_step_rows", 128, 3)
        c["rowsgrid_%s_5x12" % r] = (dict(size=12, n_snakes=5, rules=r, obs_mode="grid", **ms("rowsgrid")), "k_step_rows (grid)", 128, 3)
    c["tile512_classic_1x23"] = (dict(size=23, n_snakes=1, rules="classic"), "k_step_tile", 512, 1)  # E = 1875
    c["rowsgrid_cut_16x24"] = (dict(size=24, n_snakes=16, rules="cut", obs_mode="grid"), "k_step_rows (grid)", 128, 3)
    # the tile kernel into the native buffer, then k_upscale84<0, 0> (C = 15) with several envs per CTA
    c["atari84_tile_classic_5x10"] = (dict(size=10, n_snakes=5, rules="classic", obs_mode="atari84"), "k_step_tile", 256, 1)
    return c


CASES = _case_table()

# every ring-family kernel instantiation: (launch_info()["kernel"], rules, block)
INSTANTIATIONS = {
    ("k_step_tile", "classic", 256), ("k_step_tile", "adversarial", 256), ("k_step_tile", "cut", 256),
    ("k_step_tile", "classic", 512), ("k_step_tile", "adversarial", 512), ("k_step_tile", "cut", 512),
    ("k_step_dense", "classic", 256), ("k_step_dense", "adversarial", 256), ("k_step_dense", "cut", 256),
    ("k_step_rows", "classic", 128), ("k_step_rows", "adversarial", 128), ("k_step_rows", "cut", 128),
    ("k_step_rows (grid)", "classic", 128), ("k_step_rows (grid)", "adversarial", 128), ("k_step_rows (grid)", "cut", 128),
}


@pytest.fixture(scope="module")
def sb():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import snakes_b200
    return snakes_b200


def _check_plan(name, info):
    _, kernel, block, kind = CASES[name]
    got = (info["kernel"], info["block"], info["kind"])
    assert got == (kernel, block, kind), "%s: planned %s, expected %s (%s)" % (name, got, (kernel, block, kind), info)


def _probe(sb, name):
    """launch_info() of a small handle of the case.  The ring family's plan depends on N only through `grid`."""
    kw = CASES[name][0]
    env = sb.SnakeVecEnv(64, seed=SEED, **kw)
    info = env.launch_info()
    env.close()
    _check_plan(name, info)
    return info


class Layout(object):
    """Where env e sits in the launch: work item e // epc, CTA item % grid, loop iteration item // grid."""

    def __init__(self, N, info, n_sm):
        self.N, self.info = N, info
        self.epc, self.grid = info["envs_per_cta"], info["grid"]
        self.wave = n_sm * info["occupancy"] * self.epc

    def where(self, e):
        item = e // self.epc
        return "env %d (CTA %d, iteration %d)" % (e, item % self.grid, item // self.grid)

    def boundary_ranges(self):
        """The envs straddling each wave boundary, the first and the last 2 * epc envs, as disjoint [lo, hi)."""
        epc, N = self.epc, self.N
        rs = [(0, 2 * epc), (N - 2 * epc, N)] + [(k * self.wave - epc, k * self.wave + epc) for k in (1, 2, 3)]
        rs = sorted((max(0, lo), min(N, hi)) for lo, hi in rs)
        out = [list(rs[0])]
        for lo, hi in rs[1:]:
            if lo <= out[-1][1]:
                out[-1][1] = max(out[-1][1], hi)
            else:
                out.append([lo, hi])
        return [tuple(r) for r in out]


def _size(sb, name):
    """N = 3 waves + half a wave + (epc // 2 + 1): three full waves, a ragged fourth, and a partial last tile group."""
    import torch
    info = _probe(sb, name)
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    epc = info["envs_per_cta"]
    wave = n_sm * info["occupancy"] * epc
    return (3 * wave + wave // 2) // epc * epc + epc // 2 + 1, info, n_sm


def _first_bad(got, want):
    bad = np.flatnonzero((np.asarray(got) != np.asarray(want)).reshape(len(want), -1).any(1))
    return int(bad[0]) if len(bad) else None


def _check_scalars(env, lay, cres, ctx):
    _, crew, cdone, cinfo = cres
    for what, dev, cpu in (("reward", env.rewards, crew), ("done", env._done_u8, cdone.astype(np.uint8)),
                           ("num_snakes", env.num_alive, cinfo["num_snakes"]), ("rewards_all", env.rewards_all, cinfo["rewards_all"]),
                           ("Monitor r", env.episode_return, cinfo["episode_r"]), ("Monitor l", env.episode_len, cinfo["episode_l"])):
        e = _first_bad(dev.cpu().numpy(), cpu)
        if e is not None:
            raise AssertionError("%s: %s differs first in %s" % (ctx, what, lay.where(e)))


def _check_obs(sb, env, co, lay, lo, hi, ctx):
    """Observations of envs [lo, hi) against the oracle's native images, compared on the device: a grid env's cell codes
    expanded to all K views, an atari84 env's image against the native one repeated 84 / V times along both axes."""
    import torch
    want = torch.from_numpy(co.obs[lo:hi]).to(env.device)
    if env.obs_mode == "grid":
        got = sb.expand_views(env.obs[lo:hi], env.K)
    elif env.obs_mode == "atari84":
        r = 84 // env.V
        want = want.repeat_interleave(r, dim=1).repeat_interleave(r, dim=2)
        got = env.obs[lo:hi]
    else:
        got = env.obs[lo:hi]
    if not torch.equal(got, want):
        bad = (got != want).reshape(hi - lo, -1).any(1).nonzero().flatten()
        raise AssertionError("%s: obs differs in %d of envs [%d, %d), first in %s" % (ctx, len(bad), lo, hi, lay.where(lo + int(bad[0]))))


def _check_all_obs(sb, env, co, lay, ctx):
    per_env = (84 * 84 if env.obs_mode == "atari84" else env.V * env.V) * 3 * env.K
    chunk = max(1, (256 << 20) // per_env)
    for lo in range(0, env.N, chunk):
        _check_obs(sb, env, co, lay, lo, min(env.N, lo + chunk), ctx)


@pytest.mark.parametrize("name", sorted(CASES))
def test_ring_kernel_waves_match_oracle(sb, name):
    import torch
    N, probe, n_sm = _size(sb, name)
    kw = dict(CASES[name][0])
    obs_mode = kw.pop("obs_mode", "native")
    kw.update(seed=SEED, env_id_base=ENV_ID_BASE)
    env = sb.SnakeVecEnv(N, obs_mode=obs_mode, **kw)
    info = env.launch_info()
    _check_plan(name, info)
    lay = Layout(N, info, n_sm)
    epc = lay.epc
    assert (info["occupancy"], epc) == (probe["occupancy"], probe["envs_per_cta"]), (probe, info)
    assert info["grid"] == n_sm * info["occupancy"], info
    assert math.ceil(N / epc) > 3 * info["grid"], (N, info)          # three full waves ...
    assert math.ceil(N / epc) % info["grid"] != 0, (N, info)         # ... and a ragged last one
    assert epc == 1 or N % epc == epc // 2 + 1, (N, epc)             # whose last tile group is partial
    print("\n%s: N=%d  %s  grid=%d occupancy=%d envs_per_cta=%d wave=%d envs -> %.3f waves"
          % (name, N, info["kernel"], info["grid"], info["occupancy"], epc, lay.wave, N / lay.wave))

    co = c_oracle.COracle(N, **kw)
    env.reset()
    co.reset()
    _check_all_obs(sb, env, co, lay, "%s reset" % name)
    ranges = lay.boundary_ranges()
    nact = env.action_space.n
    for t in range(STEPS):
        if t == LOAD_AT:
            # long bodies in every env, re-encoded by a masked reset of nothing
            blob = helpers.tiled_long_snake_states(co.lay, co.cfg, np.random.RandomState(5))
            co.load_state(blob)
            env.load_state_blob(blob)
            env.reset(mask=torch.zeros(N, dtype=torch.bool, device=env.device))
            co.observe()
            _check_all_obs(sb, env, co, lay, "%s after load" % name)
        a = c_oracle.gen_actions(co.cfg, t, ACTION_SEED, nact)
        env.step(torch.from_numpy(a).to(env.device))
        cres = co.step(a)
        ctx = "%s step %d" % (name, t)
        _check_scalars(env, lay, cres, ctx)
        if t % FULL_EVERY == FULL_EVERY - 1 or t == STEPS - 1:
            _check_all_obs(sb, env, co, lay, ctx)
        else:
            for lo, hi in ranges:
                _check_obs(sb, env, co, lay, lo, hi, ctx)
    dev, cpu = env.dump_state(), co.state()
    for k in cpu:
        e = _first_bad(dev[k], cpu[k])
        assert e is None, "%s: state field %r differs first in %s" % (name, k, lay.where(e))
    stats, cstats = env.stats(reduce=False), dict(zip(sb._lib.STAT_NAMES, co.stats()))
    for k in sb._lib.STAT_NAMES:
        if k == "return_sum":
            assert np.allclose(stats[k], cstats[k]), (name, k, stats[k], cstats[k])
        else:
            assert stats[k] == cstats[k], (name, k, stats[k], cstats[k])
    assert stats["env_steps"] == float(N) * STEPS
    env.check_errors()
    assert co.errors() == 0
    env.close()


def test_cases_cover_every_ring_kernel(sb):
    """The case table reaches all 15 ring-family instantiations: tile at 256 and 512 threads, dense, rows and the rows
    kernel's grid form, each for the three rule-sets."""
    seen = set()
    for name in sorted(CASES):
        info = _probe(sb, name)
        seen.add((info["kernel"], CASES[name][0]["rules"], info["block"]))
    assert seen == INSTANTIATIONS, (sorted(INSTANTIATIONS - seen), sorted(seen - INSTANTIATIONS))
