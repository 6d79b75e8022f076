"""A/B timing of one library build (SNK_LIB=variants/libsnk_X.so): every shape is timed through the CUDA-graph step loop
(one launch per measurement, CUDA events), so Python is out of the numbers.

    python tools/ab.py short long c3 c2 1m atari rows      # any subset; default: short long
    extra lines: c3c (3 snakes classic 10x10), adv (adversarial 2x19x19), grid (obs_mode grid 2x19x19), roll (graph with
    per-step observation outputs, 2x19x19), e2e (eager step_scalars_async loop, 2x19x19)
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import snakes_b200

PEAK = 6548.2


def timed_graph(env, g, reps=3):
    best = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); g.launch(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def report(tag, env, us, N):
    st = env.stats(False)
    es = max(st["env_steps"], 1)
    sl = st["body_cells"] / es
    ab = env.algorithmic_bytes_per_step(sl)
    print("%-44s %8.2f us  sumL %5.1f  frac %.3f  (per env-step: %.3f fruits, %.3f draws, %.4f episodes) %s" % (
        tag, us, sl, ab * N / us / 1e3 / PEAK, st["fruits"] / es, st["draws"] / es, st["episodes"] / es, env.launch_info()["kernel"]), flush=True)


def short(N, T=400, reps=3, tag="short", **kw):
    env = snakes_b200.SnakeVecEnv(N, **kw); env.reset()
    acts = torch.stack([env.gen_actions(t, 1).clone() for t in range(16)])
    g = env.make_graph(acts, T=T)
    g.launch()
    env.reset_stats()
    us = timed_graph(env, g, reps) / T * 1e3
    report("%s N=%d %s" % (tag, N, kw), env, us, N)
    g.close(); env.close()


def roll(N, T=16, reps=3, **kw):
    """A graph that writes every step's observations into its own [T] output (rollout slots): whole images."""
    env = snakes_b200.SnakeVecEnv(N, **kw); env.reset()
    acts = torch.stack([env.gen_actions(t, 1).clone() for t in range(T)])
    obs = torch.empty((T,) + tuple(env.obs.shape), dtype=torch.uint8, device="cuda")
    g = env.make_graph(acts, T=T, obs_out=obs)
    g.launch()
    env.reset_stats()
    us = timed_graph(env, g, reps) / T * 1e3
    report("roll N=%d %s" % (N, kw), env, us, N)
    g.close(); env.close()


def e2e(N, K=320, **kw):
    """Eager steps with numpy actions in and per-env scalars out, four in flight (bench.py's e2e_obs_resident)."""
    import time
    import numpy as np
    env = snakes_b200.SnakeVecEnv(N, **kw); env.reset()
    acts = [np.random.RandomState(t).randint(0, 5, size=(N, env.S)).astype(np.int8) for t in range(8)]
    for t in range(8):
        env.wait_scalars(env.step_scalars_async(acts[t]))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    tickets = []
    for t in range(K):
        tickets.append(env.step_scalars_async(acts[t % 8]))
        if t >= 2:
            env.wait_scalars(tickets[t - 2])
    for tk in tickets[-2:]:
        env.wait_scalars(tk)
    torch.cuda.synchronize()
    us = (time.perf_counter() - t0) / K * 1e6
    report("e2e N=%d %s" % (N, kw), env, us, N)
    env.close()


def long_(N, warm=400, T=100, eps=0.05, **kw):
    """Fruit-seeking policy: policy kernel + step kernel (what bench.py's scripted_policy times), and the step kernel alone
    on the recorded actions from the same start state."""
    env = snakes_b200.SnakeVecEnv(N, **kw); env.reset()
    gw = env.make_scripted_graph(warm, 0, 7, eps); gw.launch(); gw.close()
    torch.cuda.synchronize()
    for t in range(3):  # a few eager steps: the regime-adaptive path decides from the statistics the kernels post
        env.step_async(env.gen_scripted_actions(warm + t, 7, eps)); env._pending = False
    torch.cuda.synchronize()
    warm += 3
    blob = env.dump_state_blob()
    acts = torch.empty((T, N, env.S), dtype=torch.int8, device="cuda")
    for t in range(T):
        env.gen_scripted_actions(warm + t, 7, eps, out=acts[t]); env.step_async(acts[t]); env._pending = False
    torch.cuda.synchronize()
    gs = env.make_scripted_graph(T, warm, 7, eps)
    ga = env.make_graph(acts, T=T)
    both = step = 1e9
    for _ in range(3):
        env.load_state_blob(blob); env.reset_stats()
        both = min(both, timed_graph(env, gs, 1) / T * 1e3)
    for _ in range(3):
        env.load_state_blob(blob); env.reset_stats()
        step = min(step, timed_graph(env, ga, 1) / T * 1e3)
    report("long eps=%.2f N=%d %s step only" % (eps, N, kw), env, step, N)
    print("%-44s %8.2f us  (%.3e agent-steps/s)" % ("      policy kernel + step kernel", both, N * env.S / both * 1e6), flush=True)
    gs.close(); ga.close(); env.close()


if __name__ == "__main__":
    print("lib:", os.environ.get("SNK_LIB", "default"), " SNK_DEBUG:", os.environ.get("SNK_DEBUG", ""))
    which = sys.argv[1:] or ["short", "long"]
    if "short" in which: short(131072, size=19, n_snakes=2)
    for w in which:
        if w.startswith("long"): long_(131072, eps=(int(w[4:]) / 100.0 if len(w) > 4 else 0.05), size=19, n_snakes=2)
    if "c3" in which: short(65536, tag="c3", size=10, n_snakes=3, rules="cut")
    if "c3c" in which: short(65536, tag="c3 classic", size=10, n_snakes=3, rules="classic")
    if "c2" in which: short(4096, T=1000, tag="c2", size=10, n_snakes=2)
    if "1m" in which: short(1048576, T=60, reps=1, tag="1m", size=19, n_snakes=2)
    if "atari" in which: short(131072, T=40, reps=2, tag="atari84", size=19, n_snakes=2, obs_mode="atari84")
    if "rows" in which: short(32768, T=30, reps=2, tag="rows", size=64, n_snakes=16, rules="cut")
    if "adv" in which: short(131072, tag="adv", size=19, n_snakes=2, rules="adversarial")
    if "grid" in which: short(131072, tag="grid", size=19, n_snakes=2, obs_mode="grid")
    if "roll" in which: roll(131072, size=19, n_snakes=2)
    if "e2e" in which: e2e(131072, size=19, n_snakes=2)
