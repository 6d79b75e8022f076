"""Fused kernel (lane=fused) against the two-kernel form (lane=split) on the same start state and the same actions, for the
planner's threshold between them (plan_launch / regime_update in snk_api.cu).  Every time is a CUDA-graph step loop timed
with CUDA events, the two forms alternated; the mean body cells per env (sumL) is what the running statistics report.

    python tools/crossover.py [N ...]            # default: 4096 32768 131072 1048576
    python tools/crossover.py --profile          # torch.profiler split of the headline two-kernel step (logic vs writer)
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import snakes_b200

KW = dict(size=19, n_snakes=2, rules="classic", seed=0)
REGIMES = [("random", None), ("seek70", 0.70), ("seek40", 0.40), ("seek20", 0.20), ("seek05", 0.05)]


def timed(g, reps):
    best = 1e9
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); g.launch(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def start_state(N, eps, warm):
    """The state after `warm` steps of random actions (eps None) or of the fruit-seeking policy, and the next T actions."""
    env = snakes_b200.SnakeVecEnv(N, **KW); env.reset()
    if eps is None:
        for t in range(warm):
            env.step_async(env.gen_actions(t, 1)); env._pending = False
    else:
        g = env.make_scripted_graph(warm, 0, 7, eps); g.launch(); g.close()
    torch.cuda.synchronize()
    return env


def one(N, name, eps, T, reps, warm):
    src = start_state(N, eps, warm)
    blob = src.dump_state_blob()
    acts = torch.empty((T, N, 2), dtype=torch.int8, device="cuda")
    for t in range(T):
        if eps is None: src.gen_actions(warm + t, 1, out=acts[t])
        else: src.gen_scripted_actions(warm + t, 7, eps, out=acts[t])
        src.step_async(acts[t]); src._pending = False
    torch.cuda.synchronize()
    src.close()
    envs = {f: snakes_b200.SnakeVecEnv(N, debug="lane=" + f, **KW) for f in ("fused", "split")}
    graphs = {f: e.make_graph(acts, T=T) for f, e in envs.items()}
    best = {f: 1e9 for f in envs}
    sl = 0.0
    for r in range(reps):
        for f in (("fused", "split") if r % 2 == 0 else ("split", "fused")):
            e = envs[f]
            e.load_state_blob(blob); e.step_async(acts[0]); e._pending = False  # one eager step: the frame is the state's
            e.reset_stats()
            best[f] = min(best[f], timed(graphs[f], 1) / T * 1e3)
            st = e.stats(False)
            sl = st["body_cells"] / max(st["env_steps"], 1)
    kinds = {f: e.launch_info()["kernel"] for f, e in envs.items()}
    print("N=%-8d %-7s sumL %5.1f  fused %8.2f us  split %8.2f us  split/fused %.3f   (%s | %s)" % (
        N, name, sl, best["fused"], best["split"], best["split"] / best["fused"], kinds["fused"], kinds["split"]), flush=True)
    for f in envs:
        graphs[f].close(); envs[f].check_errors(); envs[f].close()


def profile(out_dir):
    from torch.profiler import profile as prof, ProfilerActivity
    N = 131072
    for f in ("split", "fused"):
        env = snakes_b200.SnakeVecEnv(N, debug="lane=" + f, **KW); env.reset()
        acts = torch.stack([env.gen_actions(t, 1).clone() for t in range(16)])
        g = env.make_graph(acts, T=100)
        g.launch(); torch.cuda.synchronize()
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            g.launch(); torch.cuda.synchronize()
        print("---- torch.profiler, 100-step graph, 131072 envs 2x19x19, random actions, lane=%s" % f)
        print(p.key_averages().table(sort_by="cuda_time_total", row_limit=6))
        if out_dir:
            p.export_chrome_trace(os.path.join(out_dir, "crossover_%s.pt.trace.json" % f))
        g.close(); env.close()


if __name__ == "__main__":
    print(torch.cuda.get_device_name(0))
    if "--profile" in sys.argv:
        profile(os.environ.get("SNK_TRACE_DIR"))
        sys.exit(0)
    sizes = [int(a) for a in sys.argv[1:]] or [4096, 32768, 131072, 1048576]
    for N in sizes:
        T = 30 if N >= 1 << 20 else 100
        for name, eps in REGIMES:
            one(N, name, eps, T, reps=4, warm=400 if eps is not None else 100)
