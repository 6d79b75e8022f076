"""Step time of obs_mode 'grid' against the native RGB observation, shape by shape, and the expander on its own.

    python tools/grid_probe.py [--rounds R] [--out FILE]

Native and grid handles of each shape are alternated in one process, `rounds` times; every timing is CUDA events around
one launch of a graph of T steps (uniform Philox actions, 16 batches resident in HBM, or the fruit-seeking policy kernel),
after one untimed launch of the same graph.  Rows report the mean and the spread over the rounds.  Observation bytes are
what a step writes (N*V*V*3K native, N*V*V grid); the expander row compares against the 6.2 TB/s a write stream sustains on
a B200 (DESIGN.md section 4.11).  The split of a grid step into k_lane_logic and k_lane_grid comes from a separate
torch.profiler run.  The card's name and power limit are printed with the numbers.  Needs a GPU; writes nothing but --out."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FLOOR_BPS = 6.2e12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:  # noqa: BLE001
        q = "power limit unknown (%s)" % exc
    return "%s, power limit / max SM clock: %s" % (name, q)


def time_launch(fn):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe needs a CUDA device"
    import snakes_b200 as sb

    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    say("%d rounds, native and grid alternated; us per step = one graph launch of T steps / T" % args.rounds)
    say("%-52s %6s %-8s %22s %10s %12s" % ("shape", "T", "obs", "us/step mean [min-max]", "MB obs/st", "kernel"))

    def shape_rows(label, N, kw, T, scripted=False, warm=0, debug_grid=None):
        envs, graphs = {}, {}
        for mode in ("native", "grid"):
            dbg = debug_grid if mode == "grid" and debug_grid else None
            env = sb.SnakeVecEnv(N, seed=0, obs_mode=mode, debug=dbg, **kw)
            env.reset()
            if scripted:
                for t in range(warm):
                    env.step(env.gen_scripted_actions(t, seed=2, eps=0.05))
                g = env.make_scripted_graph(T, step0=warm, seed=2, eps=0.05)
            else:
                acts = torch.stack([env.gen_actions(t, 1).clone() for t in range(16)])
                g = env.make_graph(acts, T)
                env._probe_acts = acts
            g.launch()  # untimed warm-up launch
            torch.cuda.synchronize()
            envs[mode], graphs[mode] = env, g
        times = {"native": [], "grid": []}
        for _ in range(args.rounds):
            for mode in ("native", "grid"):
                times[mode].append(time_launch(graphs[mode].launch) / T)
        for mode in ("native", "grid"):
            env, ts = envs[mode], times[mode]
            obs_mb = env.obs.numel() / 1e6
            say("%-52s %6d %-8s %8.2f [%6.2f-%6.2f] %10.1f %12s" % (label, T, mode, np.mean(ts), min(ts), max(ts), obs_mb,
                                                                      env.launch_info()["kernel"].replace(" ", "")))
        if scripted:
            st = envs["grid"].stats()
            say("%-52s mean body cells per env over the run: %.1f" % ("", st["body_cells"] / max(st["env_steps"], 1)))
        for mode in ("native", "grid"):
            graphs[mode].close()
            envs[mode].close()
        torch.cuda.synchronize()
        return np.mean(times["native"]), np.mean(times["grid"])

    head = dict(size=19, n_snakes=2, rules="classic")
    shape_rows("headline: 131072 x 2 snakes 19x19 classic, random", 131072, head, 2000)
    shape_rows("configs[1]: 4096 x 2 snakes 10x10 classic", 4096, dict(size=10, n_snakes=2, rules="classic"), 2000)
    shape_rows("configs[2]: 65536 x 3 snakes 10x10 cut", 65536, dict(size=10, n_snakes=3, rules="cut"), 2000)
    shape_rows("headline shape, fruit-seeking stream (eps 0.05)", 131072, head, 500, scripted=True, warm=300)
    shape_rows("configs[4] shard: 32768 x 16 snakes 64x64 classic", 32768, dict(size=64, n_snakes=16, rules="classic"), 40)
    shape_rows("configs[4] shard: 32768 x 16 snakes 64x64 cut", 32768, dict(size=64, n_snakes=16, rules="cut"), 40)
    say("grid un-paint: walk (restore_thr=0) against the default zero-fill threshold, native rows repeated for reference")
    shape_rows("headline, random, grid restore_thr=0", 131072, head, 2000, debug_grid="restore_thr=0")
    shape_rows("headline, fruit-seeking, grid restore_thr=0", 131072, head, 500, scripted=True, warm=300, debug_grid="restore_thr=0")

    # the expander alone: grid [N,21,21] -> [N,21,21,3n]
    say("")
    say("expand_views at the headline shape (131072 x 21 x 21 cells), 200 calls per row, mean per call")
    say("%-40s %10s %12s %9s %10s %7s" % ("call", "us/call", "bytes", "GB/s", "floor us", "x floor"))
    grd = sb.SnakeVecEnv(131072, seed=0, obs_mode="grid", **head)
    grd.reset()
    for t in range(64):
        grd.step(grd.gen_actions(t, 1))
    for nv, first in ((2, 0), (1, 0), (1, 1), (3, 0), (16, 0)):
        out = torch.empty(tuple(grd.obs.shape) + (3 * nv,), dtype=torch.uint8, device=grd.device)
        sb.expand_views(grd.obs, nv, first_view=first, out=out)
        torch.cuda.synchronize()
        us = time_launch(lambda: [sb.expand_views(grd.obs, nv, first_view=first, out=out) for _ in range(200)]) / 200
        nbytes = out.numel() + grd.obs.numel()
        floor = out.numel() / FLOOR_BPS * 1e6
        say("%-40s %10.2f %12d %9.0f %10.2f %7.2f" % ("n_views=%d first_view=%d" % (nv, first), us, nbytes, nbytes / us / 1e3, floor, us / floor))
        del out

    # host_io: steps per second through pinned host buffers (H2D actions, step, D2H results, synchronise)
    say("")
    say("host_io steps at the headline shape: numpy actions in, numpy obs / rewards / dones out, 20 steps per round")
    host = {}
    for mode in ("native", "grid"):
        host[mode] = sb.SnakeVecEnv(131072, seed=0, obs_mode=mode, host_io=True, **head)
        host[mode].reset()
    acts = np.random.RandomState(0).randint(0, 5, size=(131072, 2)).astype(np.int8)
    rates = {"native": [], "grid": []}
    for _ in range(args.rounds):
        for mode in ("native", "grid"):
            host[mode].step(acts)
            t0 = time.perf_counter()
            for _ in range(20):
                host[mode].step(acts)
            rates[mode].append(20 / (time.perf_counter() - t0))
    for mode in ("native", "grid"):
        r = rates[mode]
        say("%-10s %8.1f steps/s [%6.1f-%6.1f]  %8.1f MB D2H per step" % (mode, np.mean(r), min(r), max(r), host[mode].obs.numel() / 1e6))
        host[mode].close()

    # split of a grid step into its two kernels (separate profiler run, eager steps)
    say("")
    from torch.profiler import ProfilerActivity, profile
    for label, scripted in (("random actions", False), ("fruit-seeking, after 300 steps", True)):
        if scripted:
            for t in range(300):
                grd.step(grd.gen_scripted_actions(t, seed=2, eps=0.05))
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for t in range(50):
                a = grd.gen_scripted_actions(300 + t, seed=2, eps=0.05) if scripted else grd.gen_actions(64 + t, 1)
                grd.step(a)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            for k in ("k_lane_logic", "k_lane_grid", "k_scripted_actions", "k_gen_actions"):
                if k in ev.key:
                    per[k] = per.get(k, 0.0) + ev.device_time_total / max(ev.count, 1)
        say("grid step split (%s, torch.profiler, mean kernel time): %s" % (label, ", ".join("%s %.2f us" % kv for kv in sorted(per.items()))))
    grd.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
