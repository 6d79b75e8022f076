"""The self-play learner on grids against the RGB learner: the first conv layer alone, then Runner.run and Model.train.

    python tools/grid_learner_probe.py [--rounds R] [--out FILE] [--arch custom|nature]

1. Input stage at n in {1 024, 32 768, 131 072} grids of V in {21, 12} (live grid envs, 2 snakes, after 30 steps):
   grid_conv_in forward (snk_grid_conv_in) and backward (snk_grid_conv_in_wgrad + the fold into dW / dbias; also the two
   kernels alone), against CnnPolicy's RGB input stage on expand_views of the same grids, view 0 (uint8 NHWC -> float,
   x 1/255, channels_last, cuDNN conv1, ReLU; backward: ReLU backward + cuDNN weight gradient) with cuDNN TF32 on and off.
   Bytes are the algorithmic ones: forward n V^2 (1 + 128), backward n V^2 (1 + 2 * 128); the forward is compared with the
   6.2 TB/s a write stream sustains on a B200 (DESIGN.md section 4.11), the backward, a read stream, with the data sheet's
   7.7 TB/s (not a measured ceiling).
2. Runner.run time per rollout step (16 steps, main model and one opponent) and Model.train time per minibatch
   (N * 16 / 4 samples, at most 32 768) for 2 snakes on 19 x 19 at N in {32, 4 096, 16 384}, native env + RGB models
   against grid env + grid models, torch defaults (cuDNN TF32 on).  And the bytes of mb_obs.
--arch nature: the same for nature_cnn on the 84 x 84 WarpFrame view: grid_conv84_in (snk_grid_conv84_in / _wgrad) against
the RGB stage on the WarpFrame of the same grids (uint8 84 x 84 -> float, channels_last, cuDNN 8x8 stride-4 conv1 + ReLU),
bytes n V^2 + n 400 * 128 forward and n V^2 + 2 n 400 * 128 backward; and the learner as obs_mode 'atari84' env + RGB
nature models against grid env + grid nature models.
Every time is CUDA events (or a host clock around work that ends in a synchronise) over repeated calls after untimed warm-up
calls of the same shapes; native and grid alternate `rounds` times, rows give the mean and the spread over the rounds.  The
card's name and power limit are printed with the numbers.  Needs a GPU; writes nothing but --out."""
import argparse
import ctypes as C
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.grid_probe import card  # noqa: E402

WRITE_BPS, DATASHEET_BPS = 6.2e12, 7.7e12


def events(fn, reps):
    """mean us per call of fn over `reps` calls, CUDA events around the whole run."""
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3 / reps


def spread(xs):
    return "%9.1f [%.1f-%.1f]" % (np.mean(xs), min(xs), max(xs))


def live_grids(sb, n, V, seed=0):
    env = sb.SnakeVecEnv(n, size=V - 2, n_snakes=2, seed=seed, obs_mode="grid")
    env.reset()
    for t in range(30):
        env.step(env.gen_actions(t, 1))
    g = env.obs.clone()
    env.close()
    return g


def input_stage(sb, say, rounds, arch="custom"):
    from snakes_b200 import _lib
    torch.manual_seed(0)
    nature = arch == "nature"
    conv = (torch.nn.Conv2d(3, 32, 8, 4) if nature else torch.nn.Conv2d(3, 32, 3, 1, 1)).cuda()
    w, b = conv.weight, conv.bias
    conv_in, wgrad = (sb.grid_conv84_in, "snk_grid_conv84_in_wgrad") if nature else (sb.grid_conv_in, "snk_grid_conv_in_wgrad")
    say("\n1. input stage (first conv + bias + ReLU), view 0; us per call, mean [min-max] over %d rounds" % rounds
        + ("; nature_cnn on the 84x84 WarpFrame" if nature else ""))
    say("%-14s %-26s %24s %24s %10s %10s" % ("shape", "path", "forward", "backward", "fwd GB/s", "bwd GB/s"))
    for V in (21, 12):
        for n in (1024, 32768, 131072):
            g = live_grids(sb, n, V)
            x = sb.expand_views(g, 1)
            if nature:   # the obs_mode 'atari84' view: every cell replicated 84 / V times
                x = x.repeat_interleave(84 // V, 1).repeat_interleave(84 // V, 2).contiguous()
            cells = n * V * V
            side = 20 if nature else V   # output rows and columns
            outs = n * side * side
            reps = max(3, min(50, int(2e10 // (outs * 128))))
            gy = torch.randn((n, side, side, 32), device="cuda").permute(0, 3, 1, 2)   # channels_last, as conv2 hands it back
            if nature:
                _, P, Cb, wbytes = _lib.grid_conv84_geometry(V, n)
                hist = torch.empty((P, P, Cb, Cb, 7, 32), device="cuda")
            else:
                wbytes = _lib.grid_conv_work_bytes(cells)
                hist = torch.empty((9, 7, 32), device="cuda")
            work = torch.empty((wbytes // 4,), device="cuda")
            L, st = _lib.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)

            def grid_fwd():
                with torch.no_grad():
                    return conv_in(g, 0, w, b)

            yg = conv_in(g, 0, w, b)
            go = gy.permute(0, 2, 3, 1)
            yo = yg.permute(0, 2, 3, 1)

            def grid_bwd():
                torch.autograd.grad(yg, (w, b), gy, retain_graph=True)

            def grid_wgrad_kernels():
                _lib.check(getattr(L, wgrad)(C.c_void_p(g.data_ptr()), n, V - 2, 0, C.c_void_p(yo.data_ptr()),
                                             C.c_void_p(go.data_ptr()), 32, C.c_void_p(hist.data_ptr()),
                                             C.c_void_p(work.data_ptr()), work.numel() * 4, 0, st))

            def rgb_out():
                xf = x.permute(0, 3, 1, 2).float() * (1.0 / 255.0)
                return F.relu(conv(xf.contiguous(memory_format=torch.channels_last)))

            def rgb_fwd():
                with torch.no_grad():
                    return rgb_out()

            res = {k: ([], []) for k in ("grid", "grid kernels", "rgb tf32", "rgb fp32")}
            for _ in range(rounds):
                for tf32 in (True, False):
                    torch.backends.cudnn.allow_tf32 = tf32
                    yr = rgb_out()
                    rgb_fwd(); torch.autograd.grad(yr, (w, b), gy, retain_graph=True)
                    key = "rgb tf32" if tf32 else "rgb fp32"
                    res[key][0].append(events(rgb_fwd, reps))
                    res[key][1].append(events(lambda: torch.autograd.grad(yr, (w, b), gy, retain_graph=True), reps))
                    del yr
                grid_fwd(); grid_bwd(); grid_wgrad_kernels()
                res["grid"][0].append(events(grid_fwd, reps))
                res["grid"][1].append(events(grid_bwd, reps))
                res["grid kernels"][0].append(res["grid"][0][-1])
                res["grid kernels"][1].append(events(grid_wgrad_kernels, reps))
            torch.backends.cudnn.allow_tf32 = True
            fb, bb = cells + outs * 128, cells + outs * 256
            for k, (f, bw) in res.items():
                gf, gb = fb / (np.mean(f) * 1e-6) / 1e9, bb / (np.mean(bw) * 1e-6) / 1e9
                note = ""
                if k == "grid kernels":
                    note = "  fwd %.0f%% of 6.2 TB/s write, wgrad %.0f%% of 7.7 TB/s data sheet" % (100 * gf * 1e9 / WRITE_BPS,
                                                                                                   100 * gb * 1e9 / DATASHEET_BPS)
                say("%-14s %-26s %24s %24s %10.0f %10.0f%s" % ("V=%d n=%d" % (V, n), k, spread(f), spread(bw), gf, gb, note))
            del g, x, gy, yg, go, yo, work
            torch.cuda.empty_cache()


def learner(sb, say, rounds, arch="custom"):
    from snakes_b200 import selfplay
    nsteps = 16
    nature = arch == "nature"
    say("\n2. learner, 2 snakes on 19x19, nsteps %d, one opponent model; ms, mean [min-max] over %d rounds" % (nsteps, rounds)
        + ("; nature_cnn, atari84 env + RGB models against grid env + grid models" if nature else ""))
    say("%-8s %-7s %28s %28s %16s" % ("N", "mode", "Runner.run per step", "Model.train per minibatch", "mb_obs bytes"))
    for N in (32, 4096, 16384):
        setups = {}
        for mode in ("atari84" if nature else "native", "grid"):
            torch.manual_seed(0)
            env = sb.SnakeVecEnv(N, size=19, n_snakes=2, seed=1, obs_mode=mode)
            grid = mode == "grid"
            shape = (84, 84, 3) if mode == "atari84" else (21, 21, 3)
            model = selfplay.Model(shape, 5, arch=arch, device=env.device, grid=grid)
            opp = selfplay.Model(shape, 5, arch=arch, device=env.device, trainable=False, grid=grid)
            runner = selfplay.Runner(env, model, [opp], nsteps)
            setups[mode] = (env, model, runner)
        mb_size = min(N * nsteps // 4, 32768)
        res = {m: ([], []) for m in setups}
        for _ in range(rounds):
            for mode, (env, model, runner) in setups.items():
                out = runner.run()   # warm-up of this round's shapes
                torch.cuda.synchronize()
                t = time.perf_counter()
                for _ in range(3):
                    out = runner.run()
                torch.cuda.synchronize()
                res[mode][0].append((time.perf_counter() - t) * 1e3 / (3 * nsteps))
                obs, returns, masks, actions, values, neglogp = out[:6]
                mb = torch.randperm(N * nsteps, device=env.device)[:mb_size]
                args = (obs[mb], returns[mb], masks[mb], actions[mb], values[mb], neglogp[mb])
                model.train(2.5e-4, 0.2, *args)
                torch.cuda.synchronize()
                t = time.perf_counter()
                for _ in range(5):
                    model.train(2.5e-4, 0.2, *args)
                torch.cuda.synchronize()
                res[mode][1].append((time.perf_counter() - t) * 1e3 / 5)
        for mode, (env, model, runner) in setups.items():
            r, tr = res[mode]
            say("%-8d %-7s %28s %28s %16d   (minibatch %d)" % (N, mode, "%.3f [%.3f-%.3f]" % (np.mean(r), min(r), max(r)),
                                                          "%.3f [%.3f-%.3f]" % (np.mean(tr), min(tr), max(tr)),
                                                          runner.mb_obs.numel(), mb_size))
            env.close()
        del setups
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--part", choices=("all", "input", "learner"), default="all")
    ap.add_argument("--arch", choices=("custom", "nature"), default="custom")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe needs a CUDA device"
    import snakes_b200 as sb
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("card: %s" % card())
    say("torch %s, cuDNN %s" % (torch.__version__, torch.backends.cudnn.version()))
    if args.part in ("all", "input"):
        input_stage(sb, say, args.rounds, args.arch)
    if args.part in ("all", "learner"):
        learner(sb, say, args.rounds, args.arch)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
