"""Cost of the arena (snk_tally, snakes_b200.arena; DESIGN.md section 4.18) on one GPU:

    python tools/arena_probe.py [--out profiles/r10_arena_probe.txt]

1. k_tally alone, CUDA events over 2 000 back-to-back launches after one real step, at 131 072 envs x 2 seats (lane
   family, 2x19x19 classic) and 32 768 envs x 16 seats (ring family, 16x64x64 cut).  episodes_per_env is set out of
   reach, so every launch does the full work of a step (no env is ever retired); the step kernel alone is timed the
   same way for scale.  The bytes it must move are counted from the shapes.
2. The per-step split of `arena.play`'s loop at 16 384 envs on 2x19x19 grid with two `custom` grid models: policy
   forwards, env step, tally (CUDA events around each part) and the finished-count poll (host clock around the 8-byte
   read, which synchronises), over 256 steps after 32 warm-up steps, and play() end to end for comparison."""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import snakes_b200 as sb  # noqa: E402
from snakes_b200 import _lib, arena  # noqa: E402
from snakes_b200.selfplay import Model  # noqa: E402

lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def tally_fn(env, n_groups, E):
    L = _lib.lib()
    out = (C.c_size_t * 2)()
    _lib.check(L.snk_tally_layout(env._h, out))
    work = torch.zeros(-(-int(out[0]) // 4), dtype=torch.int32, device=env.device)
    counts = torch.zeros((n_groups, env.S, int(out[1])), dtype=torch.int64, device=env.device)
    done = torch.zeros(1, dtype=torch.int64, device=env.device)
    group = (torch.arange(env.N, device=env.device) * n_groups // env.N).to(torch.int32)
    args = (C.c_void_p(group.data_ptr()), n_groups, E, C.c_void_p(work.data_ptr()), C.c_void_p(counts.data_ptr()),
            C.c_void_p(done.data_ptr()))
    keep = (work, counts, done, group)

    def f():
        _lib.check(L.snk_tally(env._h, *args, env._stream()))
    f.keep = keep
    return f, done


def events_us(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1000.0 / iters


def tally_alone(N, S, size, rules, iters=2000):
    env = sb.SnakeVecEnv(N, size=size, n_snakes=S, rules=rules, seed=1)
    env.reset()
    act = env.gen_actions(0, 1)
    for t in range(40):   # past the first deaths, so a step's outputs hold dones and fruit
        env.step(env.gen_actions(t, 1, out=act))
    tally, _ = tally_fn(env, 2, 1 << 30)
    done_frac = env._done_u8.float().mean().item()
    us = events_us(tally, iters)
    step_us = events_us(lambda: env.step(act), 200)
    # per env: reward_all 4S + done 1 + t 4 (read and written); on done also group, length, episodes and the 8S of the
    # per-seat values; fruit and death updates are rare
    bytes_ = N * (4 * S + 1 + 8) + done_frac * N * (4 + 4 + 8 + 16 * S)
    say("k_tally  N=%-7d S=%-2d %-10s %-5s kernel %-26s  %.2f us/launch (%d launches)  step %.2f us  done fraction %.3f"
        "  ~%.2f MB -> %.0f GB/s" % (N, S, "%dx%d" % (size, size), rules, env.launch_info()["kernel"], us, iters, step_us,
                                     done_frac, bytes_ / 1e6, bytes_ / us / 1e3))
    env.close()
    return us


def play_split(N=16384, steps=256, warm=32):
    env = sb.SnakeVecEnv(N, size=19, n_snakes=2, seed=3, obs_mode="grid")
    torch.manual_seed(0)
    A, B = [Model((env.V, env.V, 3), env.action_space.n, device=env.device, trainable=False, grid=True) for _ in range(2)]
    lay = arena.blocks(N, 1, 2)
    calls = []
    for _, r, b0, b1 in lay:
        for i, p in enumerate((A, B)):
            calls.append((p, b0, b1, arena.seat_of(i, r, 2)))
    tally, done = tally_fn(env, 2, 1 << 30)
    actions = torch.zeros((N, 2), dtype=torch.int8, device=env.device)
    env.reset()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    tot = [0.0, 0.0, 0.0]
    poll_s, polls = 0.0, 0
    for t in range(warm + steps):
        ev[0].record()
        obs = env.obs
        for p, b0, b1, s in calls:
            actions[b0:b1, s] = p.step(obs[b0:b1], s)[0].to(torch.int8)
        ev[1].record()
        env.step(actions)
        ev[2].record()
        tally()
        ev[3].record()
        if (t + 1) % arena.POLL_STEPS == 0:
            h0 = time.perf_counter()
            int(done.item())
            dt = time.perf_counter() - h0
            if t >= warm:
                poll_s += dt
                polls += 1
        ev[3].synchronize()
        if t >= warm:
            for k in range(3):
                tot[k] += ev[k].elapsed_time(ev[k + 1]) * 1000.0
    fwd, stp, tal = (x / steps for x in tot)
    # the poll's own cost: a synchronising 8-byte read right after a synchronise (the queue is empty) -- its latency
    torch.cuda.synchronize()
    h0 = time.perf_counter()
    for _ in range(200):
        int(done.item())
    poll_us = (time.perf_counter() - h0) / 200 * 1e6
    per_step_poll = poll_us / arena.POLL_STEPS
    total = fwd + stp + tal + per_step_poll
    say("play split  N=%d 2x19x19 grid, two custom grid models (4 forwards of %d grids per step), %d steps:" % (N, N // 2, steps))
    say("  policy forwards %9.1f us/step  %5.2f %%" % (fwd, 100 * fwd / total))
    say("  env step        %9.1f us/step  %5.2f %%" % (stp, 100 * stp / total))
    say("  tally           %9.1f us/step  %5.2f %%" % (tal, 100 * tal / total))
    say("  poll            %9.1f us/step  %5.2f %%  (%.1f us per 8-byte read, one read per %d steps)"
        % (per_step_poll, 100 * per_step_poll / total, poll_us, arena.POLL_STEPS))
    say("  tally + poll    %9.2f %% of the step" % (100 * (tal + per_step_poll) / total))
    torch.manual_seed(0)
    h0 = time.perf_counter()
    rec, = arena.play(env, [(A, B)], episodes=1, seed=1)
    dt = time.perf_counter() - h0
    say("play() end to end: %d envs x 1 episode, %d steps, %.2f s, %.1f us/step; score A %.4f, mean episode length %.1f"
        % (N, rec["steps"], dt, dt / rec["steps"] * 1e6, rec["players"][0]["score"], rec["episode_len"]))
    env.close()
    return tal, per_step_poll, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_arena_probe.txt"))
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    say("GPU: %s  (name, power limit, max SM clock)" % smi)
    say("torch %s" % torch.__version__)
    lane = tally_alone(131072, 2, 19, "classic")
    tally_alone(32768, 16, 64, "cut")
    tal, poll, total = play_split()
    say("goal k_tally <= 5 us at 131072 x 2: %s (%.2f us)" % ("met" if lane <= 5.0 else "MISSED", lane))
    say("goal tally + poll <= 2 %% of an arena step with model players: %s (%.2f %%)"
        % ("met" if (tal + poll) <= 0.02 * total else "MISSED", 100 * (tal + poll) / total))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
