"""Timing of the per-env state entry points at the headline shape (131 072 envs of 2 snakes on 19x19, classic).

    python tools/envstate_probe.py [--envs N] [--iters K] [--out FILE]

After warm-up, CUDA events around `iters` back-to-back launches of each operation give the mean time per call; bytes are
what the operation has to move (blob bytes plus the private record / chain / frame_ok bytes it reads or writes), and the
floor is those bytes at the 6.2 TB/s a write stream sustains on a B200 (DESIGN.md section 4.11).  The host path
(dump_state_blob + load_state_blob, synchronous, through pageable memory) is timed with a host clock for comparison.  The
card's name and power limit are printed with the numbers.  Needs a GPU; it writes nothing but --out."""
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


def timed(fn, iters):
    fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) * 1e3 / iters  # us per call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=131072)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe needs a CUDA device"
    import snakes_b200 as sb

    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    N, it = args.envs, args.iters
    env = sb.SnakeVecEnv(N, size=19, n_snakes=2, rules="classic", seed=0)
    env.reset()
    for t in range(64):  # warm-up: bodies of a few segments, as in the bench workload
        env.step(env.gen_actions(t, 1))
    torch.cuda.synchronize()
    st = env.dump_state()
    mean_len = float(st["len"].astype(np.float64).sum(1).mean())
    RW = 16                                   # record words of the lane family at S = 2
    rec_b, obs_b = 4 * RW, env.obs[0].numel()
    chain_b = lambda lens: float(4 * np.maximum(0, (lens.astype(np.int64) - 2) // 16).sum(1).mean())  # chain words >= 1
    cw = chain_b(st["len"])
    # a restore reads the scalars, len / grow_to / vel, the fruits and each body up to its length (32-byte sectors),
    # not the zero padding of the rows
    body_sectors = float((np.ceil(st["len"].astype(np.float64) * 2 / 32) * 32).sum(1).mean())
    rd = 5 * 4 + 2 * 5 + 2 * 2 + body_sectors
    say("card: %s" % card())
    say("shape: %d envs, 2 snakes on 19x19, classic; after 64 random steps mean body cells per env %.2f; %d calls per row"
        % (N, mean_len, it))
    say("%-44s %10s %12s %9s %10s %7s" % ("operation", "us/call", "bytes", "GB/s", "floor us", "x floor"))

    def row(name, us, nbytes):
        floor = nbytes / FLOOR_BPS * 1e6
        say("%-44s %10.2f %12.0f %9.0f %10.2f %7.2f" % (name, us, nbytes, nbytes / us / 1e3, floor, us / floor))

    rng = np.random.RandomState(0)
    sub = np.sort(rng.choice(N, size=N // 10, replace=False))
    d_all = torch.arange(N, dtype=torch.int64, device=env.device)
    d_sub = torch.as_tensor(sub, device=env.device)
    blob_all = sb.EnvStates.empty(env, N)
    blob_sub = sb.EnvStates.empty(env, len(sub))
    per_env_blob = blob_all.lay.total_bytes / N
    # save: the whole blob written, record (+ chain words) read; restore: the blob's live bytes read (rd), record
    # (+ chain words) and frame_ok written
    row("save_envs all", timed(lambda: env.save_envs(out=blob_all), it), N * (per_env_blob + rec_b + cw))
    row("save_envs all (index tensor)", timed(lambda: env.save_envs(d_all, out=blob_all), it), N * (per_env_blob + rec_b + cw + 8))
    row("save_envs random 10%", timed(lambda: env.save_envs(d_sub, out=blob_sub), it), len(sub) * (per_env_blob + rec_b + cw + 8))
    env.save_envs(out=blob_all); env.save_envs(d_sub, out=blob_sub)
    row("restore_envs all, observe=False", timed(lambda: env.restore_envs(blob_all, observe=False), it),
        N * (rd + rec_b + cw + 1))
    row("restore_envs random 10%, observe=False", timed(lambda: env.restore_envs(blob_sub, d_sub, observe=False), it),
        len(sub) * (rd + rec_b + cw + 1 + 8))
    row("restore_envs all, observe=True", timed(lambda: env.restore_envs(blob_all, observe=True), it),
        N * (rd + rec_b + cw + 1) + N * (rec_b + obs_b))
    row("restore_envs random 10%, observe=True", timed(lambda: env.restore_envs(blob_sub, d_sub, observe=True), it),
        len(sub) * (rd + rec_b + cw + 1 + 8) + N * (rec_b + obs_b))
    # copy: record (+ chain words) read and written, frame_ok written, two indices read
    perm = torch.as_tensor(rng.permutation(N), device=env.device)
    src, dst = perm[:65536].contiguous(), perm[65536:131072].contiguous()
    row("copy_envs 65536 disjoint pairs", timed(lambda: env.copy_envs(src, dst, observe=False), it),
        65536 * (2 * (rec_b + cw) + 1 + 16))
    src1 = torch.full((4096,), int(perm[0]), dtype=torch.int64, device=env.device)
    dst1 = perm[1:4097].contiguous()
    row("copy_envs 1 -> 4096", timed(lambda: env.copy_envs(src1, dst1, observe=False), it), 4096 * (2 * (rec_b + cw) + 1 + 16))
    pair_blob = sb.EnvStates.empty(env, 65536)

    def via_blob():
        env.save_envs(src, out=pair_blob)
        env.restore_envs(pair_blob, dst, observe=False)

    row("save + restore of the same 65536 pairs", timed(via_blob, it), 65536 * (per_env_blob + rd + 2 * (rec_b + cw + 8) + 1))
    row("one step (reference point)", timed(lambda: env.step(env._actions), it), N * (2 * rec_b + obs_b))
    # the host path
    reps = 5
    env.dump_state_blob()
    t0 = time.perf_counter()
    for _ in range(reps):
        host = env.dump_state_blob()
    t_dump = (time.perf_counter() - t0) / reps * 1e6
    t0 = time.perf_counter()
    for _ in range(reps):
        env.load_state_blob(host)
    t_load = (time.perf_counter() - t0) / reps * 1e6
    row("host dump_state_blob (synchronous)", t_dump, blob_all.lay.total_bytes)
    row("host load_state_blob (synchronous)", t_load, blob_all.lay.total_bytes)
    say("canonical blob: %.1f bytes per env, %.1f MB for %d envs; private record %d bytes per env"
        % (per_env_blob, blob_all.lay.total_bytes / 1e6, N, rec_b))
    env.check_errors()
    env.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
