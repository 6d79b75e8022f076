"""Cost and strength of rollout search (snk_clone_envs, snakes_b200.search; DESIGN.md section 4.19) on one GPU:

    python tools/search_probe.py [--out profiles/r12_search_probe.txt] [--skip-arena]

1. Moving env states into search slots, CUDA events over back-to-back launches, 2x19x19 classic: cross-handle clone
   (native game handle -> grid search handle), in-handle copy_envs (one native handle holding roots and slots) and
   save_envs + restore_envs through a canonical blob, for a 1 -> A R = 40 fan-out of 8 192 roots (327 680 slots) and for
   65 536 disjoint pairs.  Game envs hold states of 32 random steps after a reset.
2. Time per decision (one RolloutSearch.act) at M = 8 192 roots, R = 8, H = 16: 2x19x19 classic with scripted
   rollouts, and 3x10 cut with random rollouts.  act() end to end (CUDA events around 10 calls after 2 warm-up calls,
   eager launches from Python), and its parts each timed alone over back-to-back launches: clone, rollout policy, step
   of the search handle, bookkeeping (begin + H accumulates + pick).
3. Arena scores on 2x19x19 classic, 16 384 envs, 2 episodes each: Search() against 'random' and against 'scripted'."""
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

lines = []


def say(s):
    print(s, flush=True)
    lines.append(s)


def events_us(fn, iters, warm=3):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters


def primed(N, obs_mode="native", **kw):
    env = sb.SnakeVecEnv(N, obs_mode=obs_mode, seed=1, **kw)
    env.reset()
    for t in range(32):
        env.step(env.gen_actions(t, 1))
    return env


def move_states(kw, n_roots, fan):
    """(clone, copy, save + restore) in us for n_roots roots each into `fan` slots (fan = 1: disjoint pairs)."""
    n = n_roots * fan
    dev = torch.device("cuda", 0)
    game = primed(n_roots, **kw)
    dst_env = sb.SnakeVecEnv(n, obs_mode="grid", seed=2, **kw)
    src = torch.arange(n_roots, device=dev).repeat_interleave(fan) if fan > 1 else torch.randperm(n_roots, device=dev)
    slots = torch.arange(n, device=dev)
    clone = events_us(lambda: dst_env.clone_envs_from(game, src, slots, observe=False), 50)
    one = primed(n_roots + n, **kw)
    copy = events_us(lambda: one.copy_envs(src, slots + n_roots, observe=False), 50)
    blob = sb.EnvStates.empty(game, n)

    def save_restore():
        game.save_envs(src, out=blob)
        dst_env.restore_envs(blob, slots, observe=False)
    sr = events_us(save_restore, 50)
    save = events_us(lambda: game.save_envs(src, out=blob), 50)
    for e in (game, dst_env, one):
        e.check_errors()
        e.close()
    return clone, copy, sr, save, blob.blob.numel() / n


def decision(kw, M, R, H, rollout):
    game = primed(M, **kw)
    rs = sb.RolloutSearch(game, M, rollouts=R, horizon=H, rollout=rollout)
    se = rs.search_env
    roots = torch.arange(M, device=game.device)
    say("  search handle: %d envs, obs_mode %s, %s" % (se.N, se.obs_mode, se.launch_info()["kernel"]))
    for _ in range(2):
        rs.act(0, roots)
    torch.cuda.synchronize()
    h0 = time.perf_counter()
    act = events_us(lambda: rs.act(0, roots), 10, warm=0)
    host = (time.perf_counter() - h0) / 10 * 1e6
    n = M * rs.A * R
    src = roots.repeat_interleave(rs.A * R)
    clone = events_us(lambda: se.clone_envs_from(game, src, rs._slots[:n], observe=False), 50)
    if rollout == "scripted":
        policy = events_us(lambda: se.gen_scripted_actions(0, 1, 0.05, out=rs._actions), 50)
    else:
        policy = events_us(lambda: se.gen_actions(0, 1, out=rs._actions), 50)
    step = events_us(lambda: se.step(rs._actions), 50)
    L, h, st = se._L, se._h, se._stream()
    ret, active, acts = C.c_void_p(rs._ret.data_ptr()), C.c_void_p(rs._active.data_ptr()), C.c_void_p(rs._actions.data_ptr())
    begin = events_us(lambda: _lib.check(L.snk_search_begin(h, acts, 0, rs.A, R, M, ret, active, st)), 200)
    acc = events_us(lambda: _lib.check(L.snk_search_accumulate(h, 0, rs.A, R, M, ret, active, st)), 200)
    pick = events_us(lambda: _lib.check(L.snk_search_pick(h, rs.A, R, M, ret, C.c_void_p(rs.values.data_ptr()),
                                                          C.c_void_p(rs._pick.data_ptr()), 1, st)), 200)
    book = begin + H * acc + pick
    parts = clone + H * (policy + step) + book
    say("  act(): %.1f us per decision (device, events), %.1f us host clock; %.3f us per root, %.2e slot-steps/s"
        % (act, host, act / M, n * H / (act * 1e-6)))
    say("  parts timed alone: clone %.1f | policy %.1f x %d = %.1f | step %.1f x %d = %.1f | bookkeeping %.1f "
        "(begin %.2f, accumulate %.2f x %d, pick %.2f) | sum %.1f us = %.0f %% of act()"
        % (clone, policy, H, H * policy, step, H, H * step, book, begin, acc, H, pick, parts, 100 * parts / act))
    se.check_errors()
    rs.close()
    game.close()


def arena_scores():
    for opp in ("random", "scripted"):
        env = sb.SnakeVecEnv(16384, size=19, n_snakes=2, seed=1)
        h0 = time.perf_counter()
        rec, = arena.play(env, [(arena.Search(), opp)], episodes=2, seed=3)
        dt = time.perf_counter() - h0
        s, o = rec["players"]
        say("Search() vs %s: score %.4f (%d wins, %d draws, %d losses of %d episodes), fruits/episode %.2f vs %.2f, "
            "death rate %.3f vs %.3f, mean episode length %.1f, %d steps, %.1f s"
            % (opp, s["score"], s["wins"], s["draws"], s["losses"], s["episodes"], s["fruits_per_episode"],
               o["fruits_per_episode"], s["death_rate"], o["death_rate"], rec["episode_len"], rec["steps"], dt))
        env.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_search_probe.txt"))
    ap.add_argument("--skip-arena", action="store_true")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    say("GPU: %s  (name, power limit, max SM clock)" % smi)
    say("torch %s" % torch.__version__)
    classic = dict(size=19, n_snakes=2, rules="classic")
    say("1. states into search slots, 2x19x19 classic (us per call, CUDA events)")
    for roots, fan, what in ((8192, 40, "fan-out 8 192 roots x 40"), (65536, 1, "65 536 disjoint pairs")):
        clone, copy, sr, save, blob = move_states(classic, roots, fan)
        say("  %-26s clone_envs_from %.1f | copy_envs (one handle) %.1f | save_envs + restore_envs %.1f (save alone "
            "%.1f; %.0f blob bytes per env)" % (what, clone, copy, sr, save, blob))
    say("2. time per decision, M = 8192, R = 8, H = 16")
    say(" 2x19x19 classic, scripted rollouts (eps 0.05)")
    decision(classic, 8192, 8, 16, "scripted")
    say(" 3x10x10 cut, random rollouts")
    decision(dict(size=10, n_snakes=3, rules="cut"), 8192, 8, 16, "random")
    if not args.skip_arena:
        say("3. arena, 2x19x19 classic, 16 384 envs x 2 episodes, Search(rollouts=8, horizon=16, rollout='scripted')")
        arena_scores()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
