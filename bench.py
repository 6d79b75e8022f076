"""bench.py -- agent-steps/s of the batched multi-snake env step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
    python bench.py --impl reference [--gpus N] --steps K ...    # the reference's own CPU path
    torchrun --nproc-per-node N bench.py --gpus N ...            # one rank per GPU (weak scaling)
    python bench.py --steps K --warmup W --dump-outputs DIR      # also writes the last timed step's outputs as .npy

Workload: BASELINE.json configs[3] -- 2 snakes on 19x19, classic rules, 1M envs sharded over 8
GPUs, i.e. 131072 envs per GPU (weak scaling), uniform random actions from the Philox action
stream (already resident in HBM), K = S = 2 views of 21x21x3 uint8 per env.  One "step" = one
pass of the fused step kernel over every env of the rank; the K timed steps are ONE CUDA-graph
launch (snk_graph_create: K kernel nodes with programmatic dependent-launch edges and, under
N > 1, one ncclAllReduce node per step for the episode statistics).  Prints ONE JSON line on rank 0.

CPU legs (`--impl reference`, `cpu_baseline`): the reference's own SubprocVecEnv of Monitor(SnakeEnv)
(src/utils.py:34-49) when the reference is present (/root/reference, or its offline install under
baseline/_ref/ staged by oracle/stage_reference.py), else the repo's port of it (oracle/snake_oracle.py).
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 131072
SIZE, N_SNAKES, RULES = 19, 2, "classic"
WORKLOAD = "2-snake 19x19 classic, %d envs per GPU (BASELINE configs[3]: 1M envs over 8 GPUs), K=S=2 views" % ENVS_PER_GPU
METRIC, UNIT = "agent-steps/sec", "agent-steps/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


# ------------------------------------------------------------------ CPU paths
def _oracle_path():
    p = os.path.join(ROOT, "oracle")
    if p not in sys.path:
        sys.path.insert(0, p)


def _port_worker(remote, seed, rank):
    """SubprocVecEnv worker (subproc_vec_env.py:7-28) around the repo's port of the env: one env instance per
    process; step, reset at once on done, send (ob, reward, done, info) back through the pipe."""
    _oracle_path()
    import snake_oracle as so
    env = so.SnakeOracle(SIZE, N_SNAKES, N_SNAKES, 3, RULES, draws=so.PhiloxDraws(seed, rank))  # K = 3 views like SnakeEnv
    ep_r, ep_l = 0.0, 0
    while True:
        cmd, data = remote.recv()
        if cmd == "step":
            ob, r, d, info = env.step(data)
            ep_r += r
            ep_l += 1
            if d:
                info["episode"] = {"r": ep_r, "l": ep_l}
                ob = env.reset()
                ep_r, ep_l = 0.0, 0
            remote.send((ob, r, d, info))
        elif cmd == "reset":
            remote.send(env.reset())
        else:
            remote.close()
            break


class PortSubprocVecEnv(object):
    """Stand-in used ONLY when no reference tree travels with the repo: the same one-process-per-env, Pipe + pickle
    structure as the reference's SubprocVecEnv, around oracle/snake_oracle.py."""

    def __init__(self, n_procs, seed=0):
        import numpy as np
        self.np = np
        ctx = mp.get_context("fork")
        self.remotes, self.ps = [], []
        for i in range(n_procs):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_port_worker, args=(b, seed, i), daemon=True)
            p.start()
            b.close()
            self.remotes.append(a)
            self.ps.append(p)

    def reset(self):
        for r in self.remotes:
            r.send(("reset", None))
        return self.np.stack([r.recv() for r in self.remotes])

    def step(self, actions):
        for r, a in zip(self.remotes, actions):
            r.send(("step", a))
        obs, rews, dones, infos = zip(*[r.recv() for r in self.remotes])
        return self.np.stack(obs), self.np.stack(rews), self.np.stack(dones), infos

    def close(self):
        for r in self.remotes:
            r.send(("close", None))
        for p in self.ps:
            p.join(timeout=5)


def make_cpu_vec_env(n_procs):
    """(venv, kind): the reference's own SubprocVecEnv([Monitor(SnakeEnv)] * n_procs) when available, else the port."""
    _oracle_path()
    import ref_loader
    if ref_loader.available():
        return ref_loader.make_subproc_vec_env(n_procs, RULES, N_SNAKES, SIZE, seed=0), "reference", ref_loader.source()
    return PortSubprocVecEnv(n_procs), "port", None


def time_cpu_path(seconds, n_procs=None, steps=None, warmup_steps=20):
    """env-steps/s of the vectorised CPU path over `n_procs` worker processes (default: all cores)."""
    import numpy as np
    n_procs = n_procs or os.cpu_count() or 1
    venv, kind, src = make_cpu_vec_env(n_procs)
    venv.reset()
    rng = np.random.RandomState(0)
    act = lambda: [tuple(int(x) for x in row) for row in rng.randint(0, 5, size=(n_procs, N_SNAKES))]  # ppo_multi_agent_new.py:35-37
    for _ in range(warmup_steps):
        venv.step(act())
    t0 = time.perf_counter()
    n = 0
    while True:
        venv.step(act())
        n += 1
        if steps is not None:
            if n >= steps:
                break
        elif time.perf_counter() - t0 >= seconds:
            break
    dt = time.perf_counter() - t0
    venv.close()
    return {"env_steps_per_s": n * n_procs / dt, "vec_steps": n, "seconds": dt, "procs": n_procs, "kind": kind, "source": src}


def time_reference_inprocess(seconds=2.0):
    """The reference's own SnakeEnv.step in this process, one env, one core (SURVEY.md 8d: the raw in-process figure
    beside the SubprocVecEnv one); None when no reference tree is on the box."""
    _oracle_path()
    import numpy as np
    import ref_loader
    if not ref_loader.available():
        return None
    env = ref_loader.make_env(RULES, N_SNAKES, SIZE, np.random.RandomState(0))
    env.reset()
    rng = np.random.RandomState(1)
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < seconds:
        _, _, done, _ = env.step(tuple(int(x) for x in rng.randint(0, 5, size=N_SNAKES)))
        if done:
            env.reset()
        n += 1
    return n / (time.perf_counter() - t0)


def time_c_oracle(seconds=3.0, n=4096):
    """The C restatement on one core (context only: a far stronger CPU baseline than the reference's Python)."""
    _oracle_path()
    import c_oracle
    co = c_oracle.COracle(n, size=SIZE, n_snakes=N_SNAKES, rules=RULES)
    co.reset()
    acts = [c_oracle.gen_actions(co.cfg, t, 1) for t in range(16)]
    t0 = time.perf_counter()
    k = 0
    while time.perf_counter() - t0 < seconds:
        co.step(acts[k % 16])
        k += 1
    return k * n / (time.perf_counter() - t0)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _cpu_sample_text(r):
    what = ("the reference's own SubprocVecEnv of Monitor(SnakeEnv) (%s)" % r["source"]) if r["kind"] == "reference" \
        else "SubprocVecEnv-style harness around the repo's port of gym-snake (no reference tree on this box)"
    return "%d vec-steps over %d worker processes (1 env each, 3 views like SnakeEnv), %.1f s; %s; CPU %s" % (
        r["vec_steps"], r["procs"], r["seconds"], what, cpu_model())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # one host: rank 0 alone measures the CPU path
    cores = os.cpu_count() or 1
    # calibrate so that warmup + K steps end within a couple of minutes
    rate = time_cpu_path(3.0, cores)["env_steps_per_s"]
    budget = 60.0
    inner = max(1, int(budget * rate / (cores * max(args.steps, 1))))
    time_cpu_path(0, cores, steps=max(1, inner * min(args.warmup, 3)))
    r = time_cpu_path(0, cores, steps=inner * args.steps)
    agent = r["env_steps_per_s"] * N_SNAKES
    line = {
        "impl": "reference", "metric": METRIC, "value": agent, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["seconds"] * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs": cores, "reference_step": "%d vec-steps x %d envs" % (inner, cores),
                   "same_config": "same env (2 snakes, 19x19, classic, random actions); one env per host core instead of 131072 per GPU"},
        "cpu_baseline": {"value": agent, "unit": UNIT, "cores": cores, "kind": r["kind"], "sample": _cpu_sample_text(r)},
        "e2e": {"value": agent, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.005):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def git_head():
    try:
        return subprocess.check_output(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], stderr=subprocess.DEVNULL).decode().strip()
    except Exception:
        return None


# ------------------------------------------------------------------ this repo's CUDA path
def rank_parity(env, rank, steps=16, n_blocks=4, count=256):
    """VERDICT r1 item 1b: before the timed region every rank replays `steps` steps of n_blocks x count of ITS envs
    (global ids env_id_base + ...) against the C oracle -- observations, rewards, dones, num_snakes, Monitor r / l at
    every step and the full state at the end -- on the very handle the bench then times.  Returns True when bit-exact."""
    import numpy as np
    _oracle_path()
    import c_oracle
    N = env.N
    kw = dict(size=SIZE, n_snakes=N_SNAKES, rules=RULES, seed=0)
    bo = c_oracle.BlockOracles(c_oracle.BlockOracles.spread(N, n_blocks, count), env_id_base=rank * N, **kw)
    ok = True
    for (first, cnt, _), cobs in zip(bo.blocks, bo.reset()):
        ok &= np.array_equal(env.obs[first:first + cnt].cpu().numpy(), cobs)
    for t in range(steps):
        env.step(env.gen_actions(t, 1))
        for (first, cnt, co), (cobs, crew, cdone, cinfo) in zip(bo.blocks, bo.step_generated(t, 1, 5)):
            sl = slice(first, first + cnt)
            ok &= np.array_equal(env.obs[sl].cpu().numpy(), cobs)
            ok &= np.array_equal(env.rewards[sl].cpu().numpy(), crew)
            ok &= np.array_equal(env._done_u8[sl].cpu().numpy().astype(bool), cdone)
            ok &= np.array_equal(env.num_alive[sl].cpu().numpy(), cinfo["num_snakes"])
            ok &= np.array_equal(env.episode_return[sl].cpu().numpy(), cinfo["episode_r"])
            ok &= np.array_equal(env.episode_len[sl].cpu().numpy(), cinfo["episode_l"])
    for first, cnt, co in bo.blocks:
        dev, cpu = env.dump_state_range(first, cnt), co.state()
        ok &= all(np.array_equal(dev[k], cpu[k]) for k in cpu)
    return bool(ok), sum(c for _, c, _ in bo.blocks), steps


DUMP_OBS_ENVS = 4096   # 4096 x 21 x 21 x 6 float32 = 43 MB of observations: with the [N] arrays the dump stays under 64 MB


def dump_obs_envs(n):
    """The envs whose observations the dump holds: DUMP_OBS_ENVS of n drawn with a fixed seed, in ascending order."""
    import numpy as np
    return np.sort(np.random.RandomState(0).choice(n, min(DUMP_OBS_ENVS, n), replace=False))


def dump_outputs(path, env):
    """Writes what the last timed step handed its caller as float32 .npy files in `path`: reward, done, num_snakes and
    Monitor's episode return and length (where done; 0 elsewhere) of every env, and the observations of the envs
    dump_obs_envs picks.  Two builds run with the same arguments can then be compared array by array."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    idx = dump_obs_envs(env.N)
    arrays = {"obs": env.obs[torch.as_tensor(idx, device=env.device)], "reward": env.rewards, "done": env._done_u8,
              "num_snakes": env.num_alive, "episode_return": env.episode_return, "episode_length": env.episode_len}
    for name, x in arrays.items():
        np.save(os.path.join(path, name + ".npy"), x.cpu().numpy().astype(np.float32))


def time_config(sb, torch, dev, peak, name, N, kw, steps, n_batches=16, warm=40):
    """One secondary configuration through the graph path: us per step, fraction of the HBM roofline, mean body length."""
    env = sb.SnakeVecEnv(N, seed=0, device=dev.index, **kw)
    env.reset()
    acts = torch.empty((n_batches, N, env.S), dtype=torch.int8, device=dev)
    for t in range(n_batches):
        env.gen_actions(t, 1, out=acts[t])
    gw, g = env.make_graph(acts, T=warm), env.make_graph(acts, T=steps)
    gw.launch()
    env.reset_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record(); g.launch(); e1.record()
    torch.cuda.synchronize(dev)
    us = e0.elapsed_time(e1) * 1e3 / steps
    st = env.stats(reduce=False)
    env.check_errors()
    sum_len = st["body_cells"] / max(st["env_steps"], 1.0)
    alg = env.algorithmic_bytes_per_step(sum_len)
    out = {"config": name, "envs": N, "us_per_step": us, "steps": steps, "agent_steps_per_s": N * env.S / (us * 1e-6),
           "algorithmic_bytes_per_env_step": alg, "frac": alg * N / (us * 1e-6) / 1e9 / peak, "mean_sum_len": sum_len,
           "episodes_per_env_step": st["episodes"] / max(st["env_steps"], 1.0), "kernel": env.launch_info()["kernel"]}
    gw.close(); g.close(); env.close()
    del acts
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    # stdout carries exactly ONE JSON line: everything libraries print (NCCL's banner and its NCCL_DEBUG log go to
    # fd 1) is sent to stderr, the line is written to the saved descriptor at the end.  NCCL_DEBUG is left as the
    # caller set it.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import torch
    import torch.distributed as dist
    import snakes_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"

    N = ENVS_PER_GPU
    env = snakes_b200.SnakeVecEnv(N, size=SIZE, n_snakes=N_SNAKES, rules=RULES, seed=0, device=local, env_id_base=rank * N)
    S = env.S
    env.reset()
    use_comm = (world > 1 or args.collective) and not args.no_collective
    if use_comm:
        env.init_comm(mode=args.comm)   # from here on every step sums the 8 statistics doubles over all ranks

    # ---- parity of THIS rank's envs on THIS handle, before anything is timed
    ok, n_checked, n_steps = rank_parity(env, rank)
    ranks_ok = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ranks_ok)
    parity = {"ranks_ok": int(ranks_ok.item()), "ranks": world, "envs_per_rank": n_checked, "steps": n_steps,
              "checked": "obs, reward, done, num_snakes, Monitor r/l every step + full state, vs the C oracle, on the timed handle"}

    # ---- headline: K steps = ONE graph launch
    K, W = args.steps, args.warmup
    n_act = max(1, min(K, args.action_batches))  # distinct action batches resident in HBM, cycled
    acts = torch.empty((n_act, N, S), dtype=torch.int8, device=dev)
    for t in range(n_act):
        env.gen_actions(100 + t, 1, out=acts[t])
    g_warm = env.make_graph(acts, T=max(W, 1))
    g_main = env.make_graph(acts, T=K)
    g_warm.launch()
    env.reset_stats()
    l0 = env.launch_count()
    c0 = env.comm_info()["allreduces"] if use_comm else 0
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g_main.launch()
    e1.record()
    barrier()
    clocks = sampler.result()
    launches = env.launch_count() - l0
    ms = max_over_ranks(e0.elapsed_time(e1))
    stats_local = env.stats(reduce=False)
    if args.dump_outputs and rank == 0:   # before anything else steps the env
        dump_outputs(args.dump_outputs, env)
    collective = None
    if use_comm:
        barrier()                   # every rank has finished its K steps: all pushes / all-reduces have landed
        stats = env.stats_global()  # what the in-loop reduction delivered
        check = env.stats(reduce=True)  # the same sums through torch.distributed, after the fact
        info = env.comm_info()
        collective = {"bytes": 8 * 8, "per": "step", "count": info["allreduces"] - c0, "inside_timed_region": True,
                      "ranks": info["ranks"], "mode": args.comm,
                      "matches_torch_all_reduce": all(abs(stats[k] - check[k]) < 1e-6 for k in stats)}
        if args.comm == "nccl":
            collective["us"] = env.comm_latency_us(200)
            collective["nccl_version"] = info["nccl_version"]
            collective["how"] = ("raw ncclAllReduce(8 x f64, sum) issued by libsnk.so on a high-priority side stream, one graph node "
                                 "per step, overlapped with the next step and read one step late (snk_comm_init / snk_get_stats_global)")
        else:
            collective["how"] = ("fused into the step kernel: its first CTA stores the rank's 8 running sums (as of the previous step) "
                                 "into every peer's inbox over NVLink (cudaIpc peer memory, posted 8-byte stores, no fence, no "
                                 "rendezvous); a reader adds its own sums and the peers' latest pushes "
                                 "(snk_peer_connect / snk_get_stats_global)")
        # what the reduction costs: the same K steps with it switched off, outside the headline timing
        env.comm_enable(False)
        g_off = env.make_graph(acts, T=K)
        g_off.launch()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(); g_off.launch(); f1.record()
        barrier()
        ms_off = max_over_ranks(f0.elapsed_time(f1))
        g_off.close()
        env.comm_enable(True)
        collective["us_per_step_with"] = ms / K * 1e3
        collective["us_per_step_without"] = ms_off / K * 1e3
        env.reset_stats()
    else:
        stats = stats_local
    g_warm.close(); g_main.close()

    # ---- the same stream with the action generator in the loop (SURVEY.md 8d: report both): k_gen_actions + step kernel
    # per step, issued eagerly (two C calls per step; the device is the slower side)
    Kg = min(K, 400)
    for t in range(10):
        env.step_async(env.gen_actions(5000 + t, 1, out=acts[0])); env._pending = False
    barrier()
    ga0, ga1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ga0.record()
    for t in range(Kg):
        env.step_async(env.gen_actions(5010 + t, 1, out=acts[t % n_act])); env._pending = False
    ga1.record()
    barrier()
    ms_gen = max_over_ranks(ga0.elapsed_time(ga1))
    with_action_gen = {"value": float(N) * world * Kg * S / (ms_gen * 1e-3), "unit": UNIT, "us_per_step": ms_gen / Kg * 1e3, "steps": Kg,
                       "note": "k_gen_actions (Philox uniform actions, N*S bytes) + step kernel per step, eager launches"}

    # ---- second action stream (SURVEY.md 8d): fruit-seeking policy computed on the device every step (one extra small
    # kernel per step, inside the timed region and inside the graph); snakes get long, resets get rare
    Ks = max(50, K // 4)
    g_sw = env.make_scripted_graph(300, step0=0, seed=7)
    g_sw.launch()
    torch.cuda.synchronize()
    # a few eager steps before the timed graph is captured: the lane path picks its fused or its two-kernel form from the
    # body-length statistics the step kernels post to the host (DESIGN.md 4.8), and a graph keeps the form it was captured with
    for t in range(4):
        env.step_async(env.gen_scripted_actions(300 + t, seed=7)); env._pending = False
    torch.cuda.synchronize()
    step0 = 304
    blob_s = env.dump_state_blob()
    g_s = env.make_scripted_graph(Ks, step0=step0, seed=7)
    kernel_s = env.launch_info()["kernel"]
    env.reset_stats()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    g_s.launch()
    s1.record()
    barrier()
    ms_s = max_over_ranks(s0.elapsed_time(s1))
    stats_s = env.stats(reduce=True)
    sum_len_s = stats_s["body_cells"] / max(stats_s["env_steps"], 1.0)
    alg_s = env.algorithmic_bytes_per_step(sum_len_s)
    # the step kernel(s) alone in the same regime: the first Ka action batches of that stream recorded, the state
    # restored, and the same steps replayed from HBM without the policy kernel between them
    Ka = min(Ks, 100)
    env.load_state_blob(blob_s)
    acts_s = torch.empty((Ka, N, S), dtype=torch.int8, device=dev)
    for t in range(Ka):
        env.gen_scripted_actions(step0 + t, seed=7, out=acts_s[t]); env.step_async(acts_s[t]); env._pending = False
    torch.cuda.synchronize()
    env.load_state_blob(blob_s)
    g_a = env.make_graph(acts_s, T=Ka)
    env.reset_stats()
    barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record(); g_a.launch(); a1.record()
    barrier()
    ms_a = max_over_ranks(a0.elapsed_time(a1))
    stats_a = env.stats(reduce=False)
    alg_a = env.algorithmic_bytes_per_step(stats_a["body_cells"] / max(stats_a["env_steps"], 1.0))
    g_a.close()
    scripted = {"value": float(N) * world * Ks * S / (ms_s * 1e-3), "unit": UNIT, "ms_per_step": ms_s / Ks, "steps": Ks,
                "mean_sum_len": sum_len_s, "algorithmic_bytes_per_env_step": alg_s,
                "frac": alg_s * N / (ms_s * 1e-3 / Ks) / 1e9 / peak,
                "episodes_per_env_step": stats_s["episodes"] / max(stats_s["env_steps"], 1.0),
                "kernel": kernel_s,
                "step_only": {"us_per_step": ms_a / Ka * 1e3, "steps": Ka, "value": float(N) * world * Ka * S / (ms_a * 1e-3),
                              "frac": alg_a * N / (ms_a * 1e-3 / Ka) / 1e9 / peak,
                              "note": "the same regime without the policy kernel: the stream's first action batches recorded and replayed from HBM"},
                "note": "scripted fruit-seeking policy kernel + step kernel(s) per step, all inside the timed region (one graph); "
                        "value / frac include the policy kernel, step_only excludes it"}
    g_sw.close(); g_s.close()
    env.check_errors()
    mean_sum_len = stats["body_cells"] / max(stats["env_steps"], 1.0)
    alg_bytes = env.algorithmic_bytes_per_step(mean_sum_len)
    value = float(N) * world * K * S / (ms * 1e-3)

    # ---- e2e: the same step through the reference-facing VecEnv call with HOST buffers (numpy in / numpy out like
    # SubprocVecEnv.step_wait): actions H2D, fused kernel, obs + reward + done + num_snakes D2H, every step
    Ke = max(3, min(K, args.e2e_steps))
    h_acts = [acts[t % n_act].cpu().numpy() for t in range(8)]

    def time_host(host_views):
        henv = snakes_b200.SnakeVecEnv(N, size=SIZE, n_snakes=N_SNAKES, rules=RULES, seed=0, device=local,
                                       env_id_base=rank * N, host_io=True, host_views=host_views, host_copy=False)
        henv.reset()
        for t in range(3):
            henv.step(h_acts[t % 8])
        barrier()
        t0 = time.perf_counter()
        for t in range(Ke):
            henv.step(h_acts[t % 8])
        torch.cuda.synchronize(dev)
        dt = max_over_ranks(time.perf_counter() - t0)
        node = henv.host_numa_node
        henv.close()
        return float(N) * world * Ke * S / dt, dt / Ke, node

    e2e_value, e2e_s, numa = time_host(None)
    e2e_main, e2e_main_s, _ = time_host(1)
    h2d = N * S
    d2h = N * env.V * env.V * 3 * env.K + N * 4 + 2 * N + 8 * N
    d2h_main = N * env.V * env.V * 3 + N * 4 + 2 * N + 8 * N

    # obs stays in HBM for an on-device learner (north_star): numpy actions -> pinned slot -> H2D -> fused kernel ->
    # reward + done + num_snakes + Monitor r/l D2H into the slot's pinned block, one C call per step
    # (SnakeVecEnv.step_scalars_async), up to four steps in flight; every step's scalars are waited for and read two steps late,
    # as a learner's bookkeeping would
    Kr = Ke * 16
    env.reset()   # back to the headline regime (the scripted stream above left long snakes)
    for t in range(8):
        env.wait_scalars(env.step_scalars_async(h_acts[t % 8]))
    barrier()
    t0 = time.perf_counter()
    acc, tickets = 0.0, []
    for t in range(Kr):
        tickets.append(env.step_scalars_async(h_acts[t % 8]))
        if t >= 2:   # every step's scalars are read, two steps late
            rew, done = env.wait_scalars(tickets[t - 2])[:2]
            acc += float(rew[0]) + float(done[0])
    for tk in tickets[-2:]:
        rew, done = env.wait_scalars(tk)[:2]
        acc += float(rew[0]) + float(done[0])
    torch.cuda.synchronize(dev)
    e2e_resident = float(N) * world * Kr * S / max_over_ranks(time.perf_counter() - t0)

    launch_s = ms * 1e-3 / K
    achieved = alg_bytes * N / launch_s / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj.get("dram_bytes_per_launch")
        traffic_src = {k: tj.get(k) for k in ("source", "captured_at_commit", "kernel", "note") if k in tj}
    kernel_info = env.launch_info()
    env.close()
    del acts
    torch.cuda.empty_cache()

    # ---- the other BASELINE configurations, each a few hundred steps through the same graph path (1 GPU only:
    # they are secondary lines, outside the headline timing)
    configs = None
    if world == 1 and not args.no_configs:
        configs = []
        specs = [("configs[1] 2-snake 10x10, 4096 envs", 4096, dict(size=10, n_snakes=2, rules="classic"), 400),
                 ("configs[2] 3-snake 10x10 cut, 65536 envs", 65536, dict(size=10, n_snakes=3, rules="cut"), 300),
                 ("configs[3] atari84 (WarpFrame 84x84), 2-snake 19x19, 131072 envs", 131072,
                  dict(size=19, n_snakes=2, rules="classic", obs_mode="atari84"), 60),
                 ("configs[4] 16-snake 64x64 cut, 32768 envs (per-GPU shard of 8)", 32768, dict(size=64, n_snakes=16, rules="cut"), 40),
                 ("configs[4] 16-snake 64x64 cut, 262144 envs (whole job on 1 GPU)", 262144, dict(size=64, n_snakes=16, rules="cut"), 12)]
        for name, n, kw, steps in specs:
            try:
                configs.append(time_config(snakes_b200, torch, dev, peak, name, n, kw, steps, n_batches=8 if n >= 262144 else 16,
                                           warm=8 if n >= 262144 else 40))
            except Exception as exc:  # e.g. not enough free HBM for the 262144-env large field
                configs.append({"config": name, "error": str(exc)[:200]})

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "envs_total": N * world, "rules": RULES, "size": SIZE, "n_snakes": S,
                       "obs": "uint8 [N,21,21,6]", "actions": "Philox uniform{0..4}, %d batches resident in HBM" % n_act,
                       "l2": "per-step working set (347 MB obs stream + state) exceeds the 126 MB L2; no explicit flush",
                       "step_loop": "one CUDA graph launch of K step kernels (programmatic dependent-launch edges)",
                       "kernel": kernel_info, "mean_sum_len": mean_sum_len},
            "clocks": clocks,
            "parity": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": Ke,
                    "pcie_gbs_per_gpu": (h2d + d2h) / e2e_s / 1e9, "pinned_numa_node": numa,
                    "path": "SnakeVecEnv(host_io=True).step: numpy actions -> pinned, NUMA-local -> H2D -> fused kernel -> "
                            "ALL K views + reward + done + num_snakes + Monitor r/l D2H (snk_step_host_async + sync); PCIe-bound"},
            "e2e_main_view": {"value": e2e_main, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_main, "steps": Ke,
                              "pcie_gbs_per_gpu": (h2d + d2h_main) / e2e_main_s / 1e9,
                              "note": "host_views=1: only the main snake's view crosses PCIe (all the reference learner stores, "
                                      "ppo_multi_agent_new.py:181); the other views stay in HBM"},
            "e2e_obs_resident": {"value": e2e_resident, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": N * 14,
                                 "steps": Kr, "note": "obs stays in HBM for an on-device learner (north_star); numpy actions H2D and reward + "
                                                      "done + num_snakes + Monitor r/l D2H every step through four pinned slots, the copies on their own "
                                                      "streams beside the step stream (SnakeVecEnv.step_scalars_async -> snk_step_scalars_async: "
                                                      "one C call per step, up to four steps in flight, every step's scalars read two steps late)"},
            "gpu_launches": int(launches) * world,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel_info["kernel"],
                         "algorithmic_bytes_per_env_step": alg_bytes, "env_steps_per_launch": N,
                         "launch_us": launch_s * 1e6},
            "episode_stats": stats,
            "with_action_gen": with_action_gen,
            "scripted_policy": scripted,
        }
        if collective:
            line["collective"] = collective
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            r = time_cpu_path(args.cpu_seconds, cores)
            line["cpu_baseline"] = {
                "value": r["env_steps_per_s"] * S, "unit": UNIT, "cores": cores, "kind": r["kind"],
                "sample": _cpu_sample_text(r), "c_oracle_1core": time_c_oracle(2.0) * S,
            }
            inproc = time_reference_inprocess(2.0)
            if inproc is not None:
                line["cpu_baseline"]["reference_inprocess_1core"] = inproc * S
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--action-batches", type=int, default=32,
                    help="distinct pre-sampled action batches cycled by the timed steps (each N*S bytes, resident in HBM)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the secondary BASELINE configurations")
    ap.add_argument("--collective", action="store_true", help="run the per-step statistics all-reduce even on one GPU")
    ap.add_argument("--no-collective", action="store_true", help="A/B: multi-GPU run without the in-loop all-reduce")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"],
                    help="form of the per-step statistics reduction: fused peer-memory pushes (default) or ncclAllReduce on a side stream")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0's envs) into DIR as float32 .npy files")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to this repo's CUDA path only")
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # launched without torchrun: re-exec under it, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
