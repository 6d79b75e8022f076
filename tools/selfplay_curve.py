"""f2 evidence: one self-play PPO run with the reference's training setup (src/train_snake.py:43-50 -- nsteps 64,
nminibatches 8, noptepochs 4, lam 0.95, gamma 0.99, ent_coef 0.01, lr = f * 2.5e-4, cliprange = f * 0.1; Config.USE_ATARI_SIZE
=> WarpFrame 84x84 observations and nature_cnn, src/policies.py:42, src/utils.py:18) on the batched env, to be read against
the reference's published curve (plots/ppo_self_play_2_19x19.png: `eprewmean 100` about 20 at 1e7 steps).
obs_mode 'grid' trains the same network on cell-code grids (the nature policy's first layer reads the WarpFrame from the
codes, grid_conv84_in); the board's V = size + 2 must divide 84.

    python tools/selfplay_curve.py [n_snakes=2] [size=19] [num_envs=32] [total_timesteps=1e7] [out=gpurun_out/selfplay]
                                   [obs_mode=atari84]
    torchrun --nproc-per-node G tools/selfplay_curve.py ...     # data-parallel learner: envs sharded, gradients all-reduced
"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import snakes_b200
from snakes_b200 import selfplay

S = int(sys.argv[1]) if len(sys.argv) > 1 else 2
D = int(sys.argv[2]) if len(sys.argv) > 2 else 19
N = int(sys.argv[3]) if len(sys.argv) > 3 else 32
TOTAL = int(float(sys.argv[4])) if len(sys.argv) > 4 else int(1e7)
OUT = sys.argv[5] if len(sys.argv) > 5 else "gpurun_out/selfplay"
OBS_MODE = sys.argv[6] if len(sys.argv) > 6 else "atari84"

world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local))
torch.manual_seed(0)
torch.backends.cudnn.allow_tf32 = True
torch.backends.cuda.matmul.allow_tf32 = True
base, count = snakes_b200.shard_range(N, rank, world)
env = snakes_b200.SnakeVecEnv(count, size=D, n_snakes=S, seed=0, device=local, env_id_base=base, obs_mode=OBS_MODE)
os.makedirs(os.path.dirname(OUT) or ".", exist_ok=True)
t0 = time.time()
# total_timesteps counts the steps of THIS rank's envs, as the reference counts its own (nbatch = nenvs * nsteps)
model, log = selfplay.learn(env, nsteps=64, nminibatches=8, noptepochs=4, lam=0.95, gamma=0.99, ent_coef=0.01,
                            lr=lambda f: f * 2.5e-4, cliprange=lambda f: f * 0.1, total_timesteps=TOTAL // world,
                            log_interval=max(TOTAL // (N * 64) // 100, 1), arch="nature", csv_path=OUT + ".csv" if rank == 0 else None,
                            echo=rank == 0, seed=0)
torch.cuda.synchronize()
dt = time.time() - t0
env.check_errors()
if rank == 0:
    rows = log.rows
    summary = {"n_snakes": S, "size": D, "num_envs": N, "obs_mode": OBS_MODE, "world": world, "total_timesteps": TOTAL, "seconds": dt,
               "env_steps_per_s_incl_learner": TOTAL / dt, "final_eprewmean_100": rows[-1]["eprewmean 100"],
               "final_eplenmean": rows[-1]["eplenmean"], "best_eprewmean_100": max(r["eprewmean 100"] for r in rows),
               "curve": [[r["total_timesteps"] * world, round(r["eprewmean 100"], 3), round(r["eplenmean"], 1)] for r in rows[::max(len(rows) // 25, 1)]],
               "reference": "plots/ppo_self_play_2_19x19.png: eprewmean 100 about 20 (15-25) at 1e7 steps (SURVEY.md section 6)"}
    json.dump(summary, open(OUT + ".json", "w"), indent=1)
    print(json.dumps(summary))
env.close()
if world > 1:
    torch.distributed.destroy_process_group()
