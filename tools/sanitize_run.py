"""Small run over every kernel family / rule-set / form for compute-sanitizer:
    compute-sanitizer --tool memcheck  python tools/sanitize_run.py
    compute-sanitizer --tool racecheck python tools/sanitize_run.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch, snakes_b200


def run(N, steps, debug=None, scripted=False, **kw):
    env = snakes_b200.SnakeVecEnv(N, debug=debug or "", **kw)
    env.reset()
    for t in range(steps):
        env.step(env.gen_scripted_actions(t, 7) if scripted else env.gen_actions(t, 3))
    env.dump_state()
    torch.cuda.synchronize()
    env.check_errors()
    print("ok", env.launch_info()["kernel"], debug, kw, flush=True)
    return env


run(333, 40, size=19, n_snakes=2).close()
run(333, 40, "lane=ws", size=19, n_snakes=2).close()
run(333, 120, "lane=split", scripted=True, size=19, n_snakes=2).close()             # long bodies: cta_restore
run(70, 40, "epw=4", size=10, n_snakes=2).close()                                   # small-shard batches
run(200, 60, size=10, n_snakes=3, rules="cut").close()
run(200, 60, "lane=split", size=10, n_snakes=3, rules="cut").close()
run(200, 60, size=10, n_snakes=3, rules="adversarial", n_views=3).close()
run(100, 40, "force_kernel=tile", size=10, n_snakes=3, rules="adversarial").close()
run(100, 40, "force_kernel=dense", size=10, n_snakes=3, rules="cut").close()
run(40, 30, size=64, n_snakes=16, rules="cut").close()
run(60, 30, size=12, n_snakes=5, rules="classic").close()
# atari84 with more envs than resident CTAs (two-part pipeline over several envs per CTA), main-view gather, graph, scalars
env = run(1700, 6, size=19, n_snakes=2, obs_mode="atari84")
main = torch.empty((1700, 84, 84, 3), dtype=torch.uint8, device="cuda")
env.set_main_view_target(main)
env.step(env.gen_actions(50, 3))
assert torch.equal(main, env.obs[..., 0:3])
env.set_main_view_target(None)
env.close()
env = run(512, 10, size=19, n_snakes=2)
acts = torch.stack([env.gen_actions(t, 3).clone() for t in range(8)])
g = env.make_graph(acts, T=24); g.launch(); torch.cuda.synchronize(); g.close()
gs = env.make_scripted_graph(30, 0, 7); gs.launch(); torch.cuda.synchronize(); gs.close()
tk = [env.step_scalars_async(acts[t % 8].cpu().numpy()) for t in range(3)]
for k in tk:
    env.wait_scalars(k)
main = torch.empty((512, 21, 21, 3), dtype=torch.uint8, device="cuda")
env.set_main_view_target(main); env.step(acts[0]); assert torch.equal(main, env.obs[..., 0:3])
env.check_errors()
env.close()
print("all ok")
