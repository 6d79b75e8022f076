"""Shared helpers for the parity tests: golden loading, state digests, oracle runners."""
import ctypes
import glob
import json
import os
import zlib

import numpy as np

import c_oracle
import snake_oracle as so

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden_names():
    return sorted(n for n in (os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz"))) if not n.startswith("gae_"))


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    for k in ("S", "D", "F", "K", "N", "T", "cap"):
        g[k] = int(g[k])
    g["rules"] = str(g["rules"])
    return g


def known_answers():
    with open(os.path.join(GOLDEN_DIR, "known_answers.json")) as f:
        return json.load(f)


def per_env_state_crcs(st):
    """crc32 per env of the canonical arrays (same digest as snake_oracle.state_crc)."""
    N = len(st["t"])
    out = np.zeros(N, dtype=np.uint32)
    key = "fruit_grid" if "fruit_grid" in st else "fruit"
    for e in range(N):
        c = {"t": st["t"][e], "spare": st["spare"][e], "len": st["len"][e], "grow_to": st["grow_to"][e],
             "vel": st["vel"][e], "body": st["body"][e], key: st[key][e]}
        out[e] = so.state_crc(c)
    return out


def batch_state_crc(st):
    return zlib.crc32(per_env_state_crcs(st).tobytes())


def sub_tape(g, lanes):
    """CSR tape restricted to the given lanes."""
    off = g["tape_offsets"].astype(np.int64)
    vals = [g["tape_vals"][off[i]:off[i + 1]] for i in lanes]
    bounds = [g["tape_bounds"][off[i]:off[i + 1]] for i in lanes]
    o = np.zeros(len(lanes) + 1, dtype=np.uint64)
    o[1:] = np.cumsum([len(v) for v in vals])
    cat = lambda xs: np.concatenate(xs) if xs else np.zeros(0, dtype=np.uint32)
    return cat(vals).astype(np.uint32), cat(bounds).astype(np.uint32), o


def state_blob_from_lists(lay, cfg, snakes, fruits, vels, grow_to, t, spare=0):
    """A canonical state blob for N = 1 from the reference's list-of-tuples form."""
    V = cfg.size + 2
    blob = np.zeros(lay.total_bytes, dtype=np.uint8)
    st = c_oracle.split_state(blob, lay, cfg)
    vel_code = {(0, 0): 0, (1, 0): 1, (0, 1): 2, (-1, 0): 3, (0, -1): 4}
    pid = lambda c: (c[0] + 1) * V + (c[1] + 1)
    st["t"][0] = t
    st["spare"][0] = spare
    for s, b in enumerate(snakes):
        st["len"][0, s] = len(b)
        st["body"][0, s, :len(b)] = [pid(c) for c in b]
        st["grow_to"][0, s] = grow_to[s]
        st["vel"][0, s] = vel_code[tuple(vels[s])]
    if lay.fruit_is_grid:
        for f in fruits:
            st["fruit_grid"][0, pid(f)] += 1
    else:
        st["fruit"][0, :] = [pid(f) for f in fruits]
    return blob


def lists_from_state(st, cfg, e=0):
    V = cfg.size + 2
    xy = lambda p: [int(p) // V - 1, int(p) % V - 1]
    vel_xy = {0: [0, 0], 1: [1, 0], 2: [0, 1], 3: [-1, 0], 4: [0, -1]}
    snakes = [[xy(p) for p in st["body"][e, s, :int(st["len"][e, s])]] for s in range(cfg.n_snakes)]
    if "fruit" in st:
        fruits = [xy(p) for p in st["fruit"][e]]
    else:
        fruits = sorted(xy(p) for p in np.flatnonzero(st["fruit_grid"][e]) for _ in range(int(st["fruit_grid"][e][p])))
    return {"snakes": snakes, "fruits": fruits, "vels": [vel_xy[int(v)] for v in st["vel"][e]],
            "grow_to": [int(x) for x in st["grow_to"][e]], "t": int(st["t"][e]), "spare": int(st["spare"][e])}


def random_long_snake_states(lay, cfg, rng, min_len=20, max_len=70):
    """A canonical state blob with long, self-avoiding, mutually disjoint bodies (random walks):
    exercises multi-word chain codes, ring wrap-around and crowded boards from step 0."""
    N, S, F, D = cfg.num_envs, cfg.n_snakes, cfg.n_fruits, cfg.size
    V = D + 2
    blob = np.zeros(lay.total_bytes, dtype=np.uint8)
    st = c_oracle.split_state(blob, lay, cfg)
    moves = {1: (1, 0), 2: (0, 1), 3: (-1, 0), 4: (0, -1)}
    pid = lambda x, y: (x + 1) * V + (y + 1)
    for e in range(N):
        used = set()
        for s in range(S):
            for _attempt in range(50):
                x, y = int(rng.randint(D)), int(rng.randint(D))
                if (x, y) not in used:
                    break
            walk, vel = [(x, y)], 0
            seen = {(x, y)}
            target = int(rng.randint(min_len, max_len + 1))
            while len(walk) < target:
                opts = [(a, (walk[-1][0] + dx, walk[-1][1] + dy)) for a, (dx, dy) in moves.items()]
                opts = [(a, c) for a, c in opts if 0 <= c[0] < D and 0 <= c[1] < D and c not in seen and c not in used]
                if not opts:
                    break
                a, c = opts[int(rng.randint(len(opts)))]
                walk.append(c); seen.add(c); vel = a
            used |= seen
            body = walk[::-1]  # head = last cell reached
            L = len(body)
            st["len"][e, s] = L
            st["body"][e, s, :L] = [pid(cx, cy) for cx, cy in body]
            st["grow_to"][e, s] = max(3, L + int(rng.randint(0, 3)))
            st["vel"][e, s] = vel
        st["t"][e] = int(rng.randint(0, 100))
        st["ep_len"][e] = st["t"][e]
        free = [(x, y) for x in range(D) for y in range(D) if (x, y) not in used]
        for f in range(F):
            fx, fy = free[int(rng.randint(len(free)))] if free else (0, 0)
            if lay.fruit_is_grid:
                st["fruit_grid"][e, pid(fx, fy)] += 1
            else:
                st["fruit"][e, f] = pid(fx, fy)
    return blob


def tiled_long_snake_states(lay, cfg, rng, pool=256):
    """random_long_snake_states for a batch too large to walk env by env in Python: `pool` envs are drawn and env e
    takes state e % pool.  Twins part at their first draw, which is keyed by the global env id.  `cfg` / `lay`: the
    oracle's (c_oracle.Config / Layout)."""
    sub = c_oracle.Config.from_buffer_copy(cfg)
    sub.num_envs = min(pool, cfg.num_envs)
    sub_lay = c_oracle.Layout()
    c_oracle.lib().so_state_layout_of(ctypes.byref(sub), ctypes.byref(sub_lay))
    src = c_oracle.split_state(random_long_snake_states(sub_lay, sub, rng), sub_lay, sub)
    blob = np.zeros(lay.total_bytes, dtype=np.uint8)
    dst = c_oracle.split_state(blob, lay, cfg)
    idx = np.arange(cfg.num_envs) % sub.num_envs
    for k in dst:
        dst[k][...] = src[k][idx]
    return blob
