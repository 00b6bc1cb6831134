"""Generate tests/golden/maze_real_textures_golden.npz by RUNNING THE UNMODIFIED REFERENCE with its own PNG textures
(build container only).

    python tests/golden/gen_maze_real_textures.py

Every other maze fixture renders the procedural textures of metagym_b200.textures.  This one keeps the reference's
img/ set (stored here as the uint8 arrays its loader produces), one 15x15 SURVIVAL task from the reference sampler
(random.seed(5); numpy.random.seed(5)) and a 60-step random walk at 128x128.  Every frame is recorded by its SHA-256
(int32 pixels, C order) so that the whole episode is pinned bit for bit within the fixture size budget; every tenth
frame is also stored whole as uint16 so that a mismatch can be shown pixel by pixel.
"""
import hashlib
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import _refload  # noqa: E402
from gen_maze import task_arrays  # noqa: E402
from metagym_b200.textures import load_texture_dir  # noqa: E402

STEPS = 60
KEEP_EVERY = 10


def frame_digest(obs):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(obs, dtype=np.int32).tobytes()).digest(), dtype=np.uint8)


def main():
    ns = _refload.load_reference()
    grounds, ceil = load_texture_dir(os.path.join(_refload.REF_ROOT, "metagym", "metamaze", "envs", "img"))
    ns.MAZE_TASK_MANAGER.grounds = grounds.astype(np.float32)
    ns.MAZE_TASK_MANAGER.ceil = ceil
    random.seed(5)
    np.random.seed(5)
    task = ns.MazeTaskSampler(n=15, allow_loops=True, crowd_ratio=0.35, food_density=0.05)
    ref = ns.MetaMazeDiscrete3D(enable_render=False, resolution=(128, 128), max_steps=500, task_type="SURVIVAL")
    ref.set_task(task)
    frames = [ref.reset()]
    acts = np.random.RandomState(0).randint(4, size=STEPS).astype(np.int32)
    rew, done = np.zeros(STEPS, np.float64), np.zeros(STEPS, np.uint8)
    for t, a in enumerate(acts):
        o, r, d, _ = ref.step(int(a))
        frames.append(o)
        rew[t], done[t] = r, d
    frames = np.stack(frames)
    assert frames.min() >= 0 and frames.max() < 1 << 16
    keep = np.arange(0, STEPS + 1, KEEP_EVERY)
    out = {"tex.grounds": grounds, "tex.ceil": ceil, "act": acts, "rew": rew, "done": done,
           "frame_sha256": np.stack([frame_digest(f) for f in frames]),
           "kept_idx": keep.astype(np.int32), "kept_frames": frames[keep].astype(np.uint16)}
    for k, v in task_arrays(task).items():
        out["task.%s" % k] = v
    path = os.path.join(HERE, "maze_real_textures_golden.npz")
    np.savez_compressed(path, **out)
    print("steps", STEPS, "dones", int(done.sum()), "reward>0", int((rew > 0).sum()), "max pixel", int(frames.max()))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
