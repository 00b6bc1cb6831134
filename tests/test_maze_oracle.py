"""CPU: pin the maze oracle (oracle/maze_oracle.c) against golden vectors recorded from the unmodified reference.
Everything here is integer / exact: grid state, done flags, float64 rewards and life, float32 2-D observations and the
int32 raycast images must match bit for bit."""
import numpy as np
import pytest

from oracle.maze_oracle import OracleMaze
from metagym_b200.textures import synthetic_textures
from util import MAZE_CASES, maze_case


def replay(case, make_env):
    env = make_env()
    env.set_task(case["task"])
    obs0 = env.reset()
    yield ("reset", -1, obs0, None, None, None)
    kept = {int(t): k for k, t in enumerate(case["obs_idx"])}
    for t, a in enumerate(case["act"]):
        obs, rew, done, info = env.step(int(a))
        yield ("step", t, obs, rew, done, (env.agent, env.life, kept.get(t)))
        if done:
            env.reset()


@pytest.fixture(scope="module")
def geom_golden():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "maze_geom_golden.npz"))


GEOM_CASES = ["g3d_surv", "g3d_esc"]      # non-default cell / wall / eye heights (tests/golden/gen_maze_geom.py)


@pytest.mark.parametrize("name", MAZE_CASES + GEOM_CASES)
def test_oracle_matches_reference_episode(maze_golden, geom_golden, name):
    c = maze_case(geom_golden if name in GEOM_CASES else maze_golden, name)
    tex = synthetic_textures(seed=0)

    def make():
        return OracleMaze(c["kind"], c["task_type"], c["max_steps"], c["view_grid"], c["resolution"], textures=tex)

    n_frames = 0
    for what, t, obs, rew, done, extra in replay(c, make):
        if what == "reset":
            assert np.array_equal(np.asarray(obs), c["reset_obs"].astype(obs.dtype))
            assert obs.dtype == (np.float32 if c["kind"] == "2D" else np.int32)
            continue
        agent, life, k = extra
        assert rew == c["rew"][t], (t, rew, c["rew"][t])
        assert done == bool(c["done"][t]), t
        assert tuple(agent) == tuple(int(x) for x in c["agent"][t]), t
        if c["task_type"] == "SURVIVAL":
            assert life == c["life"][t], t
        if k is not None:
            ref = c["obs"][k]
            if c["kind"] == "2D":
                assert obs.dtype == np.float32 and np.array_equal(obs, ref), t
            else:
                assert np.array_equal(obs, ref.astype(np.int32)), (t, int((obs != ref).sum()))
            n_frames += 1
    assert n_frames == len(c["obs_idx"])


def test_values_can_exceed_uint8(maze_golden):
    """Near-floor pixels are lit with v_screen / l_focal > 1 (ray_caster_utils.py:99,114): with a bright ground texture
    the reference's int32 image exceeds 255, which is why the engine offers an exact int32 mode next to the clamped
    uint8 one (MGB_OBS_I32 / MGB_OBS_U8)."""
    c = maze_case(maze_golden, "m3d_big")
    grounds, ceil = synthetic_textures(seed=0)
    grounds = grounds.copy()
    grounds[0] = 255
    env = OracleMaze("3D", "ESCAPE", 200, 1, (128, 128), textures=(grounds, ceil))
    env.set_task(c["task"])
    obs = env.reset()
    assert 300 < int(obs.max()) < 400


@pytest.mark.parametrize("name", ["c3d_surv", "c3d_esc", "gc3d"])
def test_continuous_maze_oracle_matches_reference(cont_golden, geom_golden, name):
    """MetaMazeContinuous3D (SURVEY.md 8f row 2): float32 positions, float64 headings, rewards, dones and every
    recorded frame of the reference episodes, bit for bit (numba/numpy typing of dynamics.py reproduced in C)."""
    from util import cont_case
    c = cont_case(geom_golden if name == "gc3d" else cont_golden, name)
    tex = synthetic_textures(seed=0)
    env = OracleMaze("C3D", c["task_type"], c["max_steps"], 1, c["resolution"], textures=tex)
    env.set_task(c["task"])
    assert np.array_equal(env.reset(), c["reset_obs"].astype(np.int32))
    kept = {int(t): k for k, t in enumerate(c["obs_idx"])}
    for t, a in enumerate(c["act"]):
        obs, rew, done, info = env.step(a)
        pos, ori = env.pose
        assert np.array_equal(pos, c["pos"][t]) and ori == c["ori"][t], t
        assert rew == c["rew"][t] and done == bool(c["done"][t]) and info["steps"] == int(c["steps"][t]), t
        assert tuple(env.agent[:2]) == tuple(int(x) for x in c["grid"][t])
        if c["task_type"] == "SURVIVAL":
            assert env.life == c["life"][t]
        if t in kept:
            assert np.array_equal(obs, c["obs"][kept[t]].astype(np.int32)), t
        if done:
            env.reset()
    assert c["done"].sum() >= 1 and (c["rew"] > 0).sum() >= 1


def test_oracle_vs_reference_real_textures():
    """The reference renderer with its own PNG textures vs the oracle, random walk at 128x128: every frame bit for bit
    (SHA-256 of the int32 pixels, whole frames kept for every tenth step), rewards and dones
    (tests/golden/gen_maze_real_textures.py)."""
    import hashlib
    import os
    from util import task_from_arrays
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "maze_real_textures_golden.npz"))
    task = task_from_arrays(g["task.walls"], g["task.texts"], g["task.food"], g["task.interval"], g["task.scalars"])
    ora = OracleMaze("3D", "SURVIVAL", 500, 1, (128, 128), textures=(g["tex.grounds"], g["tex.ceil"]))
    ora.set_task(task)
    kept = {int(t): k for k, t in enumerate(g["kept_idx"])}

    def check(t, obs):
        if t in kept:
            ref = g["kept_frames"][kept[t]].astype(np.int32)
            assert np.array_equal(obs, ref), (t, int((obs != ref).sum()))
        digest = hashlib.sha256(np.ascontiguousarray(obs, dtype=np.int32).tobytes()).digest()
        assert digest == g["frame_sha256"][t].tobytes(), t

    check(0, ora.reset())
    for t, a in enumerate(g["act"]):
        o2, r2, d2, _ = ora.step(int(a))
        check(t + 1, o2)
        assert r2 == g["rew"][t] and d2 == bool(g["done"][t]), t
    assert len(g["act"]) == 60 and (g["rew"] > 0).sum() >= 1
