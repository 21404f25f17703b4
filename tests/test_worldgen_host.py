"""Host-side world generation (miniworld_b200.world / envs) against the reference's, stored as golden fixtures."""
import numpy as np
import pytest

from miniworld_b200.envs import LEVELS
from conftest import golden
from helpers import CASES


@pytest.mark.parametrize("name", sorted(CASES))
def test_reset_matches_reference_golden(name):
    level, dr = CASES[name]
    g = golden(name)
    env = LEVELS[level](device=None, **({"domain_rand": True} if dr else {}))    # (Sign fixes domain_rand itself)
    n = min(g["pos"].shape[1], 4 if "maze_dr" in name else 12)
    for i in range(n):
        env.reset(seed=1000 + i)
        assert np.array_equal(env.agent.pos, g["pos"][0, i])
        assert env.agent.dir == g["dir"][0, i]
        assert len(env.entities) == g["n_ents"][0, i]
        for e, ent in enumerate(env.entities):
            assert np.array_equal(np.asarray(ent.pos, float), g["ent_pos"][0, i, e])
            assert float(ent.radius) == g["ent_radius"][0, i, e]
        assert np.array_equal(env.sky_color, g["sky_color"][0, i])
        assert np.array_equal(env.light_pos, g["light_pos"][0, i])
        a = env.agent
        assert [a.cam_height, a.cam_fwd_disp, a.cam_pitch, a.cam_fov_y] == list(g["cam"][0, i])
        if i == 0:
            assert np.array_equal(np.asarray(env.wall_segs), g["wall_segs0"])


def test_live_reference_world_generation():
    """reset(seed) of the reference levels (tests/golden/worldgen_reference.npz, oracle/gen_mirror_golden.py) vs this
    package: entity poses and radii (value and Python type), wall segments, room geometry and the next draw of
    np_random."""
    import os
    from conftest import GOLDEN
    from oracle.gen_mirror_golden import WORLDGEN_CASES, WORLDGEN_SEEDS
    with np.load(os.path.join(GOLDEN, "worldgen_reference.npz")) as z:
        ref = {k: z[k] for k in z.files}

    def take(key, n):
        """The next n rows of ref[key]."""
        at = cursor.get(key, 0)
        cursor[key] = at + n
        return ref[key][at:at + n]

    cursor, j, r = {}, 0, 0
    for eid, kw in WORLDGEN_CASES:
        mine = LEVELS[eid](device=None, **kw)
        for seed in WORLDGEN_SEEDS:
            mine.reset(seed=seed)
            n = int(ref["n_ents"][j])
            assert len(mine.entities) == n, (eid, kw, seed)
            pos, dirs, radius, rtype = take("ent_pos", n), take("ent_dir", n), take("ent_radius", n), take("ent_radius_type", n)
            for e, b in enumerate(mine.entities):
                assert np.array_equal(pos[e], np.asarray(b.pos, float)) and dirs[e] == b.dir
                assert radius[e] == b.radius and rtype[e] == type(b.radius).__name__
            assert np.array_equal(take("wall_segs", int(ref["n_wall_segs"][j])), mine.wall_segs)
            assert len(mine.rooms) == ref["n_rooms"][j]
            for rb in mine.rooms:
                for a, rows in zip(("wall_verts", "wall_texcs", "floor_texcs", "wall_norms"), ref["n_room_rows"][r]):
                    assert np.array_equal(take(a, int(rows)), getattr(rb, a)), (eid, kw, seed, a)
                r += 1
            assert ref["next_random"][j] == mine.np_random.random()
            j += 1


@pytest.mark.parametrize("name", ["fourrooms", "hallway", "mazes3"])
def test_host_move_and_turn_follow_reference(name):
    """MiniWorldEnv.move_agent / turn_agent (host-side mirrors of miniworld.py:620-668, for level code and scripts)
    reproduce the reference trajectory bit for bit up to the first episode end."""
    level, dr = CASES[name]
    g = golden(name)
    env = LEVELS[level](device=None)
    fwd = env.params.sample(None, "forward_step")
    drift = env.params.sample(None, "forward_drift")
    turn = env.params.sample(None, "turn_step")
    for i in range(4):
        env.reset(seed=1000 + i)
        moved = 0
        for t in range(g["actions"].shape[0]):
            if g["terminated"][t, i] or g["truncated"][t, i]:
                break
            a = int(g["actions"][t, i])
            if a == 0:
                env.turn_agent(turn)
            elif a == 1:
                env.turn_agent(-turn)
            elif a == 2:
                moved += bool(env.move_agent(fwd, drift))
            assert np.array_equal(env.agent.pos, g["pos"][t + 1, i]) and env.agent.dir == g["dir"][t + 1, i], (name, i, t)
        assert moved > 0


def test_levels_pickle_like_the_reference():
    """reference tests/test_miniworld.py:157-171: every level survives pickle (EzPickle: constructor arguments) and
    the copy generates the same world from the same seed."""
    import pickle
    for eid, cls in LEVELS.items():
        if "Maze-v0" in eid or "MazeS8" in eid:
            continue
        env = cls(device=None)
        twin = pickle.loads(pickle.dumps(env))
        assert type(twin) is type(env) and twin.max_episode_steps == env.max_episode_steps
        env.reset(seed=5)
        twin.reset(seed=5)
        assert np.array_equal(env.agent.pos, twin.agent.pos) and env.agent.dir == twin.agent.dir, eid
        assert len(env.entities) == len(twin.entities)
