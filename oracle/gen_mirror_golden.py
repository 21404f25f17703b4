#!/usr/bin/env python
"""TEST INFRASTRUCTURE (oracle).  Dump what the UNMODIFIED reference returns in the mirror checks of
tests/test_stream_oracle.py and tests/test_worldgen_host.py, so that those checks run without the reference.

mirror_frames.npz: for every frame a check compared, the reference's dynamic state at that moment (the entity list,
poses and step count that oracle/stream_check.Pair copies into the package mirror) and a digest of each array the
reference returned (oracle/stream_check.frame_digest), plus the few scalars the checks read (visible sets, MSAA
sample counts, means, the GL light position).  Before anything is written every record is replayed through the
mirror alone and must reproduce the reference's digests.

worldgen_reference.npz: entity poses / radii, wall segments, room geometry and the next draw of np_random after
reset(seed) of a few reference levels.

    python oracle/gen_mirror_golden.py        # needs the reference checkout (oracle/ref_stub.py)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
import miniworld_b200  # noqa: E402,F401  (the package binds its own gymnasium before ref_stub installs one)
from oracle import ref_stub, softgl  # noqa: E402
from oracle.stream_check import Mirror, Pair, frame_digest, level_ids, load_frames, pack_frames, replay  # noqa: E402

GOLDEN = os.path.join(HERE, "..", "tests", "golden")
OTHER_VIEW_LEVELS = ["MiniWorld-Hallway-v0", "MiniWorld-PickupObjects-v0", "MiniWorld-ThreeRooms-v0",
                     "MiniWorld-Sidewalk-v0", "MiniWorld-Sign-v0"]
WORLDGEN_CASES = [("MiniWorld-FourRooms-v0", {}), ("MiniWorld-FourRooms-v0", {"domain_rand": True}),
                  ("MiniWorld-PickupObjects-v0", {"domain_rand": True}), ("MiniWorld-Hallway-v0", {})]
WORLDGEN_SEEDS = (5, 6, 7)


def obs_of(obs):
    return obs["obs"] if isinstance(obs, dict) else obs


def snap(p, seed, outputs, **extra):
    idx, pos, dirs, steps = p.state()
    return dict(seed=seed, idx=idx, pos=pos, dir=dirs, steps=steps,
                digest=np.stack([frame_digest(o) for o in outputs]), **extra)


def stream_frames(level, dr, seed=1000, steps=12):
    """oracle.stream_check.compare(level, dr, steps=12): render_obs() and render_depth() of 13 frames."""
    p = Pair(level, dr)
    rng = np.random.default_rng(12345)
    obs, fresh = p.reset(seed), seed
    frames = []
    for t in range(steps + 1):
        if t > 0:
            obs, _, term, trunc, _ = p.step(int(rng.integers(0, p.ref.action_space.n)))
            if term or trunc:
                obs, fresh = p.reset(seed + t), seed + t
        frames.append(snap(p, fresh, [obs_of(obs), p.ref.render_depth()]))
        fresh = -1
    return frames


def other_view_frames(level):
    """160 x 120 observation, render_top_view() and get_visible_ents() after each of 6 random steps."""
    p = Pair(level, False, obs_width=160, obs_height=120)
    rng = np.random.default_rng(7)
    p.reset(11)
    fresh, frames = 11, []
    for t in range(6):
        obs, _, term, trunc, _ = p.step(int(rng.integers(0, p.ref.action_space.n)))
        if term or trunc:
            p.reset(12 + t)
            fresh = 12 + t
            continue
        vis = sum(1 << e for e in p.ref_visible())
        frames.append(snap(p, fresh, [obs_of(obs), p.ref.render_top_view()], vis=vis))
        fresh = -1
    return frames


def human_view_frames(view):
    """render() with render_mode="rgb_array" at 160 x 120 after reset(5) and one forward step."""
    p = Pair("MiniWorld-Hallway-v0", False, render_mode="rgb_array", window_width=160, window_height=120, view=view)
    p.reset(5)
    p.step(2)
    got = p.ref.render()
    return [snap(p, 5, [got])], ref_stub.recorder.frames[-1].samples


def own_render_test_frames():
    """The reference's tests/test_miniworld.py:17-38 on Hallway: the observation returned by reset(seed + 10) and
    the 800 x 600 human view rendered right after it."""
    p = Pair("MiniWorld-Hallway-v0", False, render_mode="rgb_array")
    frames, samples, second = [], [], []
    for seed in (0, 1):
        p.reset(seed)
        for _ in range(3):
            p.step(0)
        first_obs = p.reset(seed + 10)
        first_render = p.ref.render()
        samples.append(ref_stub.recorder.frames[-1].samples)
        frames.append(snap(p, seed + 10, [first_obs, first_render]))
        second.append(p.step(0)[0].shape)
    return frames, samples, second, p.ref.observation_space.shape


def check_replay(name, frames, outputs, **kw):
    """Replay the records through the mirror alone; outputs(mirror) must give the recorded digests."""
    level, dr = name
    m = Mirror(level, dr, **kw)
    for j, f in enumerate(replay(m, frames)):
        got = np.stack([frame_digest(o) for o in outputs(m)])
        assert np.array_equal(got, f["digest"]), "%s: frame %d of the mirror replay differs" % (name, j)


def worldgen():
    """Arrays of all (case, seed) resets concatenated; n_* give the lengths per reset (rooms: per room)."""
    cols = {k: [] for k in ("ent_pos", "ent_dir", "ent_radius", "ent_radius_type", "wall_segs", "wall_verts", "wall_texcs",
                            "floor_texcs", "wall_norms", "n_ents", "n_wall_segs", "n_rooms", "n_room_rows", "next_random")}
    for eid, kw in WORLDGEN_CASES:
        ref = ref_stub.make_reference_env(eid, **kw)
        for seed in WORLDGEN_SEEDS:
            ref.reset(seed=seed)
            cols["ent_pos"] += [np.asarray(e.pos, float) for e in ref.entities]
            cols["ent_dir"] += [float(e.dir) for e in ref.entities]
            cols["ent_radius"] += [float(e.radius) for e in ref.entities]
            cols["ent_radius_type"] += [type(e.radius).__name__ for e in ref.entities]
            cols["n_ents"].append(len(ref.entities))
            cols["wall_segs"] += list(np.asarray(ref.wall_segs, np.float64))
            cols["n_wall_segs"].append(len(ref.wall_segs))
            cols["n_rooms"].append(len(ref.rooms))
            for room in ref.rooms:
                for a in ("wall_verts", "wall_texcs", "floor_texcs", "wall_norms"):
                    cols[a] += list(np.asarray(getattr(room, a), np.float64))
                cols["n_room_rows"].append([len(getattr(room, a)) for a in ("wall_verts", "wall_texcs", "floor_texcs", "wall_norms")])
            cols["next_random"].append(ref.np_random.random())
    return {k: np.array(v) for k, v in cols.items()}


def main():
    softgl.build()
    records = {}
    for level in level_ids():
        for dr in (False, True):
            if dr and level == "MiniWorld-Sign-v0":
                continue                              # Sign fixes domain_rand=False itself (sign.py:88-93)
            frames = stream_frames(level, dr)
            check_replay((level, dr), frames, lambda m: m.mirror_frame())
            records["stream %s %d" % (level, dr)] = frames
    for level in OTHER_VIEW_LEVELS:
        frames = other_view_frames(level)
        check_replay((level, False), frames, lambda m: [m.mirror_frame(160, 120)[0], m.mirror_top_view(160, 120)],
                     obs_width=160, obs_height=120)
        records["views %s" % level] = frames
    extra = {}
    for view in ("agent", "top"):
        frames, samples = human_view_frames(view)
        draw = (lambda m: [m.mirror_frame(160, 120, 16)[0]]) if view == "agent" else (lambda m: [m.mirror_top_view(160, 120, 16)])
        check_replay(("MiniWorld-Hallway-v0", False), frames, draw, render_mode="rgb_array", window_width=160,
                     window_height=120, view=view)
        records["human %s" % view] = frames
        extra["human_%s_samples" % view] = np.array(samples)
    frames, samples, second, space = own_render_test_frames()
    check_replay(("MiniWorld-Hallway-v0", False), frames,
                 lambda m: [m.mirror_frame()[0], m.mirror_frame(800, 600, 16)[0]], render_mode="rgb_array")
    records["render_test"] = frames
    extra["render_test_samples"] = np.array(samples)
    extra["render_test_second_obs_shape"] = np.array(second)
    extra["render_test_observation_space_shape"] = np.array(space)
    env = ref_stub.make_reference_env("MiniWorld-OneRoom-v0", record=True)
    env.reset(seed=3)
    assert isinstance(env.light_pos, np.ndarray)
    extra["light_position_oneroom_seed3"] = np.asarray(ref_stub.recorder.frames[-1].light["position"], np.float32)

    path = os.path.join(GOLDEN, "mirror_frames.npz")
    np.savez_compressed(path, **pack_frames(records), **extra)
    with np.load(path) as z:                         # what is stored is what was recorded
        for name, frames in records.items():
            for f, g in zip(frames, load_frames(z, name)):
                assert all(np.array_equal(f[k], g[k]) for k in f), name
    print("%s: %d B" % (os.path.relpath(path), os.path.getsize(path)))
    path = os.path.join(GOLDEN, "worldgen_reference.npz")
    np.savez_compressed(path, **worldgen())
    print("%s: %d B" % (os.path.relpath(path), os.path.getsize(path)))


if __name__ == "__main__":
    main()
