"""Pixel parity pinned to the reference's own GL stream.

(1) The UNMODIFIED reference, run under the recording fixed-function GL (oracle/gl_record.py), returned frames from
    its render_obs() / render_depth() / render_top_view() / render() and sets from get_visible_ents() -- the
    rasterised stream of the GL calls it made.  oracle/gen_mirror_golden.py stored, for each of those frames, the
    reference's dynamic state and a digest of what it returned (tests/golden/mirror_frames.npz); here the package's
    mirror objects are put into each stored state and oracle/softgl.py's rendering of them must equal the reference's
    frame bit for bit.  All 23 reference ids (+ the MazeS8 alias), with and without domain randomisation.
(2) The kernels' arithmetic compiled for the CPU (tests/hostsim) replays the golden trajectories and is compared with
    the committed frames the reference returned (tests/golden/stream_*.npz).
The same comparison through libmwb.so on a B200 is tests/test_gpu_stream.py.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from helpers import stream_cases, stream_parity
from oracle import softgl
from oracle.stream_check import Mirror, frame_digest, load_frames, replay


@pytest.fixture(scope="module")
def recorded():
    with np.load(os.path.join(GOLDEN, "mirror_frames.npz")) as z:
        return {k: z[k] for k in z.files}


def _levels():
    from oracle.stream_check import level_ids
    return level_ids()


@pytest.mark.parametrize("level", _levels())
def test_reference_gl_stream_equals_mirror(softgl_lib, recorded, level):
    for dr in (False, True):
        if dr and level == "MiniWorld-Sign-v0":
            continue                                  # Sign fixes domain_rand=False itself (sign.py:88-93)
        m = Mirror(level, dr)
        n = bad = dbad = 0
        for f in replay(m, load_frames(recorded, "stream %s %d" % (level, dr))):
            rgb, depth = m.mirror_frame()
            n += 1
            bad += not np.array_equal(frame_digest(rgb), f["digest"][0])
            dbad += not np.array_equal(frame_digest(depth), f["digest"][1])
        assert n == 13 and bad == 0 and dbad == 0, "%s dr=%d: %d / %d frames differ, %d depth maps differ" % (
            level, dr, bad, n, dbad)


@pytest.mark.parametrize("level", ["MiniWorld-Hallway-v0", "MiniWorld-PickupObjects-v0", "MiniWorld-ThreeRooms-v0",
                                   "MiniWorld-Sidewalk-v0", "MiniWorld-Sign-v0"])
def test_reference_other_views_equal_mirror(softgl_lib, recorded, level):
    """render_top_view (with the agent marker and its leaked normal), get_visible_ents, a 160 x 120 observation."""
    m = Mirror(level, False, obs_width=160, obs_height=120)
    frames = load_frames(recorded, "views %s" % level)
    assert frames
    for f in replay(m, frames):
        assert np.array_equal(frame_digest(m.mirror_frame(160, 120)[0]), f["digest"][0])
        assert np.array_equal(frame_digest(m.mirror_top_view(160, 120)), f["digest"][1])
        assert sum(1 << e for e in m.mirror_visible(160, 120)) == f["vis"]


def test_reference_human_view_is_16_samples_and_equals_mirror(softgl_lib, recorded):
    """render() with render_mode="rgb_array": the reference's vis_fb = FrameBuffer(window_width, window_height, 16)
    (miniworld.py:518); under the recording GL (GL_MAX_SAMPLES = 16) the frame it returns is a 16-sample frame and
    equals the mirror rendered with the D3D 16-sample pattern -- agent view and map view."""
    for view in ("agent", "top"):
        assert recorded["human_%s_samples" % view] == 16
        m = Mirror("MiniWorld-Hallway-v0", False, render_mode="rgb_array", window_width=160, window_height=120, view=view)
        for f in replay(m, load_frames(recorded, "human %s" % view)):
            want = m.mirror_frame(160, 120, 16)[0] if view == "agent" else m.mirror_top_view(160, 120, 16)
            assert want.shape == (120, 160, 3)
            assert np.array_equal(frame_digest(want), f["digest"][0]), view


def test_reference_own_render_test_holds_on_the_recorded_stream(softgl_lib, recorded):
    """The one pixel-level statement the reference's test suite makes (tests/test_miniworld.py:17-38, Hallway,
    render_mode="rgb_array"): 0 < mean(obs) < 255, |mean(80x60 observation) - mean(800x600 human view)| < 5, and the
    observation shapes -- evaluated on what the unmodified reference returned under the recording GL, which the mirror
    reproduces bit for bit."""
    m = Mirror("MiniWorld-Hallway-v0", False, render_mode="rgb_array")
    frames = load_frames(recorded, "render_test")
    assert len(frames) == 2 and (recorded["render_test_samples"] == 16).all()
    for f, second_shape in zip(replay(m, frames), recorded["render_test_second_obs_shape"]):
        first_obs, first_render = m.mirror_frame()[0], m.mirror_frame(800, 600, 16)[0]
        assert np.array_equal(frame_digest(first_obs), f["digest"][0])
        assert np.array_equal(frame_digest(first_render), f["digest"][1])
        assert first_render.shape == (600, 800, 3)
        m0, m1 = first_obs.mean(), first_render.mean()
        assert 0 < m0 < 255
        assert abs(m0 - m1) < 5, (m0, m1)
        space = tuple(recorded["render_test_observation_space_shape"])
        assert first_obs.shape == space == m.mir.observation_space.shape == tuple(second_shape)


def test_reference_light_is_directional():
    """(GLfloat * 4)(*self.light_pos + [1]) with an ndarray light_pos passes THREE values, each + 1, and leaves w = 0
    (miniworld.py:1031, params.py:45-46): LIGHT0 is a directional light along light_pos + 1.  The reference's recorded
    glLightfv position after reset(seed=3) of OneRoom is what the pixel oracle passes for the mirror."""
    want = np.load(os.path.join(GOLDEN, "mirror_frames.npz"))["light_position_oneroom_seed3"]
    assert np.array_equal(want, np.array([1.0, 3.5, 1.0, 0.0], np.float32))
    m = Mirror("MiniWorld-OneRoom-v0", False)
    m.reset_mirror(3)
    assert isinstance(m.mir.light_pos, np.ndarray)
    assert softgl.light_position(m.mir) == list(want)


@pytest.mark.parametrize("name", stream_cases())
def test_hostsim_matches_reference_stream_frames(hostsim_path, name):
    # (the CPU build of the kernels is slow on mesh levels: fewer rows there; the GPU test replays every row)
    rows = {"maze_dr": 21, "pickup_160": 3, "pickup": 34, "pickup_dr": 34}.get(name, 89)
    st = stream_parity(name, hostsim_path, max_rows=rows)
    assert st["frames"] >= 4 and st["same"] / st["total"] > 0.995
    assert st["cams"] > 0 and st["cam_exact"] / st["cams"] > 0.98
