"""TEST INFRASTRUCTURE (oracle).  Stream-driven vs mirror-driven pixel oracle.

Runs the UNMODIFIED reference under the recording GL (oracle/gl_record.py) and, beside it, the package's host
mirror of the same level / seed with the reference's dynamic state copied over each step; the reference's own
render_obs() (rasterised GL stream) must equal oracle/softgl.py's rendering of the mirror objects bit for bit.
That pins everything the mirror path restates about the reference's draw code -- geometry, attributes, transforms,
colours, normals, light, camera, texels, draw order -- to what the reference actually submits.

`Pair` needs the reference checkout (oracle/ref_stub.py); `python -m oracle.stream_check` prints a table for all
level ids.  `Mirror` alone needs only the package: oracle/gen_mirror_golden.py stores the reference's state and a
digest of every frame it returned (tests/golden/mirror_frames.npz), and the tests put the mirror back into each stored
state and compare digests.
"""
import hashlib

import numpy as np

from oracle import ref_stub, softgl


def level_ids():
    from miniworld_b200.envs import LEVELS
    return sorted(k for k in LEVELS if k != "MiniWorld-MazeS8-v0") + ["MiniWorld-MazeS8-v0"]


def reference_id(level):
    return "MiniWorld-Maze-v0" if level == "MiniWorld-MazeS8-v0" else level      # SURVEY section 8: MazeS8 == Maze (8x8)


def frame_digest(a):
    """16 bytes of SHA-256 over an array's dtype, shape and contents: equal digests <=> equal arrays."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s%r" % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return np.frombuffer(h.digest()[:16], np.uint8)


class Mirror:
    """The package's host mirror of a level, drawn by the pixel oracle.  Its dynamic state is set from outside
    (`Pair.sync` from the live reference, `set_state` from a stored record): the mirror itself is never stepped."""

    def __init__(self, level, domain_rand, **kw):
        from miniworld_b200.assets import Texture
        from miniworld_b200.envs import LEVELS
        if level != "MiniWorld-Sign-v0":           # Sign passes domain_rand=False itself (sign.py:88-93)
            kw = dict(kw, domain_rand=domain_rand)
        self.kw = kw
        self.mir = LEVELS[level](device=None, **kw)
        self.Texture = Texture
        self._ts = None
        self.base = []

    def texset(self):
        n = len(self.Texture.registry)
        if self._ts is None or self._ts.n != n:
            if self._ts is not None:
                self._ts.close()
            self._ts = softgl.TextureSet([t.texels for t in self.Texture.registry])
        return self._ts

    def reset_mirror(self, seed):
        self.mir.reset(seed=seed)
        self.base = list(self.mir.entities)

    def state(self):
        """(entity list as indices into the list reset() built, their positions, directions, step count)."""
        ents = self.mir.entities
        idx = [next(k for k, b in enumerate(self.base) if b is e) for e in ents]
        return (np.array(idx, np.int32), np.array([e.pos for e in ents], np.float64).reshape(-1, 3),
                np.array([e.dir for e in ents], np.float64), int(self.mir.step_count))

    def set_state(self, idx, pos, dir, step_count):
        ents = [self.base[k] for k in idx]
        for m, p, d in zip(ents, pos, dir):
            m.pos, m.dir = np.array(p, dtype=np.float64), float(d)
        self.mir.entities = ents
        self.mir.step_count = int(step_count)

    def mirror_frame(self, width=80, height=60, samples=8, want_codes=False):
        return softgl.render(self.mir, self.texset(), lambda tex: tex.tex_id, width, height, samples, want_codes)

    def mirror_top_view(self, width=80, height=60, samples=8):
        return softgl.render_top_view(self.mir, self.texset(), lambda tex: tex.tex_id, width, height, samples)

    def mirror_visible(self, width=80, height=60):
        vis = softgl.visible_ents(self.mir, self.texset(), lambda tex: tex.tex_id, width, height)
        return {self.mir.entities.index(e) for e in vis}


def pack_frames(records):
    """{name: recorded frames} -> flat npz arrays.  A frame is a dict: seed of the reset just before it, or -1;
    idx / pos / dir / steps as Mirror.state(); digest[K, 16] of the K arrays the reference returned; optional vis."""
    frames = [f for fs in records.values() for f in fs]
    F, E = len(frames), max(len(f["idx"]) for f in frames)
    K = max(len(f["digest"]) for f in frames)
    out = {"names": np.array(list(records)), "first": np.cumsum([0] + [len(fs) for fs in records.values()]),
           "seed": np.array([f["seed"] for f in frames], np.int64), "n": np.array([len(f["idx"]) for f in frames], np.int32),
           "idx": np.full((F, E), -1, np.int32), "pos": np.zeros((F, E, 3)), "dir": np.zeros((F, E)),
           "steps": np.array([f["steps"] for f in frames], np.int64), "digest": np.zeros((F, K, 16), np.uint8),
           "k": np.array([len(f["digest"]) for f in frames], np.int32),
           "vis": np.array([f.get("vis", -1) for f in frames], np.int64)}
    for j, f in enumerate(frames):
        n = len(f["idx"])
        out["idx"][j, :n], out["pos"][j, :n], out["dir"][j, :n] = f["idx"], f["pos"], f["dir"]
        out["digest"][j, :len(f["digest"])] = f["digest"]
    return out


def load_frames(z, name):
    """Inverse of pack_frames: the recorded frames stored under `name` in the npz `z`."""
    k = list(z["names"]).index(name)
    frames = []
    for j in range(z["first"][k], z["first"][k + 1]):
        n = z["n"][j]
        frames.append({"seed": int(z["seed"][j]), "idx": z["idx"][j, :n], "pos": z["pos"][j, :n], "dir": z["dir"][j, :n],
                       "steps": int(z["steps"][j]), "digest": z["digest"][j, :z["k"][j]], "vis": int(z["vis"][j])})
    return frames


def replay(mirror, frames):
    """Yield each recorded frame after putting `mirror` into the state the reference was in when it returned it."""
    for f in frames:
        if f["seed"] >= 0:
            mirror.reset_mirror(f["seed"])
        mirror.set_state(f["idx"], f["pos"], f["dir"], f["steps"])
        yield f


class Pair(Mirror):
    """A reference env (recording GL) and the package mirror of it, kept in the same state."""

    def __init__(self, level, domain_rand, **kw):
        super().__init__(level, domain_rand, **kw)
        self.ref = ref_stub.make_reference_env(reference_id(level), record=True, **self.kw)

    def reset(self, seed):
        ref_stub.recorder.active = True
        obs, _ = self.ref.reset(seed=seed)
        self.reset_mirror(seed)
        assert len(self.ref.entities) == len(self.mir.entities)
        self.map = {id(r): m for r, m in zip(self.ref.entities, self.mir.entities)}
        self.sync()
        return obs

    def sync(self):
        """Copy the reference's dynamic state into the mirror (poses, entity list, carried object)."""
        ents = []
        for r in self.ref.entities:
            m = self.map.get(id(r))
            if m is None:                       # an entity placed after reset (CollectHealth respawn): mirror it
                raise NotImplementedError("entity created during the episode")
            m.pos, m.dir = np.array(r.pos, dtype=np.float64), float(r.dir)
            ents.append(m)
        self.mir.entities = ents
        self.mir.step_count = self.ref.step_count

    def step(self, action):
        ref_stub.recorder.active = True
        obs, rew, term, trunc, info = self.ref.step(action)
        self.sync()
        return obs, rew, term, trunc, info

    def ref_visible(self):
        return {self.ref.entities.index(e) for e in self.ref.get_visible_ents()}


def compare(level, domain_rand, seed=1000, steps=20, verbose=False):
    """Returns (frames compared, frames that differ, worst |diff|, depth-code mismatches)."""
    p = Pair(level, domain_rand)
    rng = np.random.default_rng(12345)
    obs = p.reset(seed)
    n = bad = worst = dbad = 0
    for t in range(steps + 1):
        if t > 0:
            obs, _, term, trunc, _ = p.step(int(rng.integers(0, p.ref.action_space.n)))
            if term or trunc:
                obs = p.reset(seed + t)
        if isinstance(obs, dict):              # Sign's dict observation
            obs = obs["obs"]
        want, wdepth = p.mirror_frame()
        depth = p.ref.render_depth()
        d = np.abs(obs.astype(int) - want.astype(int))
        n += 1
        if d.max() > 0:
            bad += 1
            worst = max(worst, int(d.max()))
            if verbose:
                print("  t=%d: %d channel values differ, max %d" % (t, (d > 0).sum(), d.max()))
        if not np.array_equal(depth, wdepth):
            dbad += 1
    return n, bad, worst, dbad


if __name__ == "__main__":
    import sys
    ids = sys.argv[1:] or level_ids()
    for level in ids:
        for dr in (False, True):
            try:
                print("%-32s dr=%d  frames %d  differing %d  worst %d LSB  depth-mismatch %d" % ((level, dr) + compare(level, dr)))
            except Exception as e:      # noqa: BLE001 -- a table of what breaks is the point
                print("%-32s dr=%d  ERROR %s: %s" % (level, dr, type(e).__name__, e))
