"""TEST INFRASTRUCTURE (pixel oracle harness).  Not imported by the product.

Builds the draw list of one observation from a host-side world object -- either the
UNMODIFIED reference env (oracle/ref_stub.py) or the package's host mirror -- exactly as the
reference submits it to OpenGL (Room._render miniworld.py:401-434, Box.render
entity.py:409-432 + drawBox opengl.py:460-503, MeshEnt.render entity.py:150-161), and hands
it to oracle/softgl.c.  Float conventions: whatever the reference passes through
glVertex3f / glTexCoord2f / glNormal3f / glColor3f is rounded to float32 here; model
transforms (glTranslatef / glRotatef / glScalef) are applied in float32, one rounding per
operation, in the order documented in DESIGN.md.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "libsoftgl.so")
f32 = np.float32


def build():
    subprocess.check_call(["make", "-s", "-C", HERE, "_build/libsoftgl.so"])
    return LIB


class _Scene(C.Structure):
    _fields_ = [("pos", C.c_double * 3), ("dir", C.c_double), ("cam_height", C.c_double),
                ("cam_fwd_disp", C.c_double), ("cam_pitch", C.c_double), ("cam_fov_y", C.c_double),
                ("sky", C.c_double * 3), ("light_pos", C.c_double * 3), ("light_color", C.c_double * 3),
                ("light_ambient", C.c_double * 3), ("width", C.c_int), ("height", C.c_int), ("samples", C.c_int),
                ("num_tris", C.c_int), ("tri_pos", C.c_void_p), ("tri_nrm", C.c_void_p), ("tri_uv", C.c_void_p),
                ("tri_rgb", C.c_void_p), ("tri_tex", C.c_void_p),
                ("view", C.c_int), ("ortho", C.c_double * 4), ("tri_query", C.c_void_p), ("query_out", C.c_void_p),
                ("cam_mode", C.c_int), ("eye", C.c_double * 3), ("center", C.c_double * 3), ("up", C.c_double * 3),
                ("fovy", C.c_double), ("aspect", C.c_double), ("znear", C.c_double), ("zfar", C.c_double),
                ("light_w", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            build()
        _lib = C.CDLL(LIB)
        _lib.softgl_textures_create.restype = C.c_void_p
        _lib.softgl_textures_create.argtypes = [C.c_int]
        _lib.softgl_textures_set.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        _lib.softgl_textures_destroy.argtypes = [C.c_void_p]
        _lib.softgl_render.argtypes = [C.POINTER(_Scene), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return _lib


class TextureSet:
    """name/variant -> oracle texture index; texels come from PNG-order RGB8 arrays."""

    def __init__(self, textures):
        """textures: list of uint8[H, W, 3] arrays (top row first), index = oracle texture id."""
        self.n = len(textures)
        self.h = lib().softgl_textures_create(self.n)
        for i, t in enumerate(textures):
            t = np.ascontiguousarray(t[..., :3], np.uint8)
            lib().softgl_textures_set(self.h, i, t.shape[1], t.shape[0], t.ctypes.data)

    def close(self):
        if self.h:
            lib().softgl_textures_destroy(self.h)
            self.h = None


def _fan(n):
    return [(0, k, k + 1) for k in range(1, n - 1)]


def _box_faces(sx, sy, sz):
    """drawBox(x_min=-sx/2, x_max=+sx/2, y_min=0, y_max=sy, ...) vertex order (opengl.py:460-503)."""
    x0, x1, y0, y1, z0, z1 = f32(-sx / 2), f32(sx / 2), f32(0), f32(sy), f32(-sz / 2), f32(sz / 2)
    return [
        ((0, 0, 1), [(x1, y1, z1), (x0, y1, z1), (x0, y0, z1), (x1, y0, z1)]),
        ((0, 0, -1), [(x0, y1, z0), (x1, y1, z0), (x1, y0, z0), (x0, y0, z0)]),
        ((-1, 0, 0), [(x0, y1, z1), (x0, y1, z0), (x0, y0, z0), (x0, y0, z1)]),
        ((1, 0, 0), [(x1, y1, z0), (x1, y1, z1), (x1, y0, z1), (x1, y0, z0)]),
        ((0, 1, 0), [(x1, y1, z1), (x1, y1, z0), (x0, y1, z0), (x0, y1, z1)]),
        ((0, -1, 0), [(x1, y0, z0), (x1, y0, z1), (x0, y0, z1), (x0, y0, z0)]),
    ]


def _rot_cs(deg):
    """glRotatef's angle is a GLfloat: the degrees the reference computes in float64 reach GL rounded to float32.
    Spec: c, s = float32(cos / sin(float64(angle_f32) * pi / 180))."""
    rad = float(f32(deg)) * math.pi / 180
    return f32(math.cos(rad)), f32(math.sin(rad))


def _rot_y(v, c, s):
    """glRotatef(theta, 0, 1, 0) on a float32 vector, one rounding per op: x' = x c + z s,
    z' = z c - x s."""
    x, y, z = (f32(a) for a in v)
    return (f32(f32(x * c) + f32(z * s)), y, f32(f32(z * c) - f32(x * s)))


def draw_list(env, tex_index, agent_marker=False, rooms_only=False):
    """Triangles of one frame in submission order.  tex_index(texture_object) -> oracle id.
    agent_marker: append Agent.render()'s triangle (top view, entity.py:518-539); rooms_only: stop after
    the rooms (get_visible_ents draws no entity, only their query boxes)."""
    P, Nn, UV, RGB, TX = [], [], [], [], []
    last_normal = [(0.0, 1.0, 0.0)]      # GL's "current normal": what the latest glNormal3f / array draw left behind

    def emit(verts, normals, uvs, color, tex):
        last_normal[0] = tuple(float(v) for v in normals[-1])
        for a, b, c in _fan(len(verts)):
            P.append([verts[a], verts[b], verts[c]])
            Nn.append([normals[a], normals[b], normals[c]])
            UV.append([uvs[a], uvs[b], uvs[c]])
            RGB.append([color, color, color])
            TX.append(tex)

    white = (1.0, 1.0, 1.0)
    for r in env.rooms:
        n = len(r.floor_verts)
        emit([tuple(v) for v in r.floor_verts], [(0, 1, 0)] * n, [tuple(t) for t in r.floor_texcs], white,
             tex_index(r.floor_tex))
        if not r.no_ceiling:
            emit([tuple(v) for v in r.ceil_verts], [(0, -1, 0)] * n, [tuple(t) for t in r.ceil_texcs], white,
                 tex_index(r.ceil_tex))
        for q in range(len(r.wall_verts) // 4):
            sl = slice(4 * q, 4 * q + 4)
            emit([tuple(v) for v in r.wall_verts[sl]], [tuple(v) for v in r.wall_norms[sl]],
                 [tuple(t) for t in r.wall_texcs[sl]], white, tex_index(r.wall_tex))

    def draw_entity(ent):
        kind = type(ent).__name__
        if kind == "Box":
            c, s = _rot_cs(ent.dir * (180 / math.pi))             # entity.py:421
            t = [f32(v) for v in ent.pos]
            sx, sy, sz = ent.size
            col = tuple(float(v) for v in ent.color_vec)
            for nrm, quad in _box_faces(sx, sy, sz):
                vs = []
                for v in quad:
                    rx, ry, rz = _rot_y(v, c, s)
                    vs.append((f32(rx + t[0]), f32(ry + t[1]), f32(rz + t[2])))
                nn = _rot_y(nrm, c, s)
                emit(vs, [nn] * 4, [(0.0, 0.0)] * 4, col, -1)
            last_normal[0] = (0.0, -1.0, 0.0)     # glNormal3f of drawBox's last face, object space
        elif hasattr(ent, "mesh"):
            # glTranslatef(pos) glScalef(s, s, s) glRotatef(dir): v' = pos + s * (R v); the normal
            # goes through the inverse transpose, R n / s, and is NOT renormalised
            m = ent.mesh
            # MeshEnt.render: dir * 180 / pi (entity.py:158); ImageFrame / TextFrame: dir * (180 / pi) (:206, :316)
            c, s = _rot_cs(ent.dir * 180 / math.pi if hasattr(ent, "mesh_name") or hasattr(m, "vlists")
                           else ent.dir * (180 / math.pi))
            t = np.asarray(ent.pos, dtype=np.float32)
            sc = f32(ent.scale)
            inv = f32(f32(1.0) / sc)
            if hasattr(m, "vlists"):      # the reference's ObjMesh (arrays captured by ref_stub)
                cat = lambda key, k: np.concatenate([np.asarray(v.attrs[key], np.float32).reshape(-1, 3, k)
                                                     for v in m.vlists])
                V, Nm, Tm, Cm = cat("v3f", 3), cat("n3f", 3), cat("t2f", 2), cat("c3f", 3)
                tri_tex = np.full(len(V), -1, np.int32)      # textured reference meshes: not wired up here
            else:                         # the package's host mirror (assets.ObjMesh / quad frames)
                V, Nm, Tm, Cm = m.verts, m.norms, m.texcs, m.colors
                tri_tex = m.tri_tex           # engine texture ids == oracle ids (same registry order)
            x, y, z = V[..., 0], V[..., 1], V[..., 2]
            wx = (x * c + z * s) * sc + t[0]
            wy = y * sc + t[1]
            wz = (z * c - x * s) * sc + t[2]
            nx = (Nm[..., 0] * c + Nm[..., 2] * s) * inv
            ny = Nm[..., 1] * inv
            nz = (Nm[..., 2] * c - Nm[..., 0] * s) * inv
            F = V.shape[0]
            P.extend(np.stack([wx, wy, wz], axis=-1).astype(np.float32))
            Nn.extend(np.stack([nx, ny, nz], axis=-1).astype(np.float32))
            UV.extend(np.asarray(Tm, np.float32))
            RGB.extend(np.asarray(Cm, np.float32))
            TX.extend(int(v) for v in tri_tex)
            last_normal[0] = tuple(float(v) for v in np.asarray(Nm, np.float32).reshape(-1, 3)[-1])   # object space

    # display list first (static entities), then the dynamic ones, both in list order
    if not rooms_only:
        for ent in env.entities:
            if ent.is_static and ent is not env.agent:
                draw_entity(ent)
        for ent in env.entities:
            if not ent.is_static and ent is not env.agent:
                draw_entity(ent)
    if agent_marker:
        # Agent.render(): float64 numpy arithmetic, glVertex3f rounds; red, untextured, lit with the
        # current normal (never set by the reference here: a state leak from the previous draw)
        a = env.agent
        dirv = np.array([math.cos(a.dir), 0.0, -math.sin(a.dir)])
        right = np.array([math.sin(a.dir), 0.0, math.cos(a.dir)])
        p = np.asarray(a.pos, np.float64) + np.array([0.0, 1.0, 0.0]) * a.height
        dv, rv = dirv * a.radius, right * a.radius
        p0, p1, p2 = p + dv, p + 0.75 * (rv - dv), p + 0.75 * (-rv - dv)
        tri = [tuple(f32(v) for v in q) for q in (p0, p2, p1)]
        n = last_normal[0]
        P.append(tri)
        Nn.append([n, n, n])
        UV.append([(0.0, 0.0)] * 3)
        RGB.append([(1.0, 0.0, 0.0)] * 3)
        TX.append(-1)
    T = len(P)
    return (np.asarray(P, np.float32).reshape(T, 3, 3), np.asarray(Nn, np.float32).reshape(T, 3, 3),
            np.asarray(UV, np.float32).reshape(T, 3, 2), np.asarray(RGB, np.float32).reshape(T, 3, 3),
            np.asarray(TX, np.int32))


def _query_boxes(env):
    """get_visible_ents' drawBox(pos -/+ 0.1, pos.y .. pos.y + 0.2) per entity except the agent, world space
    (miniworld.py:1299-1314): (triangles float32[12 Q, 3, 3], query id per triangle, entity per query)."""
    tris, qid, ents = [], [], []
    for ent in env.entities:
        if ent is env.agent:
            continue
        q = len(ents)
        ents.append(ent)
        pos = ent.pos
        x0, x1 = f32(pos[0] - 0.1), f32(pos[0] + 0.1)
        y0, y1 = f32(pos[1]), f32(pos[1] + 0.2)
        z0, z1 = f32(pos[2] - 0.1), f32(pos[2] + 0.1)
        faces = [[(x1, y1, z1), (x0, y1, z1), (x0, y0, z1), (x1, y0, z1)], [(x0, y1, z0), (x1, y1, z0), (x1, y0, z0), (x0, y0, z0)],
                 [(x0, y1, z1), (x0, y1, z0), (x0, y0, z0), (x0, y0, z1)], [(x1, y1, z0), (x1, y1, z1), (x1, y0, z1), (x1, y0, z0)],
                 [(x1, y1, z1), (x1, y1, z0), (x0, y1, z0), (x0, y1, z1)], [(x1, y0, z0), (x1, y0, z1), (x0, y0, z1), (x0, y0, z0)]]
        for quad in faces:
            for a, b, c in _fan(4):
                tris.append([quad[a], quad[b], quad[c]])
                qid.append(q)
    return np.asarray(tris, np.float32).reshape(-1, 3, 3), np.asarray(qid, np.int32), ents


def visible_ents(env, texset, tex_index, width=80, height=60, samples=8):
    """Oracle of MiniWorldEnv.get_visible_ents: the set of entities whose occlusion query passes."""
    pos, nrm, uv, rgb, tx = draw_list(env, tex_index, rooms_only=True)
    bpos, qid, ents = _query_boxes(env)
    nb = len(qid)
    if nb == 0:
        return set()
    query = np.concatenate([np.full(len(tx), -1, np.int32), qid])
    pos = np.concatenate([pos, bpos]).astype(np.float32)
    nrm = np.concatenate([nrm, np.tile(np.float32([0, 1, 0]), (nb, 3, 1))]).astype(np.float32)
    uv = np.concatenate([uv, np.zeros((nb, 3, 2), np.float32)]).astype(np.float32)
    rgb = np.concatenate([rgb, np.ones((nb, 3, 3), np.float32)]).astype(np.float32)
    tx = np.concatenate([tx, np.full(nb, -1, np.int32)]).astype(np.int32)
    flags = np.zeros(len(ents), np.uint8)
    _run(env, texset, (pos, nrm, uv, rgb, tx), width, height, samples, query=query, query_out=flags)
    return {e for e, f in zip(ents, flags) if f}


def top_view_extents(env, fb_width, fb_height):
    """(min_x, max_x, min_z, max_z) of render_top_view after the aspect adjustment (miniworld.py:1109-1133)."""
    min_x, max_x, min_z, max_z = env.min_x - 1, env.max_x + 1, env.min_z - 1, env.max_z + 1
    width, height = max_x - min_x, max_z - min_z
    aspect, fb_aspect = width / height, fb_width / fb_height
    if aspect > fb_aspect:
        h_diff = width / fb_aspect - height
        min_z -= h_diff / 2
        max_z += h_diff / 2
    elif aspect < fb_aspect:
        w_diff = height * fb_aspect - width
        min_x -= w_diff / 2
        max_x += w_diff / 2
    return float(min_x), float(max_x), float(min_z), float(max_z)


def render_top_view(env, texset, tex_index, width=80, height=60, samples=8, render_agent=True):
    """Oracle of MiniWorldEnv.render_top_view: rgb u8[H, W, 3]."""
    lst = draw_list(env, tex_index, agent_marker=render_agent)
    x0, x1, z0, z1 = top_view_extents(env, width, height)
    return _run(env, texset, lst, width, height, samples, ortho=(x0, x1, -z1, -z0))[0]


def render(env, texset, tex_index, width=80, height=60, samples=8, want_codes=False):
    """Oracle observation of `env` (reference env or host mirror): (rgb u8[H,W,3], depth f32[H,W,1])."""
    return _run(env, texset, draw_list(env, tex_index), width, height, samples, want_codes=want_codes)


def light_position(env):
    """The four GLfloats of GL_LIGHT0's position as the reference passes them."""
    # glLightfv(GL_LIGHT0, GL_POSITION, (GLfloat * 4)(*self.light_pos + [1])) (miniworld.py:1031), restated
    # literally: light_pos is an ndarray (params.py:45-46), so `+ [1]` adds 1 to each component, three GLfloats are
    # passed and w stays 0 -- a DIRECTIONAL light along light_pos + 1.  (A plain list would give a positional light.)
    lp = list(env.light_pos + [1])
    return [float(f32(v)) for v in lp] + [0.0] * (4 - len(lp))


def _run(env, texset, lst, width, height, samples, want_codes=False, ortho=None, query=None, query_out=None):
    pos, nrm, uv, rgb, tx = lst
    sc = _Scene()
    if ortho is not None:
        sc.view = 1
        for k in range(4):
            sc.ortho[k] = float(ortho[k])
    if query is not None:
        sc.tri_query, sc.query_out = query.ctypes.data, query_out.ctypes.data
    a = env.agent
    for k in range(3):
        sc.pos[k] = float(a.pos[k])
        sc.sky[k] = float(env.sky_color[k])
        sc.light_color[k] = float(env.light_color[k])
        sc.light_ambient[k] = float(env.light_ambient[k])
    lp = light_position(env)
    for k in range(3):
        sc.light_pos[k] = lp[k]
    sc.light_w = lp[3]
    sc.dir = float(a.dir)
    sc.cam_height, sc.cam_fwd_disp = float(a.cam_height), float(getattr(a, "cam_fwd_disp", 0.0))
    sc.cam_pitch, sc.cam_fov_y = float(a.cam_pitch), float(a.cam_fov_y)
    sc.width, sc.height, sc.samples = width, height, samples
    sc.num_tris = len(tx)
    sc.tri_pos, sc.tri_nrm, sc.tri_uv = pos.ctypes.data, nrm.ctypes.data, uv.ctypes.data
    sc.tri_rgb, sc.tri_tex = rgb.ctypes.data, tx.ctypes.data
    out = np.zeros((height, width, 3), np.uint8)
    depth = np.zeros((height, width, 1), np.float32)
    codes = np.zeros((height, width), np.uint16)
    rc = lib().softgl_render(C.byref(sc), texset.h, out.ctypes.data, depth.ctypes.data, codes.ctypes.data)
    assert rc == 0
    return (out, depth, codes) if want_codes else (out, depth)


_TOP_VIEW_MATRIX = (1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, -1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0)


def run_stream(cam, texset, lst, width, height, samples, query=None, query_out=None):
    """Rasterise one frame recorded from the reference's GL stream (oracle/gl_record.py): `cam` carries the
    glClearColor / glLightfv / gluPerspective|glOrtho / gluLookAt|glLoadMatrixf arguments, `lst` the world-space
    triangles.  Returns (rgb u8[H,W,3], depth f32[H,W,1] for near / far = 0.04 / 100, codes u16[H,W])."""
    pos, nrm, uv, rgb, tx = (np.ascontiguousarray(a) for a in lst)
    sc = _Scene()
    proj, view = cam["proj"], cam["view"]
    if proj is None:                       # nothing was drawn: only the clear colour matters
        proj, view = ("perspective", 60.0, width / height, 0.04, 100.0), ("lookat", 0, 0, 0, 1, 0, 0, 0, 1, 0)
    if proj[0] == "perspective" and view[0] == "lookat":
        sc.cam_mode = 1
        sc.fovy, sc.aspect, sc.znear, sc.zfar = proj[1:5]
        for k in range(3):
            sc.eye[k], sc.center[k], sc.up[k] = view[1 + k], view[4 + k], view[7 + k]
    elif proj[0] == "ortho" and view[0] == "loadmatrix":
        if tuple(view[1:]) != _TOP_VIEW_MATRIX or proj[5:] != (-100.0, 100.0):
            raise NotImplementedError("ortho view other than render_top_view's")
        sc.view = 1
        for k in range(4):
            sc.ortho[k] = proj[1 + k]
    else:
        raise NotImplementedError("camera %r / %r" % (proj[0], view[0]))
    light = cam["light"]
    for k in range(3):
        sc.sky[k] = float(cam["clear"][k])
        if light is not None:
            sc.light_pos[k] = float(light["position"][k])
            sc.light_color[k] = float(light["diffuse"][k])
            sc.light_ambient[k] = float(light["ambient"][k])
    sc.light_w = 1.0 if light is None else float(light["position"][3])
    if query is not None:
        sc.tri_query, sc.query_out = query.ctypes.data, query_out.ctypes.data
    sc.width, sc.height, sc.samples = width, height, samples
    sc.num_tris = len(tx)
    sc.tri_pos, sc.tri_nrm, sc.tri_uv = pos.ctypes.data, nrm.ctypes.data, uv.ctypes.data
    sc.tri_rgb, sc.tri_tex = rgb.ctypes.data, tx.ctypes.data
    out = np.zeros((height, width, 3), np.uint8)
    depth = np.zeros((height, width, 1), np.float32)
    codes = np.zeros((height, width), np.uint16)
    rc = lib().softgl_render(C.byref(sc), texset.h, out.ctypes.data, depth.ctypes.data, codes.ctypes.data)
    assert rc == 0
    return out, depth, codes
