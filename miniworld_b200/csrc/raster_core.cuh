// raster_core.cuh -- K2 arithmetic: camera, vertex pipeline, triangle setup, coverage,
// depth, shading.  The kernel that drives these functions is in raster.cuh.
//
// What is restated here (reference = Farama-Foundation/Miniworld @ c660156, the GL state it
// programs, and the OpenGL 2.1 fixed-function rules those calls select):
//   MiniWorldEnv.render_obs      miniworld.py:1177-1221  clear to sky_color / depth 1,
//                                gluPerspective(fov_y, W/H, 0.04, 100), gluLookAt(cam_pos,
//                                cam_pos + cam_dir, +Y)
//   Agent.cam_pos / cam_dir      entity.py:476-503
//   _render_static/_render_world miniworld.py:1019-1086  LIGHT0 positional at light_pos,
//                                COLOR_MATERIAL(AMBIENT_AND_DIFFUSE), SMOOTH shading,
//                                rooms -> entities in list order, DEPTH_TEST LESS, CULL_FACE
//   Room._render                 miniworld.py:401-434    floor / ceiling polygons, wall quads
//   Box.render + drawBox         entity.py:409-432, opengl.py:460-503
//   Texture.load                 opengl.py:147-184       RGB8, mipmaps, trilinear, REPEAT
//   FrameBuffer                  opengl.py:197-435       N-sample MSAA, DEPTH_COMPONENT16,
//                                box-filter resolve to unorm8, depth -> metres (:400-435)
//
// Arithmetic contract (DESIGN.md "pixel spec"): everything that decides WHICH surface a
// sample sees -- vertex transform, homogeneous edge functions, the z plane, the 16-bit
// depth code -- is float32 with one rounding per operation in a fixed order (f*_rn
// helpers; never contracted), so the CPU oracle (oracle/softgl.c) reproduces coverage and
// depth bit for bit.  Colour (lighting, perspective-correct interpolation, trilinear
// filtering, resolve) is ordinary float32 where FMA contraction is allowed; it is
// continuous in its inputs and is held to <= 1 LSB against the oracle.
#pragma once
#include "libm_sincos.cuh"
#include "state.h"

#define MWB_NEAR 0.04
#define MWB_FAR 100.0
#define MWB_MAX_LEVELS 12
#define MWB_SKY_KEY 0xFFFF0000u

struct TexDev {
  int32_t w, h, nlev, pad;
  int32_t lw[MWB_MAX_LEVELS], lh[MWB_MAX_LEVELS];
  int32_t off[MWB_MAX_LEVELS];   // texel offset of each level in the pool
  float ax[MWB_MAX_LEVELS], ay[MWB_MAX_LEVELS];   // atlas position of texel (0, 0) of each level (see RenderAssets.atlas)
};

struct MeshDev {
  int32_t first, count;          // triangle range in the mesh pool
};

struct RenderAssets {
  const TexDev* tex;
  unsigned long long atlas;      // CUDA texture object over ONE 2-D array holding every mip level of every texture, each
                                 //   with a one-texel wrapped border (so a bilinear footprint never leaves its rectangle):
                                 //   K2 reads the 2x2 footprint with tld4 through a warp-uniform handle; 0 = use the pool
  float atlas_iw, atlas_ih;      // 1 / atlas width, height (powers of two: the scaling is exact)
  const uint32_t* texels;        // RGBA8 pool, row 0 = bottom of the image
  int32_t num_tex;
  const MeshDev* meshes;
  const float* mesh_pos;         // [T][3][3]
  const float* mesh_nrm;
  const float* mesh_uv;          // [T][3][2]
  const float* mesh_rgb;
  const int32_t* mesh_tex;       // [T] texture id of each triangle's material, or -1
  int32_t num_meshes;
};

// D3D standard sample patterns (1, 4, 8 and 16 samples), offsets from the pixel's top-left corner, image space
// (x right, y down).  All are multiples of 1/16: sample coordinates are exact in float32.
// Indexed with compile-time (unrolled) s so the offsets fold into immediates.
template <int MSAA>
MWB_DEV float sample_x(int s) {
  if (MSAA == 1) return 0.5f;
  if (MSAA == 16) return s == 0 ? 0.5625f : s == 1 ? 0.4375f : s == 2 ? 0.3125f : s == 3 ? 0.7500f : s == 4 ? 0.1875f : s == 5 ? 0.6250f : s == 6 ? 0.8125f : s == 7 ? 0.6875f : s == 8 ? 0.3750f : s == 9 ? 0.5000f : s == 10 ? 0.2500f : s == 11 ? 0.1250f : s == 12 ? 0.0000f : s == 13 ? 0.9375f : s == 14 ? 0.8750f : 0.0625f;
  if (MSAA == 4) return s == 0 ? 0.375f : s == 1 ? 0.875f : s == 2 ? 0.125f : 0.625f;
  return s == 0 ? 0.5625f : s == 1 ? 0.4375f : s == 2 ? 0.8125f : s == 3 ? 0.3125f
       : s == 4 ? 0.1875f : s == 5 ? 0.0625f : s == 6 ? 0.6875f : 0.9375f;
}
template <int MSAA>
MWB_DEV float sample_y(int s) {
  if (MSAA == 1) return 0.5f;
  if (MSAA == 16) return s == 0 ? 0.5625f : s == 1 ? 0.3125f : s == 2 ? 0.6250f : s == 3 ? 0.4375f : s == 4 ? 0.3750f : s == 5 ? 0.8125f : s == 6 ? 0.6875f : s == 7 ? 0.1875f : s == 8 ? 0.8750f : s == 9 ? 0.0625f : s == 10 ? 0.1250f : s == 11 ? 0.7500f : s == 12 ? 0.5000f : s == 13 ? 0.2500f : s == 14 ? 0.9375f : 0.0000f;
  if (MSAA == 4) return s == 0 ? 0.125f : s == 1 ? 0.375f : s == 2 ? 0.625f : 0.875f;
  return s == 0 ? 0.3125f : s == 1 ? 0.6875f : s == 2 ? 0.5625f : s == 3 ? 0.1875f
       : s == 4 ? 0.8125f : s == 5 ? 0.4375f : s == 6 ? 0.9375f : 0.0625f;
}

// the same offsets for a run-time sample index: sixteenths packed four bits per sample
template <int MSAA>
MWB_DEV void sample_xy_dyn(int s, float& x, float& y) {
  const uint64_t XN = MSAA == 16 ? 0x1ef02486bda3c579ull : MSAA == 8 ? 0xfb135d79ull : (MSAA == 4 ? 0xa2e6ull : 0x8ull);
  const uint64_t YN = MSAA == 16 ? 0xf48c21e3bd67a59ull : MSAA == 8 ? 0x1f7d39b5ull : (MSAA == 4 ? 0xea62ull : 0x8ull);
  x = (float)(uint32_t)((XN >> (4 * s)) & 15ull) * 0.0625f;
  y = (float)(uint32_t)((YN >> (4 * s)) & 15ull) * 0.0625f;
}

struct Camera {
  float ex, ey, ez;              // eye
  float sx, sy, sz;              // right   (gluLookAt's s)
  float ux, uy, uz;              // up      (u = s x f)
  float fx, fy, fz;              // forward (f)
  float px, py;                  // projection scales cot/aspect, cot
  float za, zb;                  // z_clip = za * w_clip - zb
  float halfw, halfh;
  float light[3], lamb[3], ldif[3], sky[3];   // light = DIRECTION towards LIGHT0 (see camera_common)
  float linv;                    // 1 / |light|
  float sample_ext;              // largest |offset| of a sample from the pixel centre: 7/16 (1, 4, 8 samples), 8/16 (16)
  int ortho;                     // 1: render_top_view's orthographic map projection
  float osx, otx, osy, oty;      // x_clip = osx x + otx, y_clip = osy (-z) + oty, z_clip = -0.01 y, w = 1
};

// Which view a render launch draws: the agent's camera (render_obs, miniworld.py:1177-1221) or the
// orthographic map of render_top_view (miniworld.py:1088-1175): glOrtho(l, r, b, t, -100, 100) under
// the model-view that maps world (x, y, z) to eye (x, -z, y), plus the agent's marker triangle.
struct ViewSpec {
  int mode;                      // 0 = agent camera, 1 = top view
  int render_agent;              // top view: draw Agent.render()'s triangle (entity.py:518-539)
  double l, r, b, t;             // glOrtho extents (top view)
};

// The three camera angles of env i (heading, pitch, half the vertical field of view), float64.
MWB_DEV void camera_angles(const DevState& S, int i, double ang[3]) {
  const size_t N = S.N;
  const int as = S.agent_slot[i];
  ang[0] = S.ent_dir[as * N + i];
  ang[1] = d_div(d_mul(S.cam[2 * N + i], 3.141592653589793), 180.0);
  ang[2] = d_div(d_mul(S.cam[3 * N + i], 3.141592653589793), 360.0);
}

// view-independent part: viewport scale, sky colour, light.
// LIGHT0 is DIRECTIONAL: the reference issues glLightfv(GL_LIGHT0, GL_POSITION, (GLfloat * 4)(*self.light_pos + [1]))
// (miniworld.py:1031) with light_pos a numpy array (params.py:45-46 turns every default into one, rng.uniform returns
// one), so `+ [1]` adds 1 to each component, three GLfloats are passed and w stays 0: a light at infinity in the
// direction float32(light_pos + 1).  Pinned by the recorded GL stream (oracle/gl_record.py, tests/test_stream_oracle.py).
MWB_DEV void camera_common(const DevState& S, int i, Camera& c) {
  const size_t N = S.N;
  c.halfw = 0.5f * (float)S.obs_w;
  c.halfh = 0.5f * (float)S.obs_h;
  c.sample_ext = S.msaa == 16 ? 0.5f : 0.4375f;
  for (int k = 0; k < 3; ++k) {
    c.sky[k] = (float)S.envp[(0 + k) * N + i];
    c.light[k] = (float)d_add(S.envp[(3 + k) * N + i], 1.0);
    c.ldif[k] = (float)S.envp[(6 + k) * N + i];
    c.lamb[k] = (float)S.envp[(9 + k) * N + i];
  }
  c.linv = 1.0f / sqrtf(c.light[0] * c.light[0] + c.light[1] * c.light[1] + c.light[2] * c.light[2]);
}

// Camera of env i from trig = {cos, sin} of those angles.  Angles go through the glibc-exact
// sin / cos so that the oracle, fed the same (pos, dir, cam_*) doubles on the host, derives the
// identical float32 basis.  (The six evaluations are independent: the kernel spreads them over
// six threads.)
MWB_DEV Camera make_camera(const DevState& S, int i, const double trig[6]) {
  const size_t N = S.N;
  const int as = S.agent_slot[i];
  double px = S.ent_px[as * N + i], py = S.ent_py[as * N + i], pz = S.ent_pz[as * N + i];
  double h = S.cam[0 * N + i], fd = S.cam[1 * N + i];
  const double ct = trig[0], st = trig[1], cp = trig[2], sp = trig[3];
  Camera c;
  c.ex = (float)d_add(px, d_mul(fd, ct));
  c.ey = (float)d_add(py, h);
  c.ez = (float)d_sub(pz, d_mul(fd, st));
  c.sx = (float)st;
  c.sy = 0.0f;
  c.sz = (float)ct;
  c.ux = (float)(-d_mul(ct, sp));
  c.uy = (float)cp;
  c.uz = (float)d_mul(st, sp);
  c.fx = (float)d_mul(cp, ct);
  c.fy = (float)sp;
  c.fz = (float)(-d_mul(cp, st));
  double cot = d_div(trig[4], trig[5]);
  c.py = (float)cot;
  c.px = (float)d_div(cot, d_div((double)S.obs_w, (double)S.obs_h));
  c.za = (float)((MWB_FAR + MWB_NEAR) / (MWB_FAR - MWB_NEAR));
  c.zb = (float)(2.0 * MWB_FAR * MWB_NEAR / (MWB_FAR - MWB_NEAR));
  c.ortho = 0;
  c.osx = c.otx = c.osy = c.oty = 0.0f;
  camera_common(S, i, c);
  return c;
}

// render_top_view's camera: the projection matrix entries are formed in float64 and rounded once, as
// glOrtho's GLdouble arguments end up in a float32 matrix.
MWB_DEV Camera make_top_camera(const DevState& S, int i, const ViewSpec& v) {
  Camera c;
  c.ex = c.ey = c.ez = 0.0f;
  c.sx = c.sy = c.sz = c.ux = c.uy = c.uz = c.fx = c.fy = c.fz = 0.0f;
  c.px = c.py = c.za = c.zb = 0.0f;
  c.ortho = 1;
  c.osx = (float)d_div(2.0, d_sub(v.r, v.l));
  c.otx = (float)(-d_div(d_add(v.r, v.l), d_sub(v.r, v.l)));
  c.osy = (float)d_div(2.0, d_sub(v.t, v.b));
  c.oty = (float)(-d_div(d_add(v.t, v.b), d_sub(v.t, v.b)));
  camera_common(S, i, c);
  return c;
}

MWB_DEV Camera make_camera(const DevState& S, int i) {
  double ang[3], trig[6];
  camera_angles(S, i, ang);
  for (int k = 0; k < 3; ++k) {
    trig[2 * k] = mwb_libm::cos_glibc(ang[k]);
    trig[2 * k + 1] = mwb_libm::sin_glibc(ang[k]);
  }
  return make_camera(S, i, trig);
}

// vertex after the exact part of the pipeline: window-homogeneous position + z numerator
struct HVert {
  float X, Y, w, zeta;           // X/w = column, Y/w = row (y down), zeta/w = window z in [0,1]
  float xc, yc, zc;              // clip x, y, z (frustum tests)
};

MWB_DEV float dot3_rn(float ax, float ay, float az, float bx, float by, float bz) {
  return f_add(f_add(f_mul(ax, bx), f_mul(ay, by)), f_mul(az, bz));
}

MWB_DEV HVert transform_vertex(const Camera& c, float x, float y, float z) {
  HVert v;
  float w;
  if (c.ortho) {               // eye = (x, -z, y); clip = glOrtho row by row, w = 1
    w = 1.0f;
    v.xc = f_add(f_mul(c.osx, x), c.otx);
    v.yc = f_add(f_mul(c.osy, -z), c.oty);
    v.zc = f_mul((float)(-2.0 / 200.0), y);
  } else {
    float rx = f_sub(x, c.ex), ry = f_sub(y, c.ey), rz = f_sub(z, c.ez);
    float xe = dot3_rn(c.sx, c.sy, c.sz, rx, ry, rz);
    float ye = dot3_rn(c.ux, c.uy, c.uz, rx, ry, rz);
    w = dot3_rn(c.fx, c.fy, c.fz, rx, ry, rz);   // distance along the view axis
    v.xc = f_mul(c.px, xe);
    v.yc = f_mul(c.py, ye);
    v.zc = f_sub(f_mul(c.za, w), c.zb);
  }
  v.w = w;
  v.X = f_mul(f_add(v.xc, w), c.halfw);
  v.Y = f_mul(f_sub(w, v.yc), c.halfh);
  v.zeta = f_mul(0.5f, f_add(v.zc, w));
  return v;
}

// Fixed-function vertex lighting (one directional light, no specular):
// clamp01(m * (0.2 + L_amb + L_diff * max(N . norm(L), 0))); N is NOT renormalised
// (neither GL_NORMALIZE nor GL_RESCALE_NORMAL is enabled by the reference).
MWB_DEV void light_vertex(const Camera& c, float nx, float ny, float nz, const float m[3], float out[3]) {
  float ndl = (nx * c.light[0] + ny * c.light[1] + nz * c.light[2]) * c.linv;
  ndl = ndl > 0.0f ? ndl : 0.0f;
  for (int k = 0; k < 3; ++k) {
    float v = m[k] * (0.2f + c.lamb[k] + c.ldif[k] * ndl);
    out[k] = v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
  }
}

// One set-up triangle, 44 words (176 B, 16-byte aligned so the rasteriser's hot part -- the
// first 64 bytes -- moves as four 128-bit loads).  Edge k is opposite vertex k, so
// E_k / sum(E) is the perspective-correct weight of vertex k's attributes.
struct MWB_ALIGN16 TriRec {
  float A[3], B[3], C[3];        // homogeneous edge functions E_k(x, y) = A x + B y + C  (exact)
  float R[3];                    // conservative half-extent of E_k over a pixel (+ rounding margin)
  float Za, Zb, Zc;              // window z plane (exact)
  float Zr;                      // conservative half-extent of z over a pixel (+ rounding margin)
  float T[3];                    // tie rule as a threshold: sample inside edge k  <=>  E_k >= T[k]
  int32_t tex;                   // texture id or -1       (T = 0 if the edge owns E == 0, else the
  int32_t bx, by;                //                         smallest positive float, i.e. E > 0)
  float u[3], v[3];              // texcoords per vertex
  float r[3], g[3], b[3];        // lit colour per vertex
  float UA, UB, VA, VB, SA, SB;  // sum_k u_k A_k, sum_k u_k B_k, ... : per-triangle parts of du/dx, dv/dx, ...
  float K[3];                    // half-tile rejection: max of E_k over an 8x4 block at (x0, y0) is A x0 + B y0 + K
  float Kz;                      // likewise min of z - Zr: Za x0 + Zb y0 + Kz
  int32_t flat;                  // 1: the three lit vertex colours are identical (flat normal under the directional light)
};

// the hot 76 bytes of a TriRec, held in registers while a tile is rasterised
struct HotTri {
  float A[3], B[3], C[3], R[3];
  float Za, Zb, Zc, Zr;
  float T[3];
};

MWB_DEV HotTri load_hot(const TriRec* t) {
  HotTri h;
#ifdef __CUDA_ARCH__
  const float4* p = reinterpret_cast<const float4*>(t);
  const float4 q0 = p[0], q1 = p[1], q2 = p[2], q3 = p[3], q4 = p[4];
  h.A[0] = q0.x; h.A[1] = q0.y; h.A[2] = q0.z; h.B[0] = q0.w;
  h.B[1] = q1.x; h.B[2] = q1.y; h.C[0] = q1.z; h.C[1] = q1.w;
  h.C[2] = q2.x; h.R[0] = q2.y; h.R[1] = q2.z; h.R[2] = q2.w;
  h.Za = q3.x; h.Zb = q3.y; h.Zc = q3.z; h.Zr = q3.w;
  h.T[0] = q4.x; h.T[1] = q4.y; h.T[2] = q4.z;
#else
  for (int k = 0; k < 3; ++k) { h.A[k] = t->A[k]; h.B[k] = t->B[k]; h.C[k] = t->C[k]; h.R[k] = t->R[k]; h.T[k] = t->T[k]; }
  h.Za = t->Za; h.Zb = t->Zb; h.Zc = t->Zc; h.Zr = t->Zr;
#endif
  return h;
}

struct VertAttr {
  float u, v, r, g, b;
};

MWB_DEV bool frustum_reject(const HVert& a, const HVert& b, const HVert& c) {
  if (a.xc < -a.w && b.xc < -b.w && c.xc < -c.w) return true;
  if (a.xc > a.w && b.xc > b.w && c.xc > c.w) return true;
  if (a.yc < -a.w && b.yc < -b.w && c.yc < -c.w) return true;
  if (a.yc > a.w && b.yc > b.w && c.yc > c.w) return true;
  if (a.zc < -a.w && b.zc < -b.w && c.zc < -c.w) return true;
  if (a.zc > a.w && b.zc > b.w && c.zc > c.w) return true;
  return false;
}

MWB_DEV void edge_rn(const HVert& a, const HVert& b, float& A, float& B, float& C) {
  A = f_sub(f_mul(a.Y, b.w), f_mul(a.w, b.Y));
  B = f_sub(f_mul(a.w, b.X), f_mul(a.X, b.w));
  C = f_sub(f_mul(a.X, b.Y), f_mul(a.Y, b.X));
}

// GL triangle (v0, v1, v2), counter-clockwise = front in GL's y-up window.  In image space
// (y down) front faces have negative signed area, so edges are built on (v0, v2, v1): then
// det > 0 <=> front-facing and the interior is E_k >= 0.  Returns false if culled.
MWB_DEV bool setup_triangle(const HVert& g0, const HVert& g1, const HVert& g2, const VertAttr& a0,
                            const VertAttr& a1, const VertAttr& a2, int tex, int W, int H, TriRec& t,
                            float ext = 0.4375f /* Camera.sample_ext */) {
  if (frustum_reject(g0, g1, g2)) return false;
  const HVert& v0 = g0;
  const HVert& v1 = g2;
  const HVert& v2 = g1;
  edge_rn(v1, v2, t.A[0], t.B[0], t.C[0]);
  edge_rn(v2, v0, t.A[1], t.B[1], t.C[1]);
  edge_rn(v0, v1, t.A[2], t.B[2], t.C[2]);
  float det = f_add(f_add(f_mul(v0.X, t.A[0]), f_mul(v0.Y, t.B[0])), f_mul(v0.w, t.C[0]));
  if (!(det > 0.0f)) return false;   // back-facing or degenerate (GL_CULL_FACE, GL_BACK)
  t.Za = f_div(f_add(f_add(f_mul(v0.zeta, t.A[0]), f_mul(v1.zeta, t.A[1])), f_mul(v2.zeta, t.A[2])), det);
  t.Zb = f_div(f_add(f_add(f_mul(v0.zeta, t.B[0]), f_mul(v1.zeta, t.B[1])), f_mul(v2.zeta, t.B[2])), det);
  t.Zc = f_div(f_add(f_add(f_mul(v0.zeta, t.C[0]), f_mul(v1.zeta, t.C[1])), f_mul(v2.zeta, t.C[2])), det);
  // |z(sample) - z(centre)| <= ext (|Za| + |Zb|); plus a bound on evaluation rounding
  t.Zr = ext * (fabsf(t.Za) + fabsf(t.Zb)) + 4e-6f * (fabsf(t.Za) * (float)W + fabsf(t.Zb) * (float)H + fabsf(t.Zc)) + 1e-6f;
  t.Kz = t.Zc - t.Zr + 8.0f * fminf(t.Za, 0.0f) + 4.0f * fminf(t.Zb, 0.0f);
  for (int k = 0; k < 3; ++k) {
    float aa = fabsf(t.A[k]), ab = fabsf(t.B[k]);
    // |E(sample) - E(centre)| <= ext (|A| + |B|); plus a bound on evaluation rounding
    t.R[k] = ext * (aa + ab) + 4e-6f * (aa * (float)W + ab * (float)H + fabsf(t.C[k])) + 1e-30f;
    // tie rule: the edge with A > 0, or A == 0 and B > 0, owns samples with E == 0
    t.T[k] = (t.A[k] > 0.0f || (t.A[k] == 0.0f && t.B[k] > 0.0f)) ? 0.0f : 1.401298464e-45f;
    t.K[k] = t.C[k] + t.R[k] + 8.0f * fmaxf(t.A[k], 0.0f) + 4.0f * fmaxf(t.B[k], 0.0f);
  }
  const VertAttr& b0 = a0;
  const VertAttr& b1 = a2;
  const VertAttr& b2 = a1;
  t.u[0] = b0.u; t.u[1] = b1.u; t.u[2] = b2.u;
  t.v[0] = b0.v; t.v[1] = b1.v; t.v[2] = b2.v;
  t.r[0] = b0.r; t.r[1] = b1.r; t.r[2] = b2.r;
  t.g[0] = b0.g; t.g[1] = b1.g; t.g[2] = b2.g;
  t.b[0] = b0.b; t.b[1] = b1.b; t.b[2] = b2.b;
  t.tex = tex;
  t.flat = (b0.r == b1.r && b1.r == b2.r && b0.g == b1.g && b1.g == b2.g && b0.b == b1.b && b1.b == b2.b) ? 1 : 0;
  t.UA = t.u[0] * t.A[0] + t.u[1] * t.A[1] + t.u[2] * t.A[2];
  t.UB = t.u[0] * t.B[0] + t.u[1] * t.B[1] + t.u[2] * t.B[2];
  t.VA = t.v[0] * t.A[0] + t.v[1] * t.A[1] + t.v[2] * t.A[2];
  t.VB = t.v[0] * t.B[0] + t.v[1] * t.B[1] + t.v[2] * t.B[2];
  t.SA = t.A[0] + t.A[1] + t.A[2];
  t.SB = t.B[0] + t.B[1] + t.B[2];
  // screen bbox (conservative); any vertex at or behind the eye plane -> whole frame
  int x0 = 0, x1 = W - 1, y0 = 0, y1 = H - 1;
  const float weps = 1e-3f;
  if (v0.w > weps && v1.w > weps && v2.w > weps) {
    float xa = v0.X / v0.w, xb = v1.X / v1.w, xc = v2.X / v2.w;
    float ya = v0.Y / v0.w, yb = v1.Y / v1.w, yc = v2.Y / v2.w;
    float fx0 = fminf(xa, fminf(xb, xc)) - 1.0f, fx1 = fmaxf(xa, fmaxf(xb, xc)) + 1.0f;
    float fy0 = fminf(ya, fminf(yb, yc)) - 1.0f, fy1 = fmaxf(ya, fmaxf(yb, yc)) + 1.0f;
    if (fx1 < 0.0f || fy1 < 0.0f || fx0 > (float)W || fy0 > (float)H) return false;
    x0 = fx0 > 0.0f ? (int)fx0 : 0;
    y0 = fy0 > 0.0f ? (int)fy0 : 0;
    x1 = fx1 < (float)(W - 1) ? (int)fx1 : W - 1;
    y1 = fy1 < (float)(H - 1) ? (int)fy1 : H - 1;
  }
  t.bx = x0 | (x1 << 16);
  t.by = y0 | (y1 << 16);
  return true;
}

// Exact edge value at a sample.  Shared edges are watertight: the neighbouring triangle sees
// the exactly negated (A, B, C), and exactly one of the two owns E == 0 (threshold T).
MWB_DEV float edge_value(float A, float B, float C, float xs, float ys) {
  return f_add(f_add(f_mul(A, xs), f_mul(B, ys)), C);
}

template <int MSAA>
MWB_DEV uint32_t max_key(const uint32_t (&keys)[MSAA]) {
  uint32_t m = keys[0];
#pragma unroll
  for (int s = 1; s < MSAA; ++s) m = keys[s] > m ? keys[s] : m;
  return m;
}

// Depth-tested visibility of triangle `slot` over the MSAA samples of pixel (px, py).
// keys[s] = depth16 << 16 | slot of the nearest surface so far (GL_LESS on 16-bit codes;
// slots ascend in draw order, so on equal codes the earlier draw keeps the sample).
// `kmax` caches max(keys): a triangle whose nearest possible depth code over the pixel is
// already behind every stored sample cannot win any GL_LESS test and is skipped.
template <int MSAA>
MWB_DEV void raster_pixel(const HotTri& t, int slot, int px, int py, uint32_t (&keys)[MSAA], uint32_t& kmax) {
  const float cx = (float)px + 0.5f, cy = (float)py + 0.5f;
  const float e0 = t.A[0] * cx + t.B[0] * cy + t.C[0];
  const float e1 = t.A[1] * cx + t.B[1] * cy + t.C[1];
  const float e2 = t.A[2] * cx + t.B[2] * cy + t.C[2];
  if (e0 + t.R[0] < 0.0f || e1 + t.R[1] < 0.0f || e2 + t.R[2] < 0.0f) return;  // certainly outside
  const float zc = t.Za * cx + t.Zb * cy + t.Zc;
  const float zlo = zc - t.Zr;
  if (zlo > 1.0f || zc + t.Zr < 0.0f) return;                                 // beyond far / before near
  // smallest code any sample of this pixel can get (one code of slack for the rounding of z * 65535)
  if (zlo * 65535.0f - 1.0f > (float)(kmax >> 16)) return;                    // certainly occluded
  const bool full = e0 - t.R[0] > 0.0f && e1 - t.R[1] > 0.0f && e2 - t.R[2] > 0.0f;   // certainly inside
  const float fx = (float)px, fy = (float)py;
  bool changed = false;
#pragma unroll
  for (int s = 0; s < MSAA; ++s) {
    const float xs = fx + sample_x<MSAA>(s), ys = fy + sample_y<MSAA>(s);
    bool in = true;
    if (!full)
      in = edge_value(t.A[0], t.B[0], t.C[0], xs, ys) >= t.T[0] && edge_value(t.A[1], t.B[1], t.C[1], xs, ys) >= t.T[1] &&
           edge_value(t.A[2], t.B[2], t.C[2], xs, ys) >= t.T[2];
    const float z = f_add(f_add(f_mul(t.Za, xs), f_mul(t.Zb, ys)), t.Zc);
    in = in && z >= 0.0f && z <= 1.0f;   // near / far clip (also drops NaN)
    const uint32_t code = (uint32_t)f_add(f_mul(z, 65535.0f), 0.5f);
    const uint32_t key = (code << 16) | (uint32_t)slot;
    if (in && key < keys[s]) {
      keys[s] = key;
      changed = true;
    }
  }
  if (changed) kmax = max_key<MSAA>(keys);
}

// ---------------------------------------------------------------------------- shading

// ---- lazy visibility ---------------------------------------------------------------------
// Most pixels of a frame end up entirely inside ONE triangle.  For them the eight exact
// per-sample depth codes are never needed: PixelState keeps such a pixel in LAZY mode ("all
// samples belong to triangle `lazy_slot`, whose depth codes lie in [lazy_clo, lazy_chi]") and only
// MATERIALISES the explicit per-sample keys when a later triangle cannot be ordered against
// it by conservative bounds alone.  Every shortcut is one-sided: a triangle is skipped only if
// it would certainly lose every GL_LESS test, installed lazily only if it certainly covers all
// samples, is not clipped and certainly wins them all.  The final image is therefore identical
// to plain per-sample processing (and independent of the order triangles are visited in, since
// the per-sample result is min over (depth code, slot)).
#define MWB_PX_EMPTY 0
#define MWB_PX_LAZY 1
#define MWB_PX_EXPLICIT 2

template <int MSAA>
struct PixelState {
  uint32_t keys[MSAA];
  uint32_t kmax;
  int32_t mode;
  int32_t lazy_slot;
  float lazy_clo, lazy_chi;      // conservative bounds of the lazy triangle's depth codes here
  float bound;                   // EXPLICIT mode: an upper bound of every stored depth code
  int32_t pair_skip;             // slot whose samples at this pixel are already accounted for (see classify_pixel), or -1
};

template <int MSAA>
MWB_DEV void pixel_init(PixelState<MSAA>& p) {
#pragma unroll
  for (int s = 0; s < MSAA; ++s) p.keys[s] = MWB_SKY_KEY;
  p.kmax = MWB_SKY_KEY;
  p.mode = MWB_PX_EMPTY;
  p.lazy_slot = -1;
  p.lazy_clo = p.lazy_chi = 65535.0f;
  p.bound = 65535.0f;
  p.pair_skip = -1;
}

// A lazy pixel held by a PAIR: the two fan triangles (0,1,2), (0,2,3) of one planar quad together cover every sample.
template <int MSAA>
MWB_DEV bool lazy_is_pair(const PixelState<MSAA>& p) { return p.pair_skip == (p.lazy_slot ^ 1); }

// largest depth code that can currently be stored at any sample of the pixel
template <int MSAA>
MWB_DEV float pixel_bound(const PixelState<MSAA>& p) {
  return p.mode == MWB_PX_LAZY ? p.lazy_chi : p.bound;
}

// the 16 floats classification needs (A, B, C, R, Z plane), broadcast to the whole warp
struct ClassTri {
  float A[3], B[3], C[3], R[3];
  float Za, Zb, Zc, Zr;
};

MWB_DEV ClassTri load_class(const TriRec* t) {
  ClassTri h;
#ifdef __CUDA_ARCH__
  const float4* p = reinterpret_cast<const float4*>(t);
  const float4 q0 = p[0], q1 = p[1], q2 = p[2], q3 = p[3];
  h.A[0] = q0.x; h.A[1] = q0.y; h.A[2] = q0.z; h.B[0] = q0.w;
  h.B[1] = q1.x; h.B[2] = q1.y; h.C[0] = q1.z; h.C[1] = q1.w;
  h.C[2] = q2.x; h.R[0] = q2.y; h.R[1] = q2.z; h.R[2] = q2.w;
  h.Za = q3.x; h.Zb = q3.y; h.Zc = q3.z; h.Zr = q3.w;
#else
  for (int k = 0; k < 3; ++k) { h.A[k] = t->A[k]; h.B[k] = t->B[k]; h.C[k] = t->C[k]; h.R[k] = t->R[k]; }
  h.Za = t->Za; h.Zb = t->Zb; h.Zc = t->Zc; h.Zr = t->Zr;
#endif
  return h;
}

// Cheap per-pixel triage of one triangle.  Returns 0 if it was skipped or installed lazily; else it
// still needs exact per-sample processing at this pixel: 1 = partial coverage possible, 2 = it
// certainly covers every sample (edge tests can be skipped).
//
// Quad pairs.  Room quads and box faces reach the rasteriser as the fan triangles (0,1,2), (0,2,3) of a planar quad,
// stored in adjacent records / slots (2k, 2k + 1); the shared diagonal is edge 2 of the first and edge 1 of the
// second, with exactly negated coefficients and complementary tie thresholds, so a sample inside the quad's four
// OUTER edges belongs to exactly one of the two.  `partner` (or null) is the other record of such a pair: a pixel
// whose samples are all certainly inside the four outer edges is held lazily by the pair -- which triangle owns a
// given sample is only decided if the exact keys are ever needed (materialisation queues both; the depth map
// evaluates the diagonal at sample 0).  Without this every pixel a diagonal crosses would go through the exact
// per-sample path although it shows a single flat surface.
template <int MSAA>
MWB_DEV int classify_pixel(const ClassTri& t, int slot, int px, int py, PixelState<MSAA>& p, const TriRec* partner = nullptr,
                           int diag = 0) {
  if (slot == p.pair_skip) return 0;                      // already covered through its partner at this pixel
  const float cx = (float)px + 0.5f, cy = (float)py + 0.5f;
  const float e0 = t.A[0] * cx + t.B[0] * cy + t.C[0];
  const float e1 = t.A[1] * cx + t.B[1] * cy + t.C[1];
  const float e2 = t.A[2] * cx + t.B[2] * cy + t.C[2];
  if (e0 + t.R[0] < 0.0f || e1 + t.R[1] < 0.0f || e2 + t.R[2] < 0.0f) return 0;      // certainly outside
  const float zc = t.Za * cx + t.Zb * cy + t.Zc;
  const float zlo = zc - t.Zr, zhi = zc + t.Zr;
  if (zlo > 1.0f || zhi < 0.0f) return 0;                                             // certainly clipped away
  // depth codes any sample of this pixel can get lie in [clo, chi] (one code of slack each way)
  float clo = zlo * 65535.0f - 1.0f, chi = zhi * 65535.0f + 1.5f;
  if (clo > pixel_bound(p)) return 0;                                                 // certainly occluded
  const bool in0 = e0 - t.R[0] > 0.0f, in1 = e1 - t.R[1] > 0.0f, in2 = e2 - t.R[2] > 0.0f;
  const bool full = in0 && in1 && in2;                                                // covers every sample
  bool pair = false;
  if (partner != nullptr && !full && in0 && (diag == 1 ? in2 : in1)) {
    // only the diagonal is undecided here: do the partner's two outer edges certainly contain every sample too?
    // (the partner's diagonal is edge 3 - diag; its plane is this one up to rounding: one more code of slack)
    const int pd = 3 - diag, k1 = pd == 1 ? 2 : 1;
    const float f0 = partner->A[0] * cx + partner->B[0] * cy + partner->C[0] - partner->R[0];
    const float f1 = partner->A[k1] * cx + partner->B[k1] * cy + partner->C[k1] - partner->R[k1];
    pair = f0 > 0.0f && f1 > 0.0f && zlo >= 2e-5f;
    if (pair) { clo -= 1.0f; chi += 1.0f; }
  }
  const bool unclipped = zlo >= 0.0f && zhi <= 1.0f && chi < 65535.0f;
  if ((full || pair) && unclipped) {
    const bool wins = p.mode == MWB_PX_EMPTY || (p.mode == MWB_PX_LAZY && chi < p.lazy_clo);
    if (wins) {                      // every sample now certainly belongs to this triangle (or its pair)
      p.mode = MWB_PX_LAZY;
      p.lazy_slot = slot;
      p.lazy_clo = clo;
      p.lazy_chi = chi;
      if (pair) p.pair_skip = slot ^ 1;
      return 0;
    }
  }
  return full ? 2 : 1;
}

// Record that no sample can ever hit (the culled half of a quad pair keeps its slot)
MWB_DEV void empty_record(TriRec& r) {
  for (int k = 0; k < 3; ++k) {
    r.A[k] = r.B[k] = 0.0f;
    r.C[k] = -1.0f;
    r.R[k] = 0.0f;
    r.T[k] = 0.0f;
    r.K[k] = -1.0f;
    r.u[k] = r.v[k] = r.r[k] = r.g[k] = r.b[k] = 0.0f;
  }
  r.Za = r.Zb = 0.0f;
  r.Zc = 2.0f;
  r.Zr = 0.0f;
  r.Kz = 2.0f;
  r.tex = -1;
  r.flat = 1;
  r.bx = 1;          // x0 = 1 > x1 = 0
  r.by = 1;
  r.UA = r.UB = r.VA = r.VB = r.SA = r.SB = 0.0f;
}

// Which record of a pair owns sample (xs, ys) that lies inside the quad: the one whose diagonal edge says so
MWB_DEV bool pair_sample_in_first(const TriRec& t, int diag, float xs, float ys) {
  return edge_value(t.A[diag], t.B[diag], t.C[diag], xs, ys) >= t.T[diag];
}

// One sample of the exact path: coverage by the three edge functions (unless the triangle is
// known to cover the whole pixel), window z, 16-bit depth code.  Returns the packed key, or
// 0xFFFFFFFF if the sample is not covered / clipped.
MWB_DEV uint32_t sample_key(const HotTri& t, int slot, float xs, float ys, bool full) {
  bool in = true;
  if (!full)
    in = edge_value(t.A[0], t.B[0], t.C[0], xs, ys) >= t.T[0] && edge_value(t.A[1], t.B[1], t.C[1], xs, ys) >= t.T[1] &&
         edge_value(t.A[2], t.B[2], t.C[2], xs, ys) >= t.T[2];
  const float z = f_add(f_add(f_mul(t.Za, xs), f_mul(t.Zb, ys)), t.Zc);
  in = in && z >= 0.0f && z <= 1.0f;
  const uint32_t code = (uint32_t)f_add(f_mul(z, 65535.0f), 0.5f);
  return in ? ((code << 16) | (uint32_t)slot) : 0xFFFFFFFFu;
}

// GL_REPEAT + GL_LINEAR on one mip level.  The texcoord is reduced to [0, 1) first (exact in
// float32), so the texel index needs one conditional add instead of an integer modulo; 8-bit
// texels are widened with the 2^23 "magic number" trick (byte dropped into the mantissa of
// 8388608.0f), which also makes the differences c10 - c00 exact.
MWB_DEV float texel_f(uint32_t t, int k) {
#ifdef __CUDA_ARCH__
  return __uint_as_float(__byte_perm(t, 0x4B000000u, k == 0 ? 0x7650u : (k == 1 ? 0x7651u : 0x7652u)));
#else
  union { uint32_t u; float f; } c;
  c.u = 0x4B000000u | ((t >> (8 * k)) & 255u);
  return c.f;
#endif
}

MWB_DEV void bilinear(const RenderAssets& A, const TexDev& T, int level, float u, float v, float out[3]) {
  const int w = T.lw[level], h = T.lh[level];
  const float x = (u - floorf(u)) * (float)w - 0.5f, y = (v - floorf(v)) * (float)h - 0.5f;   // in [-0.5, size - 0.5)
  const float xf = floorf(x), yf = floorf(y);
  const float fx = x - xf, fy = y - yf;
#ifdef __CUDA_ARCH__
  if (A.atlas != 0ull) {
    // The texture unit fetches the footprint: tld4 (texture gather) at the texel CORNER shared by the four texels
    // (xf, yf) .. (xf + 1, yf + 1) -- half a texel away from every footprint boundary, so the unit's own fixed-point
    // coordinate arithmetic cannot pick another 2x2 block -- returns one channel of the four texels per instruction,
    // already converted to float (exactly c / 255).  xf ranges over -1 .. w - 1: GL_REPEAT is the atlas rectangle's
    // wrapped border.  The weights fx, fy stay in float32 as above: addressing and unpacking moved to the TMU.
    const float gu = (T.ax[level] + (xf + 1.0f)) * A.atlas_iw, gv = (T.ay[level] + (yf + 1.0f)) * A.atlas_ih;
    const cudaTextureObject_t obj = (cudaTextureObject_t)A.atlas;
    const float4 c0 = tex2Dgather<float4>(obj, gu, gv, 0), c1 = tex2Dgather<float4>(obj, gu, gv, 1), c2 = tex2Dgather<float4>(obj, gu, gv, 2);
    // gather order (tools/gather_probe.cu): x = (x0, y1), y = (x1, y1), z = (x1, y0), w = (x0, y0)
    float top = c0.w + fx * (c0.z - c0.w), bot = c0.x + fx * (c0.y - c0.x);
    out[0] = top + fy * (bot - top);
    top = c1.w + fx * (c1.z - c1.w); bot = c1.x + fx * (c1.y - c1.x);
    out[1] = top + fy * (bot - top);
    top = c2.w + fx * (c2.z - c2.w); bot = c2.x + fx * (c2.y - c2.x);
    out[2] = top + fy * (bot - top);
    return;
  }
#endif
  const uint32_t* base = A.texels + T.off[level];
  int x0 = (int)xf, y0 = (int)yf;
  x0 = x0 < 0 ? x0 + w : (x0 >= w ? x0 - w : x0);
  y0 = y0 < 0 ? y0 + h : (y0 >= h ? y0 - h : y0);
  const int x1 = x0 + 1 == w ? 0 : x0 + 1, y1 = y0 + 1 == h ? 0 : y0 + 1;
  const uint32_t t00 = base[y0 * w + x0], t10 = base[y0 * w + x1], t01 = base[y1 * w + x0], t11 = base[y1 * w + x1];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float m00 = texel_f(t00, k), m10 = texel_f(t10, k), m01 = texel_f(t01, k), m11 = texel_f(t11, k);
    const float top = (m00 - 8388608.0f) + fx * (m10 - m00), bot = (m01 - 8388608.0f) + fx * (m11 - m01);
    out[k] = (top + fy * (bot - top)) * (1.0f / 255.0f);
  }
}

// Colour of triangle t at the centre of pixel (px, py): Gouraud colour x trilinear texture
// (GL_MODULATE), both interpolated perspective-correctly.  LOD from analytic derivatives.
MWB_DEV void shade_pixel(const RenderAssets& A, const TriRec& t, int px, int py, float out[3]) {
  float cx = (float)px + 0.5f, cy = (float)py + 0.5f;
  float e0 = t.A[0] * cx + t.B[0] * cy + t.C[0];
  float e1 = t.A[1] * cx + t.B[1] * cy + t.C[1];
  float e2 = t.A[2] * cx + t.B[2] * cy + t.C[2];
#ifdef __CUDA_ARCH__
  const float inv = __fdividef(1.0f, e0 + e1 + e2);     // colour path: MUFU.RCP accuracy is ample (<= 1 LSB contract)
#else
  const float inv = 1.0f / (e0 + e1 + e2);
#endif
  float b0 = e0 * inv, b1 = e1 * inv, b2 = e2 * inv;
  float r = t.r[0], g = t.g[0], b = t.b[0];
  if (!t.flat) {                 // Gouraud: the weights sum to 1, so equal vertex colours need no interpolation
    r = b0 * r + b1 * t.r[1] + b2 * t.r[2];
    g = b0 * g + b1 * t.g[1] + b2 * t.g[2];
    b = b0 * b + b1 * t.b[1] + b2 * t.b[2];
  }
  if (t.tex >= 0) {
    const TexDev& T = A.tex[t.tex];
    float u = b0 * t.u[0] + b1 * t.u[1] + b2 * t.u[2];
    float v = b0 * t.v[0] + b1 * t.v[1] + b2 * t.v[2];
    const float dudx = (t.UA - u * t.SA) * inv * (float)T.w, dvdx = (t.VA - v * t.SA) * inv * (float)T.h;
    const float dudy = (t.UB - u * t.SB) * inv * (float)T.w, dvdy = (t.VB - v * t.SB) * inv * (float)T.h;
    float rho2 = fmaxf(dudx * dudx + dvdx * dvdx, dudy * dudy + dvdy * dvdy);
#ifdef __CUDA_ARCH__
    float lambda = 0.5f * __log2f(fmaxf(rho2, 1e-20f));    // MUFU.LG2: the trilinear weight moves by < 1e-6
#else
    float lambda = 0.5f * log2f(fmaxf(rho2, 1e-20f));
#endif
    // magnification: GL_LINEAR on level 0; else GL_LINEAR_MIPMAP_LINEAR between floor(lambda) and +1
    const float lmax = (float)(T.nlev - 1);
    const float lc = lambda <= 0.0f ? 0.0f : (lambda >= lmax ? lmax : lambda);
    const int l0 = (int)lc;
    const float f = lc - (float)l0;
    float tc[3] = {0.0f, 0.0f, 0.0f};
#ifdef __CUDA_ARCH__
    if (A.atlas != 0ull) {
      // texture-unit path: the gathers of BOTH mip levels are issued before any of their results is used, so the two
      // texture round trips overlap (the loop below would serialise them)
      const cudaTextureObject_t obj = (cudaTextureObject_t)A.atlas;
      const float fu = u - floorf(u), fv = v - floorf(v);
      const float xa = fu * (float)T.lw[l0] - 0.5f, ya = fv * (float)T.lh[l0] - 0.5f;
      const float xaf = floorf(xa), yaf = floorf(ya);
      const float gua = (T.ax[l0] + (xaf + 1.0f)) * A.atlas_iw, gva = (T.ay[l0] + (yaf + 1.0f)) * A.atlas_ih;
      const float4 a0 = tex2Dgather<float4>(obj, gua, gva, 0), a1 = tex2Dgather<float4>(obj, gua, gva, 1), a2 = tex2Dgather<float4>(obj, gua, gva, 2);
      float4 b0 = a0, b1 = a1, b2 = a2;
      float fxb = 0.0f, fyb = 0.0f;
      if (f > 0.0f) {                       // (f > 0 implies l0 + 1 < nlev)
        const int l1 = l0 + 1;
        const float xb = fu * (float)T.lw[l1] - 0.5f, yb = fv * (float)T.lh[l1] - 0.5f;
        const float xbf = floorf(xb), ybf = floorf(yb);
        const float gub = (T.ax[l1] + (xbf + 1.0f)) * A.atlas_iw, gvb = (T.ay[l1] + (ybf + 1.0f)) * A.atlas_ih;
        b0 = tex2Dgather<float4>(obj, gub, gvb, 0);
        b1 = tex2Dgather<float4>(obj, gub, gvb, 1);
        b2 = tex2Dgather<float4>(obj, gub, gvb, 2);
        fxb = xb - xbf;
        fyb = yb - ybf;
      }
      const float fxa = xa - xaf, fya = ya - yaf, wa = 1.0f - f;
      // gather order (tools/gather_probe.cu): x = (x0, y1), y = (x1, y1), z = (x1, y0), w = (x0, y0)
#define MWB_BILERP(c, fx, fy) ((c.w + fx * (c.z - c.w)) + fy * ((c.x + fx * (c.y - c.x)) - (c.w + fx * (c.z - c.w))))
      tc[0] = wa * MWB_BILERP(a0, fxa, fya);
      tc[1] = wa * MWB_BILERP(a1, fxa, fya);
      tc[2] = wa * MWB_BILERP(a2, fxa, fya);
      if (f > 0.0f) {
        tc[0] += f * MWB_BILERP(b0, fxb, fyb);
        tc[1] += f * MWB_BILERP(b1, fxb, fyb);
        tc[2] += f * MWB_BILERP(b2, fxb, fyb);
      }
#undef MWB_BILERP
    } else
#endif
#pragma unroll 1
    for (int j = 0; j < 2; ++j) {
      const float wj = j == 0 ? 1.0f - f : f;
      if (wj == 0.0f) continue;
      float tj[3];
      bilinear(A, T, l0 + j, u, v, tj);
      tc[0] += wj * tj[0];
      tc[1] += wj * tj[1];
      tc[2] += wj * tj[2];
    }
    r *= tc[0];
    g *= tc[1];
    b *= tc[2];
  }
  out[0] = r;
  out[1] = g;
  out[2] = b;
}

// GreyscaleWrapper.observation (reference wrappers.py:43-46): 0.30 R + 0.59 G + 0.11 B as numpy evaluates it
// on the uint8 image -- float64, one rounding per operation, left to right
MWB_DEV double grey_f64(uint8_t r, uint8_t g, uint8_t b) {
  return d_add(d_add(d_mul(0.30, (double)r), d_mul(0.59, (double)g)), d_mul(0.11, (double)b));
}

MWB_DEV uint8_t to_unorm8(float c) {
  c = c < 0.0f ? 0.0f : (c > 1.0f ? 1.0f : c);
  return (uint8_t)(int)(c * 255.0f + 0.5f);
}

// depth16 code -> metres, the float32 arithmetic of FrameBuffer.get_depth_map
// (opengl.py:427-431): d = code / 65535; clip = (d - 0.5) * 2; z = -2 f n / (clip (f - n) - (f + n))
MWB_DEV float depth_code_to_metres(uint32_t code) {
  float d = f_div((float)code, 65535.0f);
  float clip = f_mul(f_sub(d, 0.5f), 2.0f);
  const float c0 = (float)(-2.0 * MWB_FAR * MWB_NEAR), c1 = (float)(MWB_FAR - MWB_NEAR), c2 = (float)(MWB_FAR + MWB_NEAR);
  return f_div(c0, f_sub(f_mul(clip, c1), c2));
}

// ------------------------------------------------------------------ scene -> triangles
// A frame's draw list, in the reference's submission order (miniworld.py:1052-1077): the
// static quads of every room, then the entities -- display-list (static) ones first, then the
// dynamic ones, each group in entity-list order.  It is cut into SEGMENTS: segment 0 = room
// triangles, segment 1 + k = the k-th drawn entity (a Box: <= 12 triangles set up in shared
// memory by the render kernel; a MeshEnt: set up by mesh_setup_kernel into HBM).  Triangle
// "slots" number the surviving triangles consecutively across segments, so slot order ==
// draw order and the per-sample key (depth16 << 16 | slot) implements GL_LESS exactly.

#define MWB_MAX_DRAWN 32               // = the entity-slot cap (MWB_MAX_ENTS_CAP): every non-agent entity can be drawn

struct FrameMap {
  int n_quads;                       // room quads of this env
  int n_ents;                        // drawn entities
  int n_tasks;                       // triangle tasks handled in shared memory: 2 per quad + 12 per box
  int ent_slot[MWB_MAX_DRAWN];       // entity-list slot
  int ent_proto[MWB_MAX_DRAWN];
  int ent_kind[MWB_MAX_DRAWN];       // MWB_KIND_BOX / MWB_KIND_MESH
  int ent_task0[MWB_MAX_DRAWN];      // first task index (boxes), -1 for meshes
  int agent_task;                    // task index of the agent's marker triangle (top view), else -1
};

struct EntPose {
  double x, y, z, dir;
  double col[3];
  double size;                       // per-episode Box edge length (PutNext), 0 = the prototype's size
};

MWB_DEV EntPose entity_pose(const DevState& S, int i, int e) {
  const size_t N = S.N;
  EntPose p;
  p.size = S.ent_size[e * N + i];
  if (e == S.ghost_slot[i]) {
    p.x = S.ghost_pose[0 * N + i];
    p.y = S.ghost_pose[1 * N + i];
    p.z = S.ghost_pose[2 * N + i];
    p.dir = S.ghost_pose[3 * N + i];
    for (int c = 0; c < 3; ++c) p.col[c] = S.ghost_col[c * N + i];
  } else {
    p.x = S.ent_px[e * N + i];
    p.y = S.ent_py[e * N + i];
    p.z = S.ent_pz[e * N + i];
    p.dir = S.ent_dir[e * N + i];
    for (int c = 0; c < 3; ++c) p.col[c] = S.ent_col[((size_t)e * 3 + c) * N + i];
  }
  return p;
}

MWB_DEV FrameMap build_frame_map(const DevState& S, int i, bool agent_marker = false) {
  FrameMap m;
  const size_t N = S.N;
  m.n_quads = S.num_quads[geom_index(S, i)];
  m.n_ents = 0;
  int tasks = 2 * m.n_quads;
  const int slots = S.num_slots[i];
  const int ghost = S.ghost_slot[i];
  for (int pass = 0; pass < 2; ++pass) {
    for (int e = 0; e < slots && m.n_ents < MWB_MAX_DRAWN; ++e) {
      const int p = e == ghost ? S.ghost_proto[i] : S.ent_proto[e * N + i];
      if (p < 0) continue;
      const mwb_proto& pr = S.protos[p];
      if (pr.kind != MWB_KIND_BOX && pr.kind != MWB_KIND_MESH) continue;   // the agent is never drawn
      if ((pr.is_static != 0) != (pass == 0)) continue;
      const int k = m.n_ents++;
      m.ent_slot[k] = e;
      m.ent_proto[k] = p;
      m.ent_kind[k] = pr.kind;
      m.ent_task0[k] = -1;
      if (pr.kind == MWB_KIND_BOX) {
        m.ent_task0[k] = tasks;
        tasks += 12;
      }
    }
  }
  m.agent_task = agent_marker ? tasks++ : -1;   // drawn last (miniworld.py:1079-1080)
  m.n_tasks = tasks;
  return m;
}

struct TriInput {
  float pos[3][3];
  float nrm[3][3];
  float uv[3][2];
  float mat[3][3];
  int tex;
};

// world-space triangle -> set-up record (transform, light, cull)
MWB_DEV bool finish_triangle(const Camera& cam, const TriInput& in, int W, int H, TriRec& out) {
  HVert hv[3];
  VertAttr at[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    hv[k] = transform_vertex(cam, in.pos[k][0], in.pos[k][1], in.pos[k][2]);
    float col[3];
    light_vertex(cam, in.nrm[k][0], in.nrm[k][1], in.nrm[k][2], in.mat[k], col);
    at[k].u = in.uv[k][0];
    at[k].v = in.uv[k][1];
    at[k].r = col[0];
    at[k].g = col[1];
    at[k].b = col[2];
  }
  return setup_triangle(hv[0], hv[1], hv[2], at[0], at[1], at[2], in.tex, W, H, out, cam.sample_ext);
}

// half `half` (fan (0,1,2) / (0,2,3)) of static quad q of env i
MWB_DEV bool room_triangle(const DevState& S, const RenderAssets& A, const mwb_quad* quads, int i, int q, int half,
                           TriInput& in) {
  const mwb_quad& Q = quads[q];   // this env's static quads: HBM/L2, or the TMA-staged shared-memory copy
  if (half == 1 && Q.num_verts < 4) return false;
  const int tex = S.room_tex[((size_t)i * S.R + Q.room) * 3 + Q.surf];
  const TexDev& T = A.tex[tex];
  // gen_texcs_wall / gen_texcs_floor: float64 multiply by TEX_DENSITY / size, then float32
  const double xc = 512.0 / (double)T.w, yc = 512.0 / (double)T.h;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int v = k == 0 ? 0 : k + half;
    in.pos[k][0] = Q.pos[v][0];
    in.pos[k][1] = Q.pos[v][1];
    in.pos[k][2] = Q.pos[v][2];
    in.uv[k][0] = (float)d_mul(Q.uvm[v][0], xc);
    in.uv[k][1] = (float)d_mul(Q.uvm[v][1], yc);
    in.nrm[k][0] = Q.nrm[0];
    in.nrm[k][1] = Q.nrm[1];
    in.nrm[k][2] = Q.nrm[2];
    in.mat[k][0] = in.mat[k][1] = in.mat[k][2] = 1.0f;   // glColor3f(1, 1, 1)
  }
  in.tex = tex;
  return true;
}

// cos / sin of an entity's model rotation.  glRotatef takes a GLfloat: the angle in degrees the reference forms in
// float64 -- `dir * (180 / math.pi)` for Box / ImageFrame / TextFrame (entity.py:206, 316, 421), `dir * 180 / math.pi`
// for MeshEnt (entity.py:158) -- reaches GL rounded to float32.  Spec: c, s = float32(cos / sin(float64(a32) * pi / 180)).
MWB_DEV void model_rotation(double dir, int mesh_form, float& c, float& s) {
  const double deg = mesh_form ? d_div(d_mul(dir, 180.0), 3.141592653589793) : d_mul(dir, 57.29577951308232);
  const double rad = d_div(d_mul((double)(float)deg, 3.141592653589793), 180.0);
  c = (float)mwb_libm::cos_glibc(rad);
  s = (float)mwb_libm::sin_glibc(rad);
}

// corner v (0..3) of face f of drawBox (opengl.py:460-503; faces +z, -z, -x, +x, +y, -y): which end of
// the box's x / z range (sign) and of its y range (top?) the vertex takes
MWB_DEV void box_corner(int f, int v, int& sx, int& top, int& sz) {
  const signed char X[6][4] = {{1, -1, -1, 1}, {-1, 1, 1, -1}, {-1, -1, -1, -1}, {1, 1, 1, 1}, {1, 1, -1, -1}, {1, 1, -1, -1}};
  const signed char Y[6][4] = {{1, 1, 0, 0}, {1, 1, 0, 0}, {1, 1, 0, 0}, {1, 1, 0, 0}, {1, 1, 1, 1}, {0, 0, 0, 0}};
  const signed char Z[6][4] = {{1, 1, 1, 1}, {-1, -1, -1, -1}, {1, -1, -1, 1}, {-1, 1, 1, -1}, {1, -1, -1, 1}, {-1, 1, 1, -1}};
  sx = X[f][v];
  top = Y[f][v];
  sz = Z[f][v];
}

// the angle model_rotation takes the cosine / sine of, for the Box / frame form of the degrees (see model_rotation)
MWB_DEV double box_rotation_angle(double dir) {
  const double deg = d_mul(dir, 57.29577951308232);
  return d_div(d_mul((double)(float)deg, 3.141592653589793), 180.0);
}

// triangle t (0..11) of a Box: face t / 2 in drawBox order, fan half t % 2.  cs: the box's (cos, sin) if the caller
// already has them (K2 evaluates every entity's pair once per frame, in parallel with the camera's), else null
MWB_DEV void box_triangle(const mwb_proto& pr, const EntPose& P, int t, TriInput& in, const float* cs = nullptr) {
  const int f = t >> 1, half = t & 1;
  const double ex = P.size > 0.0 ? P.size : pr.size[0], ey = P.size > 0.0 ? P.size : pr.size[1],
               ez = P.size > 0.0 ? P.size : pr.size[2];
  const float hx = (float)(ex / 2), sy = (float)ey, hz = (float)(ez / 2);
  const float NX[6] = {0, 0, -1, 1, 0, 0}, NY[6] = {0, 0, 0, 0, 1, -1}, NZ[6] = {1, -1, 0, 0, 0, 0};
  // glTranslatef(pos) * glRotatef(dir in degrees, 0, 1, 0): x' = x c + z s, z' = z c - x s
  float c, s;
  if (cs != nullptr) {
    c = cs[0];
    s = cs[1];
  } else {
    model_rotation(P.dir, 0, c, s);
  }
  const float tx = (float)P.x, ty = (float)P.y, tz = (float)P.z;
  const float nx = f_add(f_mul(NX[f], c), f_mul(NZ[f], s)), ny = NY[f], nz = f_sub(f_mul(NZ[f], c), f_mul(NX[f], s));
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int v = k == 0 ? 0 : k + half;
    int cx, top, cz;
    box_corner(f, v, cx, top, cz);
    const float x = cx > 0 ? hx : -hx, y = top ? sy : 0.0f, z = cz > 0 ? hz : -hz;
    in.pos[k][0] = f_add(f_add(f_mul(x, c), f_mul(z, s)), tx);
    in.pos[k][1] = f_add(y, ty);
    in.pos[k][2] = f_add(f_sub(f_mul(z, c), f_mul(x, s)), tz);
    in.uv[k][0] = in.uv[k][1] = 0.0f;
    in.nrm[k][0] = nx;
    in.nrm[k][1] = ny;
    in.nrm[k][2] = nz;
    for (int q = 0; q < 3; ++q) in.mat[k][q] = (float)P.col[q];
  }
  in.tex = -1;
}

// triangle t of a MeshEnt: glTranslatef(pos) glScalef(s) glRotatef(dir): v' = pos + s (R v);
// normals through the inverse transpose, R n / s, not renormalised (entity.py:150-161)
MWB_DEV void mesh_triangle(const RenderAssets& A, const mwb_proto& pr, const EntPose& P, float c, float s, int t,
                           TriInput& in) {
  const MeshDev& M = A.meshes[pr.mesh_id];
  const size_t base = (size_t)(M.first + t);
  const float sc = pr.scale, inv = f_div(1.0f, sc);
  const float tx = (float)P.x, ty = (float)P.y, tz = (float)P.z;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float* p = A.mesh_pos + (base * 3 + k) * 3;
    const float* n = A.mesh_nrm + (base * 3 + k) * 3;
    const float* m = A.mesh_rgb + (base * 3 + k) * 3;
    in.pos[k][0] = f_add(f_mul(f_add(f_mul(p[0], c), f_mul(p[2], s)), sc), tx);
    in.pos[k][1] = f_add(f_mul(p[1], sc), ty);
    in.pos[k][2] = f_add(f_mul(f_sub(f_mul(p[2], c), f_mul(p[0], s)), sc), tz);
    in.nrm[k][0] = (n[0] * c + n[2] * s) * inv;
    in.nrm[k][1] = n[1] * inv;
    in.nrm[k][2] = (n[2] * c - n[0] * s) * inv;
    in.uv[k][0] = A.mesh_uv[(base * 3 + k) * 2 + 0];
    in.uv[k][1] = A.mesh_uv[(base * 3 + k) * 2 + 1];
    in.mat[k][0] = m[0];
    in.mat[k][1] = m[1];
    in.mat[k][2] = m[2];
  }
  in.tex = A.mesh_tex[base];   // -1 for ball_* / key_* (no map_Kd, objmesh.py:226-230)
}

// Agent.render() (entity.py:518-539): a red triangle at the top of the agent's cylinder pointing along
// dir_vec; float64 vertex arithmetic as numpy evaluates it, rounded by glVertex3f.  It is untextured
// (every entity draw leaves GL_TEXTURE_2D disabled) and lit with GL's *current normal*, which the
// reference never sets here: it is whatever the previous draw left behind -- the last face normal of
// drawBox (0, -1, 0), or the last vertex normal of the last mesh / wall quad, in object space.
MWB_DEV void agent_triangle(const DevState& S, const RenderAssets& A, const FrameMap& m, const mwb_quad* quads, int i,
                            TriInput& in) {
  const size_t N = S.N;
  const int as = S.agent_slot[i];
  const mwb_proto& ap = S.protos[S.ent_proto[as * N + i]];
  const double px = S.ent_px[as * N + i], py = d_add(S.ent_py[as * N + i], ap.height), pz = S.ent_pz[as * N + i];
  const double d = S.ent_dir[as * N + i];
  const double c = mwb_libm::cos_glibc(d), s = mwb_libm::sin_glibc(d);
  const double r = ap.radius;
  const double dvx = d_mul(c, r), dvz = d_mul(-s, r);          // dir_vec * radius
  const double rvx = d_mul(s, r), rvz = d_mul(c, r);           // right_vec * radius
  double vx[3], vz[3];
  vx[0] = d_add(px, dvx);                                      // p0 = p + dv
  vz[0] = d_add(pz, dvz);
  vx[2] = d_add(px, d_mul(0.75, d_sub(rvx, dvx)));             // p1 = p + 0.75 (rv - dv)
  vz[2] = d_add(pz, d_mul(0.75, d_sub(rvz, dvz)));
  vx[1] = d_add(px, d_mul(0.75, d_sub(-rvx, dvx)));            // p2 = p + 0.75 (-rv - dv)
  vz[1] = d_add(pz, d_mul(0.75, d_sub(-rvz, dvz)));            // submitted as p0, p2, p1
  float n[3] = {0.0f, -1.0f, 0.0f};
  if (m.n_ents > 0 && m.ent_kind[m.n_ents - 1] == MWB_KIND_MESH) {
    const MeshDev& M = A.meshes[S.protos[m.ent_proto[m.n_ents - 1]].mesh_id];
    const float* q = A.mesh_nrm + ((size_t)(M.first + M.count - 1) * 3 + 2) * 3;
    n[0] = q[0]; n[1] = q[1]; n[2] = q[2];
  } else if (m.n_ents == 0 && m.n_quads > 0) {
    const mwb_quad& Q = quads[m.n_quads - 1];
    n[0] = Q.nrm[0]; n[1] = Q.nrm[1]; n[2] = Q.nrm[2];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    in.pos[k][0] = (float)vx[k];
    in.pos[k][1] = (float)py;
    in.pos[k][2] = (float)vz[k];
    in.uv[k][0] = in.uv[k][1] = 0.0f;
    in.nrm[k][0] = n[0]; in.nrm[k][1] = n[1]; in.nrm[k][2] = n[2];
    in.mat[k][0] = 1.0f; in.mat[k][1] = 0.0f; in.mat[k][2] = 0.0f;   // glColor3f(1, 0, 0)
  }
  in.tex = -1;
}

MWB_DEV const mwb_quad* env_quads(const DevState& S, int i) { return S.quads + (size_t)geom_index(S, i) * S.Q; }

// shared-memory triangle task -> (segment, record); false if culled / nonexistent
MWB_DEV bool task_triangle(const DevState& S, const RenderAssets& A, const Camera& cam, const FrameMap& m,
                           const mwb_quad* quads, int i, int task, int W, int H, TriRec& out, int& seg,
                           const float (*ent_cs)[2] = nullptr) {
  TriInput in;
  if (task < 2 * m.n_quads) {
    seg = 0;
    if (!room_triangle(S, A, quads, i, task >> 1, task & 1, in)) return false;
  } else if (task == m.agent_task) {
    seg = 1 + m.n_ents;
    agent_triangle(S, A, m, quads, i, in);
  } else {
    int k = 0;
    while (k + 1 < m.n_ents && (m.ent_task0[k] < 0 || task >= m.ent_task0[k] + 12)) ++k;
    seg = 1 + k;
    box_triangle(S.protos[m.ent_proto[k]], entity_pose(S, i, m.ent_slot[k]), task - m.ent_task0[k], in,
                 ent_cs != nullptr ? ent_cs[m.ent_slot[k]] : nullptr);
  }
  return finish_triangle(cam, in, W, H, out);
}

// one triangle list of a frame
struct Segment {
  const TriRec* tris;
  const uint2* bbox;                 // mesh lists: packed bboxes (coalesced pre-test); null for shared-memory lists
  const uint16_t* bin_idx;           // binned mesh lists: triangle indices per half-tile of the segment's box, or null
  const int* bin_off;
  int base, count;                   // slots [base, base + count)
  int bx, by;                        // bbox lo | hi << 16 (pixels)
};

struct SegLookup {                   // slot -> record
  const Segment* seg;
  int n;
  MWB_DEVM const TriRec& operator()(uint32_t slot) const {
    if ((int)slot < seg[0].count) return seg[0].tris[slot];   // room triangles: slot == position (the common case)
    int k = 1;
    while (k + 1 < n && (int)slot >= seg[k + 1].base) ++k;
    return seg[k].tris[(int)slot - seg[k].base];
  }
};

// per (env, entity slot) result of mesh_setup_kernel
struct MeshSegInfo {
  int count, bx, by;
  int binned;                        // 1: mesh_bin_off / mesh_bin_idx of this (env, slot) are valid for this frame
};

// Resolve one pixel: average the colour of the surface seen by each sample (box filter of
// the MSAA resolve blit), shading each distinct triangle once at the pixel centre.  The
// distinct-surface loop is deliberately not unrolled: one copy of the shading code.
template <int MSAA>
MWB_DEV uint32_t key_id(uint32_t key) { return key >= MWB_SKY_KEY ? 0xFFFFu : (key & 0xFFFFu); }

// exact depth code of triangle t at sample 0 of pixel (px, py) (lazy pixels: t is unclipped there)
template <int MSAA>
MWB_DEV uint32_t sample0_code(const TriRec& t, int px, int py) {
  const float xs = (float)px + sample_x<MSAA>(0), ys = (float)py + sample_y<MSAA>(0);
  const float z = f_add(f_add(f_mul(t.Za, xs), f_mul(t.Zb, ys)), t.Zc);
  return (uint32_t)f_add(f_mul(z, 65535.0f), 0.5f);
}

template <int MSAA, typename TriFetch>
MWB_DEV void resolve_pixel(const RenderAssets& A, const Camera& cam, const TriFetch& tris, const uint32_t (&keys)[MSAA],
                           int lazy_slot, int px, int py, uint8_t rgb[3]) {
  float acc[3] = {0.0f, 0.0f, 0.0f};
  const uint32_t all = (1u << MSAA) - 1u;
  uint32_t todo = lazy_slot >= 0 ? 1u : all;       // a lazy pixel is one surface on every sample: keys are not looked at
  const float wgt = 1.0f / (float)MSAA;
#pragma unroll 1
  while (todo) {
    uint32_t id = (uint32_t)lazy_slot, same = all;
    if (lazy_slot < 0) {
      // id of the first unprocessed sample (select chain: keys stay in registers)
      const uint32_t first = todo & (0u - todo);
      id = 0;
#pragma unroll
      for (int s = 0; s < MSAA; ++s)
        if (first == (1u << s)) id = key_id<MSAA>(keys[s]);
      same = 0;
#pragma unroll
      for (int s = 0; s < MSAA; ++s)
        if (key_id<MSAA>(keys[s]) == id) same |= 1u << s;
    }
    todo &= ~same;
    float c[3];
    if (id == 0xFFFFu) {
      c[0] = cam.sky[0];
      c[1] = cam.sky[1];
      c[2] = cam.sky[2];
    } else {
      shade_pixel(A, tris(id), px, py, c);
    }
#ifdef __CUDA_ARCH__
    const float f = (float)__popc(same) * wgt;
#else
    const float f = (float)__builtin_popcount(same) * wgt;
#endif
    acc[0] += f * c[0];
    acc[1] += f * c[1];
    acc[2] += f * c[2];
  }
  rgb[0] = to_unorm8(acc[0]);
  rgb[1] = to_unorm8(acc[1]);
  rgb[2] = to_unorm8(acc[2]);
}
