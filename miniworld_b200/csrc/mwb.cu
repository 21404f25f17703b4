// mwb.cu -- libmwb.so: the C ABI of include/mwb.h on top of the CUDA kernels.
//
//   step_kernel   (K1)  physics.cuh + reset.cuh   one warp per env
//   render_kernel (K2)  raster.cuh                one block per env, one warp per 8x8 tile
//   scatter / gather    host <-> SoA state exchange for host-generated worlds
//
// Built for sm_100a only.  The same file can be compiled by g++ with -DMWB_HOSTSIM into the
// test-only host simulator (tests/hostsim): there every "launch" is a plain loop over the
// identical MWB_DEV functions.  That build is a debugging aid for a box without a GPU; it is
// not part of libmwb.so and nothing in the package loads it.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/mwb.h"
#include "raster.cuh"
#include "visibility.cuh"
#include "reset.cuh"

#ifndef MWB_HOSTSIM
#include <cuda_runtime.h>
#endif

#define MWB_MAX_ENTS_CAP 32
#define MWB_STAGE_QUAD_BYTES_HOST 16384

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

// ------------------------------------------------------------------ memory space shims
#ifdef MWB_HOSTSIM
typedef void* stream_t;
static int dev_alloc(void** p, size_t n) {
  *p = calloc(1, n ? n : 1);
  return *p ? 0 : -1;
}
static void dev_free(void* p) { free(p); }
static int h2d(void* d, const void* h, size_t n, stream_t) { memcpy(d, h, n); return 0; }
static int d2h(void* h, const void* d, size_t n, stream_t) { memcpy(h, d, n); return 0; }
static int dev_memset(void* d, int v, size_t n) { memset(d, v, n); return 0; }
static int sync_stream(stream_t) { return 0; }
static bool is_device_ptr(const void*) { return false; }
#else
typedef cudaStream_t stream_t;
#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(MWB_ECUDA, std::string(#call) + " (mwb.cu:" + std::to_string(__LINE__) + "): " + cudaGetErrorString(e_)); \
  } while (0)
static int dev_alloc(void** p, size_t n) { return cudaMalloc(p, n ? n : 1) == cudaSuccess ? 0 : -1; }
static void dev_free(void* p) { cudaFree(p); }
static int h2d(void* d, const void* h, size_t n, stream_t s) {
  return cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s) == cudaSuccess ? 0 : -1;
}
static int d2h(void* h, const void* d, size_t n, stream_t s) {
  return cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s) == cudaSuccess ? 0 : -1;
}
static int dev_memset(void* d, int v, size_t n) { return cudaMemset(d, v, n) == cudaSuccess ? 0 : -1; }
static int sync_stream(stream_t s) { return cudaStreamSynchronize(s) == cudaSuccess ? 0 : -1; }
static bool is_device_ptr(const void* p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}
#endif

// ------------------------------------------------------------------ exchange records
struct WorldUpload {   // AoS image of one env's dynamic state (host <-> device staging)
  int32_t env, num_slots, agent_slot, carrying, step_count, num_picked, hold, pad1;
  double cam[4];
  double envp[12];
  mwb_entity ents[MWB_MAX_ENTS_CAP];
  mwb_rng_state rng;
};

#define MWB_DEFAULT_D2H_CHUNKS 16   // measured on B200 / PCIe 5: 4 -> 1.43 M, 8 -> 1.48 M, 16 -> 1.50 M env-steps/s end to end

struct mwb_handle {
  mwb_config cfg;
  DevState S;
  RenderAssets A;
  std::vector<void*> allocs;
  stream_t stream;
  int64_t launches;
  // staging
  int32_t* d_actions;
  double* d_step_params;
  double* d_reward;
  uint8_t* d_term;
  uint8_t* d_trunc;
  uint8_t* d_obs;
  int obs_format;                 // MWB_OBS_*: layout K2 writes observations in
  size_t obs_px_bytes;            // bytes per pixel of that layout (3, or 8 for float64 greyscale)
  size_t d_obs_bytes;             // capacity of the d_obs staging buffer
  float* d_depth;
  int32_t* d_ids;
  int* d_overflow;
  WorldUpload* d_upload;
  int tri_cap;
  bool smem_tris;
  int stage_bytes;
  bool have_params, have_protos, have_template;
  bool profiling;
  bool frames_copied;
  int obs_peer_hint;              // mwb_set_obs_peer: 1 / 0 = the caller says where observations go, -1 = look it up
  const void* peer_checked;       // last observation pointer whose home device was looked up, and the answer
  bool peer_result;
  bool obs_is_peer;               // this launch's observation buffer lives on another GPU (K2 stages whole frames)
  int k2_static_smem;             // static shared memory of the K2 instantiation in use (cudaFuncGetAttributes)
  TriRec* vis_tris;              // scratch of mwb_visible_ents, allocated on first use
  ViewSpec view;                 // what the next render launch draws (agent camera unless mwb_render_top_view)
  int k2_parts;                   // blocks per env frame (1 at 80x60, 4 at 160x120)
#ifndef MWB_HOSTSIM
  cudaStream_t copy_stream;
  cudaEvent_t chunk_done[MWB_DEFAULT_D2H_CHUNKS], copies_done;   // one per piece a host-destination frame batch is rendered + copied in
#endif
#ifndef MWB_HOSTSIM
  std::vector<cudaEvent_t> ev_k1, ev_k2;   // start/stop pairs
  // stream discipline: the last stream work on this handle's state was enqueued on, and an event recorded behind it
  cudaEvent_t last_done;
  cudaStream_t last_stream;
  bool last_valid;
#endif
#ifndef MWB_HOSTSIM
  struct AtlasEntry* atlas;                       // the (shared) texture atlas K2 gathers from, or null
#endif
  std::vector<int> mesh_counts;   // triangles per uploaded mesh (host copy)
  void* mesh_tris_buf;
  void* mesh_bbox_buf;
  void* mesh_bin_idx_buf;
  void* mesh_bin_off_buf;
  // asset storage
  void *tex_desc, *texels, *mesh_desc, *mesh_pos, *mesh_nrm, *mesh_uv, *mesh_rgb, *mesh_tex, *protos, *ops, *maze, *maze_cdf;
};

#ifndef MWB_HOSTSIM
struct AtlasEntry {
  int device;
  uint64_t hash;
  size_t texels;
  int refs;
  cudaArray_t arr;
  cudaTextureObject_t obj;
  float iw, ih;
  std::vector<float> ax, ay;       // [texture][level] position of texel (0, 0)
};
static std::vector<AtlasEntry*> g_atlases;
static void release_texture_objects(mwb_handle* h) {
  AtlasEntry* e = h->atlas;
  h->atlas = nullptr;
  if (!e || --e->refs > 0) return;
  for (size_t k = 0; k < g_atlases.size(); ++k)
    if (g_atlases[k] == e) g_atlases.erase(g_atlases.begin() + k);
  cudaDestroyTextureObject(e->obj);
  cudaFreeArray(e->arr);
  delete e;
}
#endif

template <typename T>
static int alloc_arr(mwb_handle* h, T** p, size_t count) {
  void* q = nullptr;
  if (dev_alloc(&q, count * sizeof(T)) != 0) return fail(MWB_ECUDA, "device allocation failed");
  dev_memset(q, 0, count * sizeof(T));
  h->allocs.push_back(q);
  *p = (T*)q;
  return 0;
}

// Stream discipline.  A handle's state arrays are touched by work on its own stream (set-up, state exchange,
// snapshots, resets without a stream argument) and on caller streams (step / render).  Every entry point that
// enqueues work calls stream_enter() first -- the new work waits for whatever was enqueued last on a DIFFERENT
// stream -- and stream_leave() when it is done enqueueing, so that e.g. a snapshot() after an asynchronous step() on a
// torch stream sees the finished step, and a step on another stream sees the finished reset.
#ifndef MWB_HOSTSIM
static int stream_enter(mwb_handle* h, stream_t s) {
  if (h->last_valid && h->last_stream != s) CK(cudaStreamWaitEvent(s, h->last_done, 0));
  return 0;
}
static int stream_leave(mwb_handle* h, stream_t s) {
  CK(cudaEventRecord(h->last_done, s));
  h->last_stream = s;
  h->last_valid = true;
  return 0;
}
#else
static int stream_enter(mwb_handle*, stream_t) { return 0; }
static int stream_leave(mwb_handle*, stream_t) { return 0; }
#endif

// ------------------------------------------------------------------ kernels / loops
// K1 runs an env's scalar logic on all 32 lanes of a warp with identical values (every store writes the same value).
// The read-modify-write sequences on per-env state (step counter, RNG stream, entity list edits) rely on the lanes
// not drifting apart between the loads and the stores: explicit warp barriers pin that down.
#ifdef __CUDA_ARCH__
#define MWB_WARP_SYNC() __syncwarp()
#else
#define MWB_WARP_SYNC()
#endif

MWB_DEV void step_one(const DevState& S, int i, const int32_t* actions, const double* step_params, double* reward,
                      uint8_t* term, uint8_t* trunc) {
  StepOut o;
  MWB_WARP_SYNC();
  const int nr = S.needs_reset[i];
  if (nr == 2 || (nr == 1 && S.autoreset)) {
    // "next-step" auto-reset: this step performs the reset instead of stepping.  nr == 2: the
    // host already uploaded the fresh world (mwb_set_world with hold = 1)
    if (nr == 1) device_reset(S, i);
    S.needs_reset[i] = 0;
    o.reward = 0.0;
    o.terminated = 0;
    o.truncated = 0;
  } else {
    int action = actions[i];
    if (S.act_noise) {            // wrapper.action() runs before env.step() draws its three parameters
      NpRng r = load_rng(S, i);
      if (!(rng_uniform(r, 0.0, 1.0) < S.act_prob)) action = S.act_random >= 0 ? S.act_random : (int)rng_integers(r, 6u);
      MWB_WARP_SYNC();
      store_rng(S, i, r);
      MWB_WARP_SYNC();
    }
    double fs, fd, ts;
    if (step_params) {
      fs = step_params[i * 3 + 0];
      fd = step_params[i * 3 + 1];
      ts = step_params[i * 3 + 2];
    } else if (S.domain_rand) {   // params.sample(rand, ...) x3, always, before the action is read
      NpRng r = load_rng(S, i);
      fs = rng_uniform(r, S.params.forward_step_lo, S.params.forward_step_rng);
      fd = rng_uniform(r, S.params.forward_drift_lo, S.params.forward_drift_rng);
      ts = rng_uniform(r, S.params.turn_step_lo, S.params.turn_step_rng);
      MWB_WARP_SYNC();
      store_rng(S, i, r);
      MWB_WARP_SYNC();
    } else {
      fs = S.params.forward_step;
      fd = S.params.forward_drift;
      ts = S.params.turn_step;
    }
    o = physics_step(S, i, action, fs, fd, ts);
    if (o.terminated || o.truncated) {
      if (S.autoreset) S.needs_reset[i] = 1;
#ifdef __CUDA_ARCH__
      if ((threadIdx.x & 31) == 0) atomicAdd(S.episodes_done, 1ull);
#else
      *S.episodes_done += 1ull;
#endif
    }
  }
  MWB_WARP_SYNC();
  if (reward) reward[i] = o.reward;
  if (term) term[i] = (uint8_t)o.terminated;
  if (trunc) trunc[i] = (uint8_t)o.truncated;
}

MWB_DEV void scatter_one(const DevState& S, const WorldUpload& u) {
  const size_t N = S.N;
  const int i = u.env;
  S.num_slots[i] = u.num_slots;
  S.agent_slot[i] = u.agent_slot;
  S.carrying[i] = u.carrying;
  S.step_count[i] = u.step_count;
  S.num_picked[i] = u.num_picked;
  S.needs_reset[i] = u.hold ? 2 : 0;
  S.ghost_slot[i] = -1;
  for (int k = 0; k < 4; ++k) S.cam[k * N + i] = u.cam[k];
  for (int k = 0; k < 12; ++k) S.envp[k * N + i] = u.envp[k];
  for (int e = 0; e < S.E; ++e) {
    const bool live = e < u.num_slots && e < MWB_MAX_ENTS_CAP;
    S.ent_proto[e * N + i] = live ? u.ents[e].proto : -1;
    S.ent_size[e * N + i] = 0.0;         // host-generated worlds carry each entity's own prototype
    if (!live) continue;
    S.ent_px[e * N + i] = u.ents[e].pos[0];
    S.ent_py[e * N + i] = u.ents[e].pos[1];
    S.ent_pz[e * N + i] = u.ents[e].pos[2];
    S.ent_dir[e * N + i] = u.ents[e].dir;
    for (int k = 0; k < 3; ++k) S.ent_col[((size_t)e * 3 + k) * N + i] = u.ents[e].color[k];
  }
  if (!S.shared_geom) {
    const mwb_room* rooms = S.rooms + (size_t)i * S.R;
    for (int r = 0; r < S.num_rooms[i]; ++r)
      for (int k = 0; k < 3; ++k) S.room_tex[((size_t)i * S.R + r) * 3 + k] = rooms[r].tex_id[k];
  } else {
    for (int r = 0; r < S.num_rooms[0]; ++r)
      for (int k = 0; k < 3; ++k) S.room_tex[((size_t)i * S.R + r) * 3 + k] = S.rooms[r].tex_id[k];
  }
}

MWB_DEV void gather_one(const DevState& S, int i, WorldUpload& u) {
  const size_t N = S.N;
  u.env = i;
  u.num_slots = S.num_slots[i];
  u.agent_slot = S.agent_slot[i];
  u.carrying = S.carrying[i];
  u.step_count = S.step_count[i];
  u.num_picked = S.num_picked[i];
  for (int k = 0; k < 4; ++k) u.cam[k] = S.cam[k * N + i];
  for (int k = 0; k < 12; ++k) u.envp[k] = S.envp[k * N + i];
  for (int e = 0; e < MWB_MAX_ENTS_CAP; ++e) {
    mwb_entity& d = u.ents[e];
    if (e >= S.E) {
      d.proto = -1;
      continue;
    }
    d.proto = S.ent_proto[e * N + i];
    d.pos[0] = S.ent_px[e * N + i];
    d.pos[1] = S.ent_py[e * N + i];
    d.pos[2] = S.ent_pz[e * N + i];
    d.dir = S.ent_dir[e * N + i];
    for (int k = 0; k < 3; ++k) d.color[k] = S.ent_col[((size_t)e * 3 + k) * N + i];
  }
  u.rng.state_hi = S.rng_s_hi[i];
  u.rng.state_lo = S.rng_s_lo[i];
  u.rng.inc_hi = S.rng_inc_hi[i];
  u.rng.inc_lo = S.rng_inc_lo[i];
  u.rng.has_uint32 = S.rng_has32[i];
  u.rng.uinteger = S.rng_cache[i];
}

#ifndef MWB_HOSTSIM
__global__ void step_kernel(DevState S, const int32_t* actions, const double* step_params, double* reward,
                            uint8_t* term, uint8_t* trunc) {
  int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per env (physics.cuh: circle_hits_walls)
  if (i < S.N) step_one(S, i, actions, step_params, reward, term, trunc);
}
__global__ void reset_kernel(DevState S, const int32_t* ids, int n) {
  int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per env
  if (t >= n) return;
  int i = ids ? ids[t] : t;
  device_reset(S, i);
  S.needs_reset[i] = 0;
}
__global__ void scatter_kernel(DevState S, const WorldUpload* u, int n) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) scatter_one(S, u[t]);
}
__global__ void gather_kernel(DevState S, WorldUpload* u) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S.N) gather_one(S, i, u[i]);
}
__global__ void seed_kernel(DevState S, const WorldUpload* u, int n) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  int i = u[t].env;
  S.rng_s_hi[i] = u[t].rng.state_hi;
  S.rng_s_lo[i] = u[t].rng.state_lo;
  S.rng_inc_hi[i] = u[t].rng.inc_hi;
  S.rng_inc_lo[i] = u[t].rng.inc_lo;
  S.rng_has32[i] = u[t].rng.has_uint32;
  S.rng_cache[i] = u[t].rng.uinteger;
}
#else
// host simulator: sequential stand-in for mesh_setup_kernel + render_kernel built from the
// same MWB_DEV functions
struct VecTris {
  const TriRec* t;
  const TriRec& operator()(uint32_t slot) const { return t[slot]; }
};
template <int MSAA>
static void hostsim_render_t(const DevState& S, const RenderAssets& A, const ViewSpec& view, uint8_t* obs, float* depth) {
  const int W = S.obs_w, H = S.obs_h;
  for (int i = 0; i < S.N; ++i) {
    Camera cam = view.mode == 1 ? make_top_camera(S, i, view) : make_camera(S, i);
    FrameMap fm = build_frame_map(S, i, view.mode == 1 && view.render_agent != 0);
    std::vector<TriRec> tris;
    TriRec rec;
    int seg;
    // Like K2, quads stay PAIRS in adjacent records (the culled half of a pair keeps an empty record) so that the
    // quad-pair logic of classify_pixel is exercised here too; `pairable[j]` marks records that belong to such a pair.
    std::vector<char> pairable;
    auto push_pair = [&](int task0) {
      TriRec a, b;
      int sg;
      const bool ka = task_triangle(S, A, cam, fm, env_quads(S, i), i, task0, W, H, a, sg);
      const bool kb = task_triangle(S, A, cam, fm, env_quads(S, i), i, task0 + 1, W, H, b, sg);
      if (!ka && !kb) return;
      if (tris.size() & 1) {               // pairs start at even positions (a mesh list may have left an odd count)
        TriRec e;
        empty_record(e);
        tris.push_back(e);
        pairable.push_back(0);
      }
      if (!ka) empty_record(a);
      if (!kb) empty_record(b);
      tris.push_back(a);
      tris.push_back(b);
      pairable.push_back(1);
      pairable.push_back(1);
    };
    for (int task = 0; task < 2 * fm.n_quads; task += 2) push_pair(task);
    for (int k = 0; k < fm.n_ents; ++k) {
      if (fm.ent_kind[k] == MWB_KIND_BOX) {
        for (int t = 0; t < 12; t += 2) push_pair(fm.ent_task0[k] + t);
      } else {
        const mwb_proto& pr = S.protos[fm.ent_proto[k]];
        const EntPose P = entity_pose(S, i, fm.ent_slot[k]);
        float c, s;
        model_rotation(P.dir, pr.deg_form, c, s);
        for (int t = 0; t < A.meshes[pr.mesh_id].count; ++t) {
          TriInput in;
          mesh_triangle(A, pr, P, c, s, t, in);
          if (finish_triangle(cam, in, W, H, rec)) {
            tris.push_back(rec);
            pairable.push_back(0);
          }
        }
      }
    }
    if (fm.agent_task >= 0 && task_triangle(S, A, cam, fm, env_quads(S, i), i, fm.agent_task, W, H, rec, seg)) {
      tris.push_back(rec);
      pairable.push_back(0);
    }
    // visit the triangles front to back by their nearest possible depth, as K2 does; slots keep draw order
    std::vector<int> order(tris.size());
    std::vector<float> zmin(tris.size());
    for (size_t j = 0; j < tris.size(); ++j) {
      const TriRec& t = tris[j];
      float x0 = (float)(t.bx & 0xFFFF), x1 = (float)((t.bx >> 16) + 1), y0 = (float)(t.by & 0xFFFF), y1 = (float)((t.by >> 16) + 1);
      zmin[j] = t.Zc + fminf(t.Za * x0, t.Za * x1) + fminf(t.Zb * y0, t.Zb * y1);
      order[j] = (int)j;
    }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return zmin[a] < zmin[b]; });
    VecTris fetch{tris.data()};
    for (int py = 0; py < H; ++py)
      for (int px = 0; px < W; ++px) {
        PixelState<MSAA> P;
        pixel_init(P);
        for (size_t jj = 0; jj < tris.size(); ++jj) {
          const int j = order[jj];
          const TriRec& t = tris[j];
          if ((t.bx & 0xFFFF) > px || (t.bx >> 16) < px || (t.by & 0xFFFF) > py || (t.by >> 16) < py) continue;
          const TriRec* partner = pairable[j] ? &tris[j ^ 1] : nullptr;
          if (classify_pixel<MSAA>(load_class(&t), j, px, py, P, partner, (j & 1) ? 1 : 2) == 0) continue;
          if (P.mode == MWB_PX_LAZY) {     // materialise the lazily held triangle (both halves of a lazily held pair) first
            raster_pixel<MSAA>(load_hot(&tris[P.lazy_slot]), P.lazy_slot, px, py, P.keys, P.kmax);
            if (lazy_is_pair(P)) raster_pixel<MSAA>(load_hot(&tris[P.lazy_slot ^ 1]), P.lazy_slot ^ 1, px, py, P.keys, P.kmax);
          }
          P.mode = MWB_PX_EXPLICIT;
          raster_pixel<MSAA>(load_hot(&t), j, px, py, P.keys, P.kmax);
          P.bound = (float)(P.kmax >> 16);
        }
        uint32_t code0;
        if (P.mode == MWB_PX_LAZY) {
          const TriRec& t = tris[P.lazy_slot];
          float c[3];
          shade_pixel(A, t, px, py, c);
          uint8_t rgb[3] = {to_unorm8(c[0]), to_unorm8(c[1]), to_unorm8(c[2])};
          if (obs) memcpy(obs + (((size_t)i * H + py) * W + px) * 3, rgb, 3);
          int owner = P.lazy_slot;
          if (lazy_is_pair(P)) {           // which half of the quad owns sample 0: its diagonal edge decides
            const float xs = (float)px + sample_x<MSAA>(0), ys = (float)py + sample_y<MSAA>(0);
            if (!pair_sample_in_first(t, (P.lazy_slot & 1) ? 1 : 2, xs, ys)) owner = P.lazy_slot ^ 1;
          }
          code0 = sample0_code<MSAA>(tris[owner], px, py);
        } else {
          if (obs) {
            uint8_t rgb[3];
            resolve_pixel<MSAA>(A, cam, fetch, P.keys, -1, px, py, rgb);
            memcpy(obs + (((size_t)i * H + py) * W + px) * 3, rgb, 3);
          }
          code0 = P.keys[0] >> 16;
        }
        if (depth) depth[((size_t)i * H + py) * W + px] = depth_code_to_metres(code0);
      }
  }
}
static void hostsim_render(const DevState& S, const RenderAssets& A, const ViewSpec& view, int fmt, uint8_t* obs_out, float* depth) {
  // other layouts: render HWC into a scratch frame set, then apply the same per-pixel conversion K2's epilogue does
  const size_t px = (size_t)S.obs_w * S.obs_h;
  std::vector<uint8_t> tmp;
  uint8_t* obs = obs_out;
  if (obs_out && fmt != MWB_OBS_HWC_U8) {
    tmp.resize((size_t)S.N * px * 3);
    obs = tmp.data();
  }
  if (S.msaa == 1) hostsim_render_t<1>(S, A, view, obs, depth);
  else if (S.msaa == 16) hostsim_render_t<16>(S, A, view, obs, depth);
  else if (S.msaa == 4) hostsim_render_t<4>(S, A, view, obs, depth);
  else hostsim_render_t<8>(S, A, view, obs, depth);
  if (obs_out && fmt != MWB_OBS_HWC_U8) {
    const int W = S.obs_w, H = S.obs_h;
    for (int i = 0; i < S.N; ++i)
      for (int y = 0; y < H; ++y)
        for (int x = 0; x < W; ++x) {
          const uint8_t* c = obs + (((size_t)i * H + y) * W + x) * 3;
          if (fmt == MWB_OBS_CWH_U8) {
            for (int k = 0; k < 3; ++k) obs_out[(((size_t)i * 3 + k) * W + x) * H + y] = c[k];
          } else {
            reinterpret_cast<double*>(obs_out)[((size_t)i * H + y) * W + x] = grey_f64(c[0], c[1], c[2]);
          }
        }
  }
}
#endif

#ifndef MWB_HOSTSIM
// K2's dynamic shared memory: [triangle records] [staged static quads] [visit order + depth keys] [frame stage].
// The frame stage holds one env's whole RGB frame (80x60: 14.4 KB) so that it leaves the SM as full 16-byte
// row-contiguous stores -- what makes the peer-memory observation path efficient over NVLink (8-byte
// scattered segments reach ~190 GB/s into one GPU, 128-byte lines several times that).
static int k2_list_bytes(const mwb_handle* h) {
  const K2Layout L = k2_layout(h->smem_tris, h->tri_cap, h->stage_bytes, k2_halves_per_part(h->S.obs_w, h->S.obs_h, h->k2_parts), 0);
  return (int)L.stage_off;
}
static int k2_frame_stage_bytes(const mwb_handle* h) {
  const int W = h->S.obs_w, H = h->S.obs_h, tiles_x = (W + 7) >> 3;
  // bytes one block stages: the whole frame, or (frames cut into several blocks) its band of whole half-tile rows
  const size_t rows = h->k2_parts == 1 ? (size_t)H : (size_t)(k2_halves_per_part(W, H, h->k2_parts) / tiles_x) * 4;
  const size_t bytes = rows * W * 3;
  if (h->obs_format == MWB_OBS_GREY_F64 || bytes > 16384 || (bytes & 15) != 0 || (W & 7) != 0) return 0;
  if (h->k2_parts != 1 && (h->obs_format != MWB_OBS_HWC_U8 || (H & 3) != 0)) return 0;
  // Staging pays only when the stores leave the GPU (peer memory of rank 0: full 16-byte address-ordered stores
  // instead of 8-byte row segments, 52 % -> 89 % weak-scaling efficiency on 8 GPUs); for local HBM it costs 6 %.
  if (!h->obs_is_peer) return 0;
  // not at the price of a resident block: three blocks per SM (+ 1 KB each for the system) must still fit in 227 KB
  const size_t per_block = (size_t)k2_list_bytes(h) + bytes + (size_t)h->k2_static_smem + 1024;
  if (3 * per_block > 232448) return 0;
  return (int)bytes;      // a multiple of 16: every band starts 16-byte aligned
}
static int k2_smem_bytes(const mwb_handle* h) { return k2_list_bytes(h) + k2_frame_stage_bytes(h); }

// K2's instantiation for a sample count (1, 4, 8 or 16)
static decltype(&render_kernel<8>) k2_kernel(int msaa) {
  switch (msaa) {
    case 1: return render_kernel<1>;
    case 4: return render_kernel<4>;
    case 16: return render_kernel<16>;
    default: return render_kernel<8>;
  }
}

// The opt-in for large dynamic shared memory is an attribute of the kernel FUNCTION (per device), not of a
// handle: several handles with different triangle capacities share it, so it is only ever raised.
static int g_k2_smem[16] = {};
static int ensure_k2_smem(mwb_handle* h, int smem) {
  const int dev = h->cfg.device & 15;
  if (smem <= g_k2_smem[dev]) return 0;
  for (int msaa : {1, 4, 8, 16})
    if (cudaFuncSetAttribute(k2_kernel(msaa), cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -1;
  g_k2_smem[dev] = smem;
  return 0;
}
#endif

// ------------------------------------------------------------------ ABI: lifetime
extern "C" const char* mwb_last_error(void) { return g_err.c_str(); }

extern "C" int mwb_create(const mwb_config* cfg, mwb_handle** out) {
  if (!cfg || !out) return fail(MWB_EINVAL, "null argument");
  if (cfg->abi_version != MWB_ABI_VERSION) return fail(MWB_EABI, "abi_version mismatch");
  if (cfg->num_envs <= 0 || cfg->obs_width <= 0 || cfg->obs_height <= 0) return fail(MWB_EINVAL, "bad sizes");
  if (cfg->msaa_samples != 1 && cfg->msaa_samples != 4 && cfg->msaa_samples != 8 && cfg->msaa_samples != 16)
    return fail(MWB_EINVAL, "msaa_samples must be 1, 4, 8 or 16");
  if (cfg->max_ents <= 0 || cfg->max_ents > MWB_MAX_ENTS_CAP) return fail(MWB_ECAPACITY, "max_ents out of range");
  if (cfg->max_rooms <= 0 || cfg->max_quads <= 0 || cfg->max_segs <= 0) return fail(MWB_EINVAL, "bad capacities");
#ifndef MWB_HOSTSIM
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(MWB_ENOCUDA, "no CUDA device: libmwb has no CPU execution path");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return fail(MWB_EINVAL, "bad device ordinal");
  CK(cudaSetDevice(cfg->device));
#endif
  mwb_handle* h = new mwb_handle();
  h->cfg = *cfg;
  h->launches = 0;
  h->profiling = false;
  h->frames_copied = false;
  h->have_params = h->have_protos = h->have_template = false;
#ifndef MWB_HOSTSIM
  h->atlas = nullptr;
#endif
  h->tex_desc = h->texels = h->mesh_desc = h->mesh_pos = h->mesh_nrm = h->mesh_uv = h->mesh_rgb = h->mesh_tex = nullptr;
  h->protos = h->ops = h->maze = h->maze_cdf = nullptr;
  h->mesh_tris_buf = nullptr;
  h->mesh_bbox_buf = nullptr;
  h->mesh_bin_idx_buf = h->mesh_bin_off_buf = nullptr;
  memset(&h->view, 0, sizeof(ViewSpec));
  h->vis_tris = nullptr;
  h->obs_format = MWB_OBS_HWC_U8;
  h->obs_px_bytes = 3;
  h->obs_peer_hint = -1;
  h->peer_checked = nullptr;
  h->peer_result = h->obs_is_peer = false;
  h->k2_static_smem = 19456;
  memset(&h->S, 0, sizeof(DevState));
  memset(&h->A, 0, sizeof(RenderAssets));
#ifndef MWB_HOSTSIM
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return fail(MWB_ECUDA, "cudaStreamCreate failed");
  }
  for (int c = 0; c < MWB_DEFAULT_D2H_CHUNKS; ++c) cudaEventCreateWithFlags(&h->chunk_done[c], cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->copies_done, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&h->last_done, cudaEventDisableTiming);
  h->last_stream = h->stream;
  h->last_valid = false;
#else
  h->stream = nullptr;
#endif
  DevState& S = h->S;
  const size_t N = cfg->num_envs, E = cfg->max_ents;
  S.N = cfg->num_envs;
  S.E = cfg->max_ents;
  S.R = cfg->max_rooms;
  S.Q = (cfg->max_quads + 1) & ~1;   // even: per-env quad blocks stay 16-byte aligned (TMA source)
  S.S = cfg->max_segs;
  S.shared_geom = cfg->shared_geometry;
  S.obs_w = cfg->obs_width;
  S.obs_h = cfg->obs_height;
  S.msaa = cfg->msaa_samples;
  S.rule_kind = cfg->rule_kind;
  S.rule_arg = cfg->rule_arg;
  S.domain_rand = cfg->domain_rand;
  S.max_episode_steps = cfg->max_episode_steps;
  S.autoreset = cfg->autoreset;
  const size_t G = cfg->shared_geometry ? 1 : N;
  int rc = 0;
#define AL(field, count) if (!rc) rc = alloc_arr(h, &S.field, (count))
  AL(ent_proto, E * N); AL(ent_px, E * N); AL(ent_py, E * N); AL(ent_pz, E * N); AL(ent_dir, E * N);
  AL(ent_col, E * 3 * N); AL(ent_size, E * N); AL(num_slots, N); AL(agent_slot, N); AL(carrying, N); AL(step_count, N);
  AL(num_picked, N); AL(needs_reset, N); AL(episodes_done, 1); AL(cam, 4 * N); AL(envp, 12 * N); AL(ghost_slot, N);
  AL(ghost_proto, N); AL(ghost_pose, 4 * N); AL(ghost_col, 3 * N);
  AL(rng_s_hi, N); AL(rng_s_lo, N); AL(rng_inc_hi, N); AL(rng_inc_lo, N); AL(rng_has32, N); AL(rng_cache, N);
  AL(num_rooms, G); AL(num_quads, G); AL(num_segs, G);
  AL(rooms, G * S.R); AL(quads, G * S.Q + 2); AL(segs, G * S.S); AL(room_tex, N * S.R * 3);
  AL(mesh_seg, N * E); AL(cam_trig, 6 * N); AL(ent_cs, E * 2 * N);
#undef AL
  if (!rc) rc = alloc_arr(h, &h->d_actions, N);
  if (!rc) rc = alloc_arr(h, &h->d_step_params, 3 * N);
  if (!rc) rc = alloc_arr(h, &h->d_reward, N);
  if (!rc) rc = alloc_arr(h, &h->d_term, N);
  if (!rc) rc = alloc_arr(h, &h->d_trunc, N);
  if (!rc) rc = alloc_arr(h, &h->d_obs, N * (size_t)S.obs_w * S.obs_h * 3);
  h->d_obs_bytes = N * (size_t)S.obs_w * S.obs_h * 3;
  if (!rc) rc = alloc_arr(h, &h->d_depth, N * (size_t)S.obs_w * S.obs_h);
  if (!rc) rc = alloc_arr(h, &h->d_ids, N);
  if (!rc) rc = alloc_arr(h, &h->d_overflow, 1);
  S.fault = h->d_overflow;
  if (!rc) rc = alloc_arr(h, &h->d_upload, N);
  if (rc) {
    mwb_destroy(h);
    return rc;
  }
#ifndef MWB_HOSTSIM
  {
    float* lut = nullptr;
    if (alloc_arr(h, &lut, 65536)) {
      mwb_destroy(h);
      return fail(MWB_ECUDA, "depth table allocation failed");
    }
    depth_lut_kernel<<<256, 256, 0, h->stream>>>(lut);
    h->launches++;
    S.depth_lut = lut;
  }
#endif
  // -1 in every entity slot / ghost
  dev_memset(S.ent_proto, 0xFF, E * N * sizeof(int32_t));
  dev_memset(S.ghost_slot, 0xFF, N * sizeof(int32_t));
  dev_memset(S.carrying, 0xFF, N * sizeof(int32_t));
  // every room quad and box face can yield two set-up triangles.  Up to 512 of them live in
  // shared memory; larger levels (Maze) keep the per-env lists in HBM instead.
  {
    // blocks per env frame: at least one per 150 half-tiles (80x60 -> 1, 160x120 -> 4), and more
    // when few envs are resident so that the grid still covers ~4 waves of the 148 x 3 block
    // slots (each part redoes the cheap geometry phase); never fewer than 30 half-tiles per part
    const int halves = ((cfg->obs_width + 7) / 8) * ((cfg->obs_height + 3) / 4);
    const int base = (halves + 149) / 150, want = (1776 + cfg->num_envs - 1) / cfg->num_envs;
    const int maxp = halves / 30 > 1 ? halves / 30 : 1;
    h->k2_parts = base > want ? base : want;
    if (h->k2_parts > maxp) h->k2_parts = maxp;
    if (h->k2_parts < 1) h->k2_parts = 1;
  }
  h->tri_cap = 2 * (cfg->max_quads + 6 * cfg->max_ents) + 2;   // + the top view's agent marker
  h->smem_tris = h->tri_cap <= 512;
  if (!h->smem_tris) {
    TriRec* buf = nullptr;
    if (alloc_arr(h, &buf, (size_t)N * h->k2_parts * h->tri_cap)) {
      mwb_destroy(h);
      return fail(MWB_ECUDA, "triangle list allocation failed");
    }
    S.room_tris = buf;
  }
  // static quads are staged in shared memory (TMA bulk copy) when they fit in 16 KB; the
  // quad capacity is kept even so that every env's block starts 16-byte aligned
  h->stage_bytes = (int)(((size_t)cfg->max_quads * sizeof(mwb_quad) + 15) & ~(size_t)15);
  if (h->stage_bytes > MWB_STAGE_QUAD_BYTES_HOST) h->stage_bytes = 0;
#ifndef MWB_HOSTSIM
  {
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, k2_kernel(S.msaa)) == cudaSuccess) {
      h->k2_static_smem = (int)fa.sharedSizeBytes;
    } else {
      cudaGetLastError();
      h->k2_static_smem = 19456;
    }
  }
  const int smem = k2_smem_bytes(h) + 16384;     // room for a frame stage whatever observation layout is chosen later
  if (ensure_k2_smem(h, smem)) {
    mwb_destroy(h);
    return fail(MWB_ECUDA, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed");
  }
  if (getenv("MWB_DEBUG")) {
    const int launch_smem = k2_smem_bytes(h);
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k2_kernel(S.msaa), MWB_K2_THREADS, launch_smem);
    fprintf(stderr, "[mwb] K2 %d threads, %dx MSAA: dynamic smem %d B (local destination), parts %d, resident blocks/SM %d\n",
            MWB_K2_THREADS, S.msaa, launch_smem, h->k2_parts, nb);
  }
#endif
  *out = h;
  return MWB_OK;
}

extern "C" int mwb_destroy(mwb_handle* h) {
  if (!h) return MWB_OK;
#ifndef MWB_HOSTSIM
  cudaSetDevice(h->cfg.device);
  if (h->last_valid) cudaStreamSynchronize(h->last_stream);   // work still running on a caller stream uses these buffers
  cudaStreamSynchronize(h->stream);
#endif
  for (void* p : h->allocs) dev_free(p);
  void* extra[] = {h->tex_desc, h->texels, h->mesh_desc, h->mesh_pos, h->mesh_nrm, h->mesh_uv, h->mesh_rgb, h->mesh_tex,
                   h->protos, h->ops, h->mesh_tris_buf, h->mesh_bbox_buf, h->mesh_bin_idx_buf, h->mesh_bin_off_buf,
                   h->maze, h->maze_cdf};
  for (void* p : extra)
    if (p) dev_free(p);
#ifndef MWB_HOSTSIM
  release_texture_objects(h);
  cudaStreamSynchronize(h->copy_stream);
  for (cudaEvent_t e : h->ev_k1) cudaEventDestroy(e);
  for (cudaEvent_t e : h->ev_k2) cudaEventDestroy(e);
  for (int c = 0; c < MWB_DEFAULT_D2H_CHUNKS; ++c) cudaEventDestroy(h->chunk_done[c]);
  cudaEventDestroy(h->copies_done);
  cudaEventDestroy(h->last_done);
  cudaStreamDestroy(h->copy_stream);
  cudaStreamDestroy(h->stream);
#endif
  delete h;
  return MWB_OK;
}

extern "C" int64_t mwb_launch_count(mwb_handle* h) { return h ? h->launches : 0; }

extern "C" int64_t mwb_overflow_count(mwb_handle* h) {
  if (!h) return 0;
  int v = 0;
  if (stream_enter(h, h->stream)) return -1;
  if (d2h(&v, h->d_overflow, sizeof(int), h->stream) != 0 || sync_stream(h->stream) != 0) return -1;
  return v;
}
extern "C" int mwb_abi_sizes(int32_t* out, int cap) {
  const int32_t sz[] = {(int32_t)sizeof(mwb_config), (int32_t)sizeof(mwb_params), (int32_t)sizeof(mwb_tex_desc),
                        (int32_t)sizeof(mwb_mesh_desc), (int32_t)sizeof(mwb_room), (int32_t)sizeof(mwb_quad),
                        (int32_t)sizeof(mwb_seg), (int32_t)sizeof(mwb_proto), (int32_t)sizeof(mwb_entity),
                        (int32_t)sizeof(mwb_op), (int32_t)sizeof(mwb_geometry), (int32_t)sizeof(mwb_world),
                        (int32_t)sizeof(mwb_rng_state), (int32_t)sizeof(mwb_state_view), (int32_t)sizeof(mwb_maze_desc)};
  const int n = (int)(sizeof(sz) / sizeof(sz[0]));
  for (int k = 0; k < n && k < cap; ++k) out[k] = sz[k];
  return n;
}

static int replace_buf(void** slot, const void* host, size_t bytes, stream_t s) {
  if (*slot) dev_free(*slot);
  *slot = nullptr;
  if (dev_alloc(slot, bytes) != 0) return fail(MWB_ECUDA, "device allocation failed");
  if (bytes && h2d(*slot, host, bytes, s) != 0) return fail(MWB_ECUDA, "upload failed");
  return sync_stream(s) == 0 ? 0 : fail(MWB_ECUDA, "sync failed");
}

#ifndef MWB_HOSTSIM
// Atlas for K2's tld4 path: every mip level of every texture in ONE 2-D CUDA array (so that the texture handle is
// the same for every lane whatever surface / LOD its pixel needs), each level framed by a one-texel wrapped border.
// Shelf packing, tallest first; width 4096, height the next power of two.  Atlases are shared between the handles of
// a process (keyed by device + a hash of the texel pool): building one costs ~0.1-0.5 s.  Returns null when the
// atlas would be taller than 32768 rows or a CUDA call fails; K2 then reads the texel pool instead (the path the
// host simulator always takes).
static AtlasEntry* build_atlas(int device, const std::vector<TexDev>& td, const std::vector<uint32_t>& pool) {
  const int n = (int)td.size();
  uint64_t hash = 1469598103934665603ull;
  auto mix = [&hash](uint64_t v) { hash = (hash ^ v) * 1099511628211ull; };
  mix((uint64_t)n);
  for (int t = 0; t < n; ++t) { mix((uint64_t)td[t].w << 32 | (uint32_t)td[t].h); mix((uint64_t)td[t].nlev); }
  for (size_t k = 0; k + 1 < pool.size(); k += 2) mix((uint64_t)pool[k] << 32 | pool[k + 1]);
  for (AtlasEntry* c : g_atlases)
    if (c->device == device && c->hash == hash && c->texels == pool.size()) return c;
  struct Item { int t, l, w, hgt; };
  std::vector<Item> items;
  for (int t = 0; t < n; ++t)
    for (int l = 0; l < td[t].nlev; ++l) items.push_back({t, l, td[t].lw[l] + 2, td[t].lh[l] + 2});
  std::stable_sort(items.begin(), items.end(), [](const Item& a, const Item& b) { return a.hgt > b.hgt; });
  const int AW = 4096;
  int cx = 0, cy = 0, shelf = 0;
  std::vector<std::pair<int, int>> at(items.size());
  for (size_t k = 0; k < items.size(); ++k) {
    if (cx + items[k].w > AW) { cx = 0; cy += shelf; shelf = 0; }
    at[k] = {cx, cy};
    cx += items[k].w;
    shelf = std::max(shelf, items[k].hgt);
  }
  int AH = 1;
  while (AH < cy + shelf) AH <<= 1;
  if (AH > 32768) return nullptr;
  AtlasEntry* e = new AtlasEntry();
  e->device = device;
  e->hash = hash;
  e->texels = pool.size();
  e->refs = 0;
  e->arr = nullptr;
  e->obj = 0;
  e->ax.assign((size_t)n * MWB_MAX_LEVELS, 0.0f);
  e->ay.assign((size_t)n * MWB_MAX_LEVELS, 0.0f);
  std::vector<uint32_t> atlas((size_t)AW * AH, 0u);
  for (size_t k = 0; k < items.size(); ++k) {
    const Item& it = items[k];
    const int lw = it.w - 2, lh = it.hgt - 2;
    const uint32_t* src = pool.data() + td[it.t].off[it.l];
    for (int y = -1; y <= lh; ++y) {
      uint32_t* dst = &atlas[(size_t)(at[k].second + 1 + y) * AW + at[k].first];
      const uint32_t* row = src + (size_t)((y + lh) % lh) * lw;
      dst[0] = row[lw - 1];
      memcpy(dst + 1, row, (size_t)lw * 4);
      dst[lw + 1] = row[0];
    }
    e->ax[(size_t)it.t * MWB_MAX_LEVELS + it.l] = (float)(at[k].first + 1);
    e->ay[(size_t)it.t * MWB_MAX_LEVELS + it.l] = (float)(at[k].second + 1);
  }
  const cudaChannelFormatDesc fmt = cudaCreateChannelDesc<uchar4>();
  bool ok = cudaMallocArray(&e->arr, &fmt, AW, AH, cudaArrayTextureGather) == cudaSuccess;
  if (ok) ok = cudaMemcpy2DToArray(e->arr, 0, 0, atlas.data(), (size_t)AW * 4, (size_t)AW * 4, AH, cudaMemcpyHostToDevice) == cudaSuccess;
  if (ok) {
    cudaResourceDesc rd;
    memset(&rd, 0, sizeof(rd));
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = e->arr;
    cudaTextureDesc tdesc;
    memset(&tdesc, 0, sizeof(tdesc));
    tdesc.addressMode[0] = tdesc.addressMode[1] = cudaAddressModeClamp;
    tdesc.filterMode = cudaFilterModePoint;
    tdesc.readMode = cudaReadModeNormalizedFloat;
    tdesc.normalizedCoords = 1;
    ok = cudaCreateTextureObject(&e->obj, &rd, &tdesc, nullptr) == cudaSuccess;
  }
  if (!ok) {
    cudaGetLastError();
    if (e->arr) cudaFreeArray(e->arr);
    delete e;
    return nullptr;
  }
  e->iw = 1.0f / (float)AW;
  e->ih = 1.0f / (float)AH;
  g_atlases.push_back(e);
  return e;
}
#endif

// ------------------------------------------------------------------ ABI: assets
extern "C" int mwb_upload_textures(mwb_handle* h, const mwb_tex_desc* descs, int n, const uint8_t* rgb) {
  if (!h || !descs || n <= 0 || !rgb) return fail(MWB_EINVAL, "bad arguments");
  std::vector<TexDev> td(n);
  std::vector<uint32_t> pool;
  for (int t = 0; t < n; ++t) {
    int w = descs[t].width, hgt = descs[t].height;
    if (w <= 0 || hgt <= 0) return fail(MWB_EINVAL, "bad texture size");
    const uint8_t* src = rgb + descs[t].offset;
    // level 0: flip rows so that row 0 is the image bottom (pyglet uploads bottom-up)
    std::vector<uint32_t> cur((size_t)w * hgt);
    for (int y = 0; y < hgt; ++y)
      for (int x = 0; x < w; ++x) {
        const uint8_t* p = src + ((size_t)(hgt - 1 - y) * w + x) * 3;
        cur[(size_t)y * w + x] = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | 0xFF000000u;
      }
    TexDev& T = td[t];
    T.w = w;
    T.h = hgt;
    T.pad = 0;
    int lev = 0;
    for (;;) {
      T.lw[lev] = w;
      T.lh[lev] = hgt;
      T.off[lev] = (int32_t)pool.size();
      pool.insert(pool.end(), cur.begin(), cur.end());
      ++lev;
      if ((w == 1 && hgt == 1) || lev == MWB_MAX_LEVELS) break;
      // glGenerateMipmap: 2x2 box filter on the 8-bit texels; odd sizes halve with floor and
      // clamp the second tap to the last row / column
      int nw = w > 1 ? w / 2 : 1, nh = hgt > 1 ? hgt / 2 : 1;
      std::vector<uint32_t> nxt((size_t)nw * nh);
      for (int y = 0; y < nh; ++y)
        for (int x = 0; x < nw; ++x) {
          int x0 = w > 1 ? 2 * x : 0, x1 = w > 1 ? (2 * x + 1 < w ? 2 * x + 1 : w - 1) : 0;
          int y0 = hgt > 1 ? 2 * y : 0, y1 = hgt > 1 ? (2 * y + 1 < hgt ? 2 * y + 1 : hgt - 1) : 0;
          uint32_t a = cur[(size_t)y0 * w + x0], b = cur[(size_t)y0 * w + x1];
          uint32_t c = cur[(size_t)y1 * w + x0], d = cur[(size_t)y1 * w + x1];
          uint32_t o = 0xFF000000u;
          for (int k = 0; k < 3; ++k) {
            uint32_t s = ((a >> (8 * k)) & 255u) + ((b >> (8 * k)) & 255u) + ((c >> (8 * k)) & 255u) + ((d >> (8 * k)) & 255u);
            o |= ((s + 2u) >> 2) << (8 * k);
          }
          nxt[(size_t)y * nw + x] = o;
        }
      cur.swap(nxt);
      w = nw;
      hgt = nh;
    }
    T.nlev = lev;
  }
#ifndef MWB_HOSTSIM
  release_texture_objects(h);
  h->A.atlas = 0ull;
  if (AtlasEntry* e = build_atlas(h->cfg.device, td, pool)) {
    e->refs++;
    h->atlas = e;
    for (int t = 0; t < n; ++t)
      for (int l = 0; l < td[t].nlev; ++l) {
        td[t].ax[l] = e->ax[(size_t)t * MWB_MAX_LEVELS + l];
        td[t].ay[l] = e->ay[(size_t)t * MWB_MAX_LEVELS + l];
      }
    h->A.atlas = (unsigned long long)e->obj;
    h->A.atlas_iw = e->iw;
    h->A.atlas_ih = e->ih;
  }
#endif
  int rc = replace_buf(&h->tex_desc, td.data(), td.size() * sizeof(TexDev), h->stream);
  if (!rc) rc = replace_buf(&h->texels, pool.data(), pool.size() * sizeof(uint32_t), h->stream);
  if (rc) return rc;
  h->A.tex = (const TexDev*)h->tex_desc;
  h->A.texels = (const uint32_t*)h->texels;
  h->A.num_tex = n;
  return MWB_OK;
}

extern "C" int mwb_upload_meshes(mwb_handle* h, const mwb_mesh_desc* descs, int n, const float* pos, const float* nrm,
                                 const float* uv, const float* rgb, const int32_t* tri_tex) {
  if (!h || !descs || n <= 0) return fail(MWB_EINVAL, "bad arguments");
  std::vector<MeshDev> md(n);
  size_t total = 0;
  h->mesh_counts.assign(n, 0);
  for (int m = 0; m < n; ++m) {
    md[m].first = (int32_t)descs[m].offset;
    md[m].count = descs[m].num_tris;
    h->mesh_counts[m] = descs[m].num_tris;
    size_t end = (size_t)descs[m].offset + descs[m].num_tris;
    if (end > total) total = end;
  }
  int rc = replace_buf(&h->mesh_desc, md.data(), md.size() * sizeof(MeshDev), h->stream);
  if (!rc) rc = replace_buf(&h->mesh_pos, pos, total * 9 * sizeof(float), h->stream);
  if (!rc) rc = replace_buf(&h->mesh_nrm, nrm, total * 9 * sizeof(float), h->stream);
  if (!rc) rc = replace_buf(&h->mesh_uv, uv, total * 6 * sizeof(float), h->stream);
  if (!rc) rc = replace_buf(&h->mesh_rgb, rgb, total * 9 * sizeof(float), h->stream);
  std::vector<int32_t> none;
  if (!tri_tex) {
    none.assign(total, -1);
    tri_tex = none.data();
  }
  if (!rc) rc = replace_buf(&h->mesh_tex, tri_tex, total * sizeof(int32_t), h->stream);
  if (rc) return rc;
  h->A.mesh_tex = (const int32_t*)h->mesh_tex;
  h->A.meshes = (const MeshDev*)h->mesh_desc;
  h->A.mesh_pos = (const float*)h->mesh_pos;
  h->A.mesh_nrm = (const float*)h->mesh_nrm;
  h->A.mesh_uv = (const float*)h->mesh_uv;
  h->A.mesh_rgb = (const float*)h->mesh_rgb;
  h->A.num_meshes = n;
  return MWB_OK;
}

// ------------------------------------------------------------------ ABI: level definition
extern "C" int mwb_set_params(mwb_handle* h, const mwb_params* p) {
  if (!h || !p) return fail(MWB_EINVAL, "null argument");
  h->S.params = *p;
  h->S.near_extra = 1.1 * p->max_forward_step;
  h->have_params = true;
  return MWB_OK;
}

extern "C" int mwb_set_protos(mwb_handle* h, const mwb_proto* protos, int n) {
  if (!h || !protos || n <= 0) return fail(MWB_EINVAL, "bad arguments");
  int rc = replace_buf(&h->protos, protos, (size_t)n * sizeof(mwb_proto), h->stream);
  if (rc) return rc;
  h->S.protos = (const mwb_proto*)h->protos;
  h->S.num_protos = n;
  h->have_protos = true;
  // per-frame triangle lists of mesh entities: [N][E][largest mesh]
  int cap = 0;
  for (int k = 0; k < n; ++k)
    if (protos[k].kind == MWB_KIND_MESH) {
      if (protos[k].mesh_id < 0 || protos[k].mesh_id >= (int)h->mesh_counts.size())
        return fail(MWB_ESTATE, "mesh prototype refers to a mesh that was not uploaded");
      if (h->mesh_counts[protos[k].mesh_id] > cap) cap = h->mesh_counts[protos[k].mesh_id];
    }
  if (cap > h->S.mesh_cap) {
    void** bufs[] = {&h->mesh_tris_buf, &h->mesh_bbox_buf, &h->mesh_bin_idx_buf, &h->mesh_bin_off_buf};
    for (void** b : bufs) {
      if (*b) dev_free(*b);
      *b = nullptr;
    }
    const size_t slots = (size_t)h->S.N * h->S.E;
    if (dev_alloc(&h->mesh_tris_buf, slots * cap * sizeof(TriRec)) != 0 ||
        dev_alloc(&h->mesh_bbox_buf, slots * cap * sizeof(uint2)) != 0 ||
        dev_alloc(&h->mesh_bin_idx_buf, slots * cap * MWB_BIN_REFS * sizeof(uint16_t)) != 0 ||
        dev_alloc(&h->mesh_bin_off_buf, slots * (MWB_MAX_BINS + 1) * sizeof(int32_t)) != 0)
      return fail(MWB_ECUDA, "mesh triangle buffer allocation failed");
    h->S.mesh_tris = (TriRec*)h->mesh_tris_buf;
    h->S.mesh_bbox = (uint2*)h->mesh_bbox_buf;
    h->S.mesh_bin_idx = (uint16_t*)h->mesh_bin_idx_buf;
    h->S.mesh_bin_off = (int32_t*)h->mesh_bin_off_buf;
    h->S.mesh_cap = cap;
  }
  return MWB_OK;
}

static int upload_geometry(mwb_handle* h, size_t g, const mwb_geometry* geo) {
  DevState& S = h->S;
  if (geo->num_rooms > S.R || geo->num_quads > S.Q || geo->num_segs > S.S)
    return fail(MWB_ECAPACITY, "geometry exceeds max_rooms / max_quads / max_segs");
  for (int r = 0; r < geo->num_rooms; ++r)
    if (geo->rooms[r].num_edges > MWB_MAX_EDGES) return fail(MWB_ECAPACITY, "room outline too long");
  int32_t counts[3] = {geo->num_rooms, geo->num_quads, geo->num_segs};
  int rc = 0;
  rc |= stream_enter(h, h->stream);
  rc |= h2d(S.num_rooms + g, &counts[0], sizeof(int32_t), h->stream);
  rc |= h2d(S.num_quads + g, &counts[1], sizeof(int32_t), h->stream);
  rc |= h2d(S.num_segs + g, &counts[2], sizeof(int32_t), h->stream);
  if (geo->num_rooms) rc |= h2d(S.rooms + g * S.R, geo->rooms, geo->num_rooms * sizeof(mwb_room), h->stream);
  if (geo->num_quads) rc |= h2d(S.quads + g * S.Q, geo->quads, geo->num_quads * sizeof(mwb_quad), h->stream);
  if (geo->num_segs) rc |= h2d(S.segs + g * S.S, geo->segs, geo->num_segs * sizeof(mwb_seg), h->stream);
  rc |= sync_stream(h->stream);
  return rc ? fail(MWB_ECUDA, "geometry upload failed") : MWB_OK;
}

extern "C" int mwb_set_template(mwb_handle* h, const mwb_geometry* g) {
  if (!h || !g) return fail(MWB_EINVAL, "null argument");
  if (!h->S.shared_geom) return fail(MWB_ESTATE, "handle was created with shared_geometry = 0");
  int rc = upload_geometry(h, 0, g);
  if (!rc) h->have_template = true;
  return rc;
}

extern "C" int mwb_set_program(mwb_handle* h, const mwb_op* ops, int n) {
  if (!h || !ops || n <= 0 || n > MWB_MAX_OPS) return fail(MWB_EINVAL, "bad program");
  int rc = replace_buf(&h->ops, ops, (size_t)n * sizeof(mwb_op), h->stream);
  if (rc) return rc;
  h->S.ops = (const mwb_op*)h->ops;
  h->S.num_ops = n;
  return MWB_OK;
}

extern "C" int mwb_set_maze(mwb_handle* h, const mwb_maze_desc* mz) {
  if (!h || !mz || !mz->cdf) return fail(MWB_EINVAL, "null argument");
  if (h->S.shared_geom) return fail(MWB_ESTATE, "Maze needs per-env geometry (shared_geometry = 0)");
  const int cells = mz->rows * mz->cols;
  if (cells <= 0 || cells > MWB_MAZE_MAX_CELLS) return fail(MWB_ECAPACITY, "maze too large");
  if (2 * cells - 1 > h->S.R) return fail(MWB_ECAPACITY, "max_rooms too small for this maze");
  MazeDev m;
  memset(&m, 0, sizeof(m));
  m.rows = mz->rows;
  m.cols = mz->cols;
  m.pitch = mz->pitch;
  m.cell_room = mz->cell_room;
  memcpy(m.cell_quads, mz->cell_quads, sizeof(m.cell_quads));
  memcpy(m.cell_segs, mz->cell_segs, sizeof(m.cell_segs));
  memcpy(m.open_a, mz->open_a, sizeof(m.open_a));
  memcpy(m.open_b, mz->open_b, sizeof(m.open_b));
  memcpy(m.conn_room, mz->conn_room, sizeof(m.conn_room));
  memcpy(m.conn_quads, mz->conn_quads, sizeof(m.conn_quads));
  memcpy(m.conn_segs, mz->conn_segs, sizeof(m.conn_segs));
  int rc = replace_buf(&h->maze, &m, sizeof(m), h->stream);
  if (!rc) rc = replace_buf(&h->maze_cdf, mz->cdf, (size_t)(2 * cells - 1) * sizeof(double), h->stream);
  if (rc) return rc;
  h->S.maze = (const MazeDev*)h->maze;
  h->S.maze_cdf = (const double*)h->maze_cdf;
  return MWB_OK;
}

extern "C" int mwb_get_geometry(mwb_handle* h, int env, int32_t counts[3], mwb_room* rooms, mwb_quad* quads, mwb_seg* segs) {
  if (!h || !counts) return fail(MWB_EINVAL, "null argument");
  if (env < 0 || env >= h->S.N) return fail(MWB_EINVAL, "env out of range");
  const size_t g = h->S.shared_geom ? 0 : (size_t)env;
  int rc = 0;
  rc |= stream_enter(h, h->stream);
  rc |= d2h(&counts[0], h->S.num_rooms + g, sizeof(int32_t), h->stream);
  rc |= d2h(&counts[1], h->S.num_quads + g, sizeof(int32_t), h->stream);
  rc |= d2h(&counts[2], h->S.num_segs + g, sizeof(int32_t), h->stream);
  if (rooms) rc |= d2h(rooms, h->S.rooms + g * h->S.R, (size_t)h->S.R * sizeof(mwb_room), h->stream);
  if (quads) rc |= d2h(quads, h->S.quads + g * h->S.Q, (size_t)h->cfg.max_quads * sizeof(mwb_quad), h->stream);
  if (segs) rc |= d2h(segs, h->S.segs + g * h->S.S, (size_t)h->S.S * sizeof(mwb_seg), h->stream);
  rc |= sync_stream(h->stream);
  return rc ? fail(MWB_ECUDA, "readback failed") : MWB_OK;
}

// ------------------------------------------------------------------ ABI: reset
static int launch_upload(mwb_handle* h, const std::vector<WorldUpload>& up, bool seed_only) {
  const int n = (int)up.size();
  if (stream_enter(h, h->stream)) return MWB_ECUDA;
  if (h2d(h->d_upload, up.data(), n * sizeof(WorldUpload), h->stream) != 0) return fail(MWB_ECUDA, "upload failed");
#ifndef MWB_HOSTSIM
  if (seed_only)
    seed_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->S, h->d_upload, n);
  else
    scatter_kernel<<<(n + 127) / 128, 128, 0, h->stream>>>(h->S, h->d_upload, n);
  h->launches++;
  CK(cudaGetLastError());
#else
  for (int t = 0; t < n; ++t) {
    if (seed_only) {
      const WorldUpload& u = h->d_upload[t];
      int i = u.env;
      h->S.rng_s_hi[i] = u.rng.state_hi;
      h->S.rng_s_lo[i] = u.rng.state_lo;
      h->S.rng_inc_hi[i] = u.rng.inc_hi;
      h->S.rng_inc_lo[i] = u.rng.inc_lo;
      h->S.rng_has32[i] = u.rng.has_uint32;
      h->S.rng_cache[i] = u.rng.uinteger;
    } else {
      scatter_one(h->S, h->d_upload[t]);
    }
  }
#endif
  return sync_stream(h->stream) == 0 ? MWB_OK : fail(MWB_ECUDA, "sync failed");
}

extern "C" int mwb_seed(mwb_handle* h, const int32_t* env_ids, int n, const mwb_rng_state* states) {
  if (!h || !states || n <= 0 || n > h->S.N) return fail(MWB_EINVAL, "bad arguments");
  std::vector<WorldUpload> up(n);
  for (int t = 0; t < n; ++t) {
    memset(&up[t], 0, sizeof(WorldUpload));
    up[t].env = env_ids ? env_ids[t] : t;
    if (up[t].env < 0 || up[t].env >= h->S.N) return fail(MWB_EINVAL, "env id out of range");
    up[t].rng = states[t];
  }
  return launch_upload(h, up, true);
}

extern "C" int mwb_reset(mwb_handle* h, const int32_t* env_ids, int n, void* stream) {
  if (!h) return fail(MWB_EINVAL, "null handle");
  if (!h->have_params || !h->have_protos || !h->S.ops) return fail(MWB_ESTATE, "params / protos / program not set");
  if (h->S.shared_geom && !h->have_template) return fail(MWB_ESTATE, "template not set");
  stream_t s = stream ? (stream_t)stream : h->stream;
  if (!env_ids) n = h->S.N;
  if (n <= 0 || n > h->S.N) return fail(MWB_EINVAL, "bad count");
  if (stream_enter(h, s)) return MWB_ECUDA;
  const int32_t* ids = nullptr;
  if (env_ids) {
    if (is_device_ptr(env_ids)) {
      ids = env_ids;
    } else {
      if (h2d(h->d_ids, env_ids, n * sizeof(int32_t), s) != 0) return fail(MWB_ECUDA, "upload failed");
      ids = h->d_ids;
    }
  }
#ifndef MWB_HOSTSIM
  reset_kernel<<<(n + 3) / 4, 128, 0, s>>>(h->S, ids, n);
  h->launches++;
  CK(cudaGetLastError());
  if (stream_leave(h, s)) return MWB_ECUDA;
  if (!stream) CK(cudaStreamSynchronize(s));
#else
  for (int t = 0; t < n; ++t) {
    int i = ids ? ids[t] : t;
    device_reset(h->S, i);
    h->S.needs_reset[i] = 0;
  }
#endif
  return MWB_OK;
}

extern "C" int mwb_set_world(mwb_handle* h, const int32_t* env_ids, int n, const mwb_world* worlds) {
  if (!h || !worlds || n <= 0 || n > h->S.N) return fail(MWB_EINVAL, "bad arguments");
  if (!h->have_protos) return fail(MWB_ESTATE, "protos not set");
  std::vector<WorldUpload> up(n);
  for (int t = 0; t < n; ++t) {
    const mwb_world& w = worlds[t];
    WorldUpload& u = up[t];
    memset(&u, 0, sizeof(u));
    u.env = env_ids ? env_ids[t] : t;
    if (u.env < 0 || u.env >= h->S.N) return fail(MWB_EINVAL, "env id out of range");
    if (w.num_slots > h->S.E || w.num_slots > MWB_MAX_ENTS_CAP) return fail(MWB_ECAPACITY, "too many entities");
    if (!h->S.shared_geom) {
      int rc = upload_geometry(h, (size_t)u.env, &w.geom);
      if (rc) return rc;
    }
    u.num_slots = w.num_slots;
    u.agent_slot = w.agent_slot;
    u.carrying = w.carrying;
    u.step_count = w.step_count;
    u.num_picked = w.num_picked_up;
    u.hold = w.hold;
    u.cam[0] = w.cam_height;
    u.cam[1] = w.cam_fwd_disp;
    u.cam[2] = w.cam_pitch;
    u.cam[3] = w.cam_fov_y;
    for (int k = 0; k < 3; ++k) {
      u.envp[0 + k] = w.sky_color[k];
      u.envp[3 + k] = w.light_pos[k];
      u.envp[6 + k] = w.light_color[k];
      u.envp[9 + k] = w.light_ambient[k];
    }
    for (int e = 0; e < w.num_slots; ++e) u.ents[e] = w.ents[e];
  }
  return launch_upload(h, up, false);
}

// ------------------------------------------------------------------ peer-memory buffers
extern "C" int mwb_shared_alloc(int device, size_t bytes, void** dev_ptr, unsigned char handle[64]) {
#ifndef MWB_HOSTSIM
  if (!dev_ptr || !handle) return fail(MWB_EINVAL, "null argument");
  CK(cudaSetDevice(device));
  CK(cudaMalloc(dev_ptr, bytes));
  cudaIpcMemHandle_t hd;
  static_assert(sizeof(hd) == 64, "CUDA IPC handle size");
  CK(cudaIpcGetMemHandle(&hd, *dev_ptr));
  memcpy(handle, &hd, 64);
  return MWB_OK;
#else
  return fail(MWB_ENOCUDA, "host simulator has no peer memory");
#endif
}

extern "C" int mwb_shared_open(int device, const unsigned char handle[64], void** dev_ptr) {
#ifndef MWB_HOSTSIM
  if (!dev_ptr || !handle) return fail(MWB_EINVAL, "null argument");
  CK(cudaSetDevice(device));
  cudaIpcMemHandle_t hd;
  memcpy(&hd, handle, 64);
  CK(cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess));
  return MWB_OK;
#else
  return fail(MWB_ENOCUDA, "host simulator has no peer memory");
#endif
}

extern "C" int mwb_shared_close(void* dev_ptr, int opened) {
#ifndef MWB_HOSTSIM
  if (!dev_ptr) return MWB_OK;
  if (opened) CK(cudaIpcCloseMemHandle(dev_ptr));
  else CK(cudaFree(dev_ptr));
#endif
  return MWB_OK;
}

// ------------------------------------------------------------------ stream-ordered flags (one-way completion signals)
// The multi-GPU observation path needs no rendezvous: after its K2, rank r writes the step number into a slot of
// rank 0's peer-mapped buffer, stream-ordered behind the kernel's stores (system-scope release); rank 0's stream waits
// until every slot has reached the step.  Implemented with CUDA stream memory operations (cuStreamWriteValue32 /
// cuStreamWaitValue32, looked up at run time so that the library keeps linking against cudart only); if the driver
// does not offer them -- or MWB_FLAG_MODE=kernel -- one-thread kernels do the same (st.release.sys / ld.acquire.sys).
#ifndef MWB_HOSTSIM
__global__ void flag_write_kernel(uint32_t* p, uint32_t v) {
  __threadfence_system();
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__global__ void flag_wait_kernel(const uint32_t* p, uint32_t v) {
  uint32_t cur;
  do {
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(cur) : "l"(p) : "memory");
    if ((int32_t)(cur - v) < 0) __nanosleep(200);
  } while ((int32_t)(cur - v) < 0);
}
typedef int (*mwb_memop_fn)(cudaStream_t, unsigned long long, uint32_t, unsigned int);
static mwb_memop_fn g_write32 = nullptr, g_wait32 = nullptr;
static int g_flag_mode = -1;     // 0 = stream memory operations, 1 = kernels
static void flag_init() {
  if (g_flag_mode >= 0) return;
  g_flag_mode = 1;
  const char* m = getenv("MWB_FLAG_MODE");
  if (m && strcmp(m, "kernel") == 0) return;
  void *w = nullptr, *q = nullptr;
  cudaDriverEntryPointQueryResult r1, r2;
  if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &w, cudaEnableDefault, &r1) == cudaSuccess && r1 == cudaDriverEntryPointSuccess &&
      cudaGetDriverEntryPoint("cuStreamWaitValue32", &q, cudaEnableDefault, &r2) == cudaSuccess && r2 == cudaDriverEntryPointSuccess &&
      w && q) {
    g_write32 = (mwb_memop_fn)w;
    g_wait32 = (mwb_memop_fn)q;
    g_flag_mode = 0;
  } else {
    cudaGetLastError();
  }
}
#endif

extern "C" int mwb_flag_write(void* stream, uint32_t* dev_ptr, uint32_t value) {
#ifndef MWB_HOSTSIM
  if (!dev_ptr) return fail(MWB_EINVAL, "null argument");
  flag_init();
  cudaStream_t s = (cudaStream_t)stream;
  if (g_flag_mode == 0) {
    if (g_write32(s, (unsigned long long)(uintptr_t)dev_ptr, value, 0u /* CU_STREAM_WRITE_VALUE_DEFAULT: with memory barrier */) != 0)
      return fail(MWB_ECUDA, "cuStreamWriteValue32 failed");
  } else {
    flag_write_kernel<<<1, 1, 0, s>>>(dev_ptr, value);
    CK(cudaGetLastError());
  }
  return MWB_OK;
#else
  return fail(MWB_ENOCUDA, "host simulator has no streams");
#endif
}

extern "C" int mwb_flag_wait_geq(void* stream, const uint32_t* dev_ptr, uint32_t value) {
#ifndef MWB_HOSTSIM
  if (!dev_ptr) return fail(MWB_EINVAL, "null argument");
  flag_init();
  cudaStream_t s = (cudaStream_t)stream;
  if (g_flag_mode == 0) {
    if (g_wait32(s, (unsigned long long)(uintptr_t)dev_ptr, value, 0u /* CU_STREAM_WAIT_VALUE_GEQ */) != 0)
      return fail(MWB_ECUDA, "cuStreamWaitValue32 failed");
  } else {
    flag_wait_kernel<<<1, 1, 0, s>>>(dev_ptr, value);
    CK(cudaGetLastError());
  }
  return MWB_OK;
#else
  return fail(MWB_ENOCUDA, "host simulator has no streams");
#endif
}

extern "C" int mwb_flag_mode(void) {
#ifndef MWB_HOSTSIM
  flag_init();
  return g_flag_mode;
#else
  return -1;
#endif
}

// ------------------------------------------------------------------ profiling
#ifndef MWB_HOSTSIM
static void prof_mark(mwb_handle* h, std::vector<cudaEvent_t>& v, stream_t s) {
  if (!h->profiling) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, s);
  v.push_back(e);
}
static double prof_drain(std::vector<cudaEvent_t>& v, int64_t* count) {
  double ms = 0.0;
  *count = 0;
  for (size_t k = 0; k + 1 < v.size(); k += 2) {
    float t = 0.0f;
    cudaEventSynchronize(v[k + 1]);
    if (cudaEventElapsedTime(&t, v[k], v[k + 1]) == cudaSuccess) {
      ms += t;
      ++*count;
    }
  }
  for (cudaEvent_t e : v) cudaEventDestroy(e);
  v.clear();
  return ms;
}
#endif

extern "C" int mwb_profile(mwb_handle* h, int enable) {
  if (!h) return fail(MWB_EINVAL, "null handle");
  h->profiling = enable != 0;
  return MWB_OK;
}

extern "C" int mwb_profile_read(mwb_handle* h, double* k1_ms, double* k2_ms, int64_t* k1_launches, int64_t* k2_launches) {
  if (!h) return fail(MWB_EINVAL, "null handle");
  double a = 0.0, b = 0.0;
  int64_t na = 0, nb = 0;
#ifndef MWB_HOSTSIM
  a = prof_drain(h->ev_k1, &na);
  b = prof_drain(h->ev_k2, &nb);
#endif
  if (k1_ms) *k1_ms = a;
  if (k2_ms) *k2_ms = b;
  if (k1_launches) *k1_launches = na;
  if (k2_launches) *k2_launches = nb;
  return MWB_OK;
}

// ------------------------------------------------------------------ ABI: the hot path
// Launch K2 for envs [env0, env0 + count) (obs / depth point at env 0 of the full buffers).
static int launch_k2(mwb_handle* h, uint8_t* obs, float* depth, int env0, int count, stream_t s) {
#ifndef MWB_HOSTSIM
  if (obs != h->peer_checked) {         // the observation destination rarely changes: query its home device once
    cudaPointerAttributes pa;
    h->peer_checked = obs;
    h->peer_result = obs && cudaPointerGetAttributes(&pa, obs) == cudaSuccess && pa.type == cudaMemoryTypeDevice &&
                     pa.device != h->cfg.device;
    cudaGetLastError();
  }
  h->obs_is_peer = h->obs_peer_hint >= 0 ? h->obs_peer_hint != 0 : h->peer_result;
  const int smem = k2_smem_bytes(h), fstage = k2_frame_stage_bytes(h);
  const K2Layout lay = k2_layout(h->smem_tris, h->tri_cap, h->stage_bytes, k2_halves_per_part(h->S.obs_w, h->S.obs_h, h->k2_parts), fstage);
  if (ensure_k2_smem(h, smem)) return fail(MWB_ECUDA, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed");
  prof_mark(h, h->ev_k2, s);
  k2_kernel(h->S.msaa)<<<count * h->k2_parts, MWB_K2_THREADS, smem, s>>>(h->S, h->A, h->view, h->obs_format, obs, depth, env0,
                                                                          h->k2_parts, h->tri_cap, h->stage_bytes, fstage, lay,
                                                                          h->d_overflow);
  prof_mark(h, h->ev_k2, s);
  h->launches++;
  CK(cudaGetLastError());
#endif
  return MWB_OK;
}

// Render all envs.  With host destinations the frame batch is cut into chunks: chunk c is
// copied device->host on a second stream while chunk c + 1 is being rasterised, so the PCIe
// transfer of the observations overlaps the render instead of following it.
static int launch_render(mwb_handle* h, uint8_t* obs, float* depth, stream_t s, uint8_t* host_obs = nullptr,
                         float* host_depth = nullptr) {
  if (!h->A.tex) return fail(MWB_ESTATE, "textures not uploaded");
#ifndef MWB_HOSTSIM
  {
    const long long threads = (long long)h->S.N * (6 + 2 * h->S.E);
    frame_trig_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(h->S);
    h->launches++;
    CK(cudaGetLastError());
  }
  if (h->S.mesh_cap > 0) {
    mesh_setup_kernel<<<dim3(h->S.N, h->S.E), 256, 0, s>>>(h->S, h->A, h->view);
    h->launches++;
    CK(cudaGetLastError());
  }
  const int N = h->S.N;
  const size_t px = (size_t)h->S.obs_w * h->S.obs_h;
  const bool pipelined = (host_obs || host_depth) && N >= 256;
  int chunks = pipelined ? MWB_DEFAULT_D2H_CHUNKS : 1;
  while (chunks > 1 && N / chunks < 256) --chunks;   // keep every launch a few hundred blocks wide
  for (int c = 0; c < chunks; ++c) {
    const int e0 = (int)((long long)N * c / chunks), e1 = (int)((long long)N * (c + 1) / chunks);
    int rc = launch_k2(h, obs, depth, e0, e1 - e0, s);
    if (rc) return rc;
    if (pipelined) {
      CK(cudaEventRecord(h->chunk_done[c], s));
      CK(cudaStreamWaitEvent(h->copy_stream, h->chunk_done[c], 0));
      if (host_obs)
        CK(cudaMemcpyAsync(host_obs + (size_t)e0 * px * h->obs_px_bytes, obs + (size_t)e0 * px * h->obs_px_bytes,
                           (size_t)(e1 - e0) * px * h->obs_px_bytes,
                           cudaMemcpyDeviceToHost, h->copy_stream));
      if (host_depth)
        CK(cudaMemcpyAsync(host_depth + (size_t)e0 * px, depth + (size_t)e0 * px, (size_t)(e1 - e0) * px * sizeof(float),
                           cudaMemcpyDeviceToHost, h->copy_stream));
    }
  }
  if (pipelined) {
    h->frames_copied = true;
    CK(cudaEventRecord(h->copies_done, h->copy_stream));
    CK(cudaStreamWaitEvent(s, h->copies_done, 0));   // later work on s (and its sync) sees the copies
  }
#else
  hostsim_render(h->S, h->A, h->view, h->obs_format, obs, depth);
#endif
  return MWB_OK;
}

static int finish_outputs(mwb_handle* h, uint8_t* obs, bool obs_host, float* depth, bool depth_host, double* reward,
                          uint8_t* term, uint8_t* trunc, stream_t s, bool user_stream) {
  const size_t N = h->S.N, px = (size_t)h->S.obs_w * h->S.obs_h;
  int rc = 0;
  bool any_host = false;
  if (obs && obs_host) { if (!h->frames_copied) rc |= d2h(obs, h->d_obs, N * px * h->obs_px_bytes, s); any_host = true; }
  if (depth && depth_host) { if (!h->frames_copied) rc |= d2h(depth, h->d_depth, N * px * sizeof(float), s); any_host = true; }
  h->frames_copied = false;
  if (reward && !is_device_ptr(reward)) { rc |= d2h(reward, h->d_reward, N * sizeof(double), s); any_host = true; }
  if (term && !is_device_ptr(term)) { rc |= d2h(term, h->d_term, N, s); any_host = true; }
  if (trunc && !is_device_ptr(trunc)) { rc |= d2h(trunc, h->d_trunc, N, s); any_host = true; }
  if (rc) return fail(MWB_ECUDA, "readback failed");
  if (stream_leave(h, s)) return MWB_ECUDA;
  if (any_host || !user_stream)
    if (sync_stream(s) != 0) return fail(MWB_ECUDA, "stream sync failed");
  return MWB_OK;
}

extern "C" int mwb_step(mwb_handle* h, const int32_t* actions, const double* step_params, uint8_t* obs, float* depth,
                        double* reward, uint8_t* terminated, uint8_t* truncated, void* stream) {
  if (!h || !actions) return fail(MWB_EINVAL, "null argument");
  if (!h->have_params || !h->have_protos) return fail(MWB_ESTATE, "params / protos not set");
  stream_t s = stream ? (stream_t)stream : h->stream;
  if (stream_enter(h, s)) return MWB_ECUDA;
  const size_t N = h->S.N;
  const int32_t* d_act = actions;
  if (!is_device_ptr(actions)) {
    if (h2d(h->d_actions, actions, N * sizeof(int32_t), s) != 0) return fail(MWB_ECUDA, "action upload failed");
    d_act = h->d_actions;
  }
  const double* d_sp = nullptr;
  if (step_params) {
    if (is_device_ptr(step_params)) {
      d_sp = step_params;
    } else {
      if (h2d(h->d_step_params, step_params, 3 * N * sizeof(double), s) != 0) return fail(MWB_ECUDA, "upload failed");
      d_sp = h->d_step_params;
    }
  }
  // rewards / flags go to caller device memory directly, else to staging
  double* d_rew = reward && is_device_ptr(reward) ? reward : h->d_reward;
  uint8_t* d_te = terminated && is_device_ptr(terminated) ? terminated : h->d_term;
  uint8_t* d_tr = truncated && is_device_ptr(truncated) ? truncated : h->d_trunc;
#ifndef MWB_HOSTSIM
  prof_mark(h, h->ev_k1, s);
  step_kernel<<<(unsigned)((N + 3) / 4), 128, 0, s>>>(h->S, d_act, d_sp, d_rew, d_te, d_tr);
  prof_mark(h, h->ev_k1, s);
  h->launches++;
  CK(cudaGetLastError());
#else
  for (size_t i = 0; i < N; ++i) step_one(h->S, (int)i, d_act, d_sp, d_rew, d_te, d_tr);
#endif
  const bool obs_host = obs && !is_device_ptr(obs), depth_host = depth && !is_device_ptr(depth);
  if (obs || depth) {
    int rc = launch_render(h, obs ? (obs_host ? h->d_obs : obs) : nullptr, depth ? (depth_host ? h->d_depth : depth) : nullptr, s,
                           obs_host ? obs : nullptr, depth_host ? depth : nullptr);
    if (rc) return rc;
  }
  return finish_outputs(h, obs, obs_host, depth, depth_host, reward, terminated, truncated, s, stream != nullptr);
}

extern "C" int mwb_render_obs(mwb_handle* h, uint8_t* obs, float* depth, void* stream) {
  if (!h || (!obs && !depth)) return fail(MWB_EINVAL, "null argument");
  stream_t s = stream ? (stream_t)stream : h->stream;
  if (stream_enter(h, s)) return MWB_ECUDA;
  const bool obs_host = obs && !is_device_ptr(obs), depth_host = depth && !is_device_ptr(depth);
  int rc = launch_render(h, obs ? (obs_host ? h->d_obs : obs) : nullptr, depth ? (depth_host ? h->d_depth : depth) : nullptr, s,
                         obs_host ? obs : nullptr, depth_host ? depth : nullptr);
  if (rc) return rc;
  return finish_outputs(h, obs, obs_host, depth, depth_host, nullptr, nullptr, nullptr, s, stream != nullptr);
}

extern "C" int mwb_set_obs_peer(mwb_handle* h, int peer) {
  if (!h) return fail(MWB_EINVAL, "null handle");
  h->obs_peer_hint = peer < 0 ? -1 : (peer ? 1 : 0);
  return MWB_OK;
}

extern "C" int mwb_set_obs_format(mwb_handle* h, int format) {
  if (!h) return fail(MWB_EINVAL, "null handle");
  if (format != MWB_OBS_HWC_U8 && format != MWB_OBS_CWH_U8 && format != MWB_OBS_GREY_F64) return fail(MWB_EINVAL, "unknown format");
  const size_t pxb = format == MWB_OBS_GREY_F64 ? 8 : 3;
  const size_t need = (size_t)h->S.N * h->S.obs_w * h->S.obs_h * pxb;
  if (need > h->d_obs_bytes) {     // staging for host destinations grows with the pixel size
    uint8_t* buf = nullptr;
    if (alloc_arr(h, &buf, need)) return fail(MWB_ECUDA, "staging allocation failed");
    h->d_obs = buf;
    h->d_obs_bytes = need;
  }
  h->obs_format = format;
  h->obs_px_bytes = pxb;
  return MWB_OK;
}

extern "C" int mwb_set_action_noise(mwb_handle* h, int enabled, double prob, int random_action) {
  if (!h) return fail(MWB_EINVAL, "null handle");
  if (enabled && !(prob >= 0.0 && prob <= 1.0)) return fail(MWB_EINVAL, "prob must be in [0, 1]");
  if (enabled && random_action > 7) return fail(MWB_EINVAL, "random_action must be an Actions value (0..7) or negative");
  h->S.act_noise = enabled != 0;
  h->S.act_prob = prob;
  h->S.act_random = random_action;
  return MWB_OK;
}

extern "C" int mwb_render_top_view(mwb_handle* h, const double extents[4], int render_agent, uint8_t* obs, void* stream) {
  if (!h || !extents || !obs) return fail(MWB_EINVAL, "null argument");
  if (!(extents[1] > extents[0]) || !(extents[3] > extents[2])) return fail(MWB_EINVAL, "empty extents");
  stream_t s = stream ? (stream_t)stream : h->stream;
  if (stream_enter(h, s)) return MWB_ECUDA;
  const bool obs_host = !is_device_ptr(obs);
  // glOrtho(min_x, max_x, -max_z, -min_z, -100, 100) (miniworld.py:1137)
  h->view.mode = 1;
  h->view.render_agent = render_agent != 0;
  h->view.l = extents[0];
  h->view.r = extents[1];
  h->view.b = -extents[3];
  h->view.t = -extents[2];
  int rc = launch_render(h, obs_host ? h->d_obs : obs, nullptr, s, obs_host ? obs : nullptr, nullptr);
  memset(&h->view, 0, sizeof(ViewSpec));
  if (rc) return rc;
  return finish_outputs(h, obs, obs_host, nullptr, false, nullptr, nullptr, nullptr, s, stream != nullptr);
}

extern "C" int mwb_visible_ents(mwb_handle* h, uint32_t* mask, void* stream) {
  if (!h || !mask) return fail(MWB_EINVAL, "null argument");
  if (!h->have_protos) return fail(MWB_ESTATE, "protos not set");
  stream_t s = stream ? (stream_t)stream : h->stream;
  if (stream_enter(h, s)) return MWB_ECUDA;
  const int N = h->S.N, box0 = 2 * h->cfg.max_quads, cap = box0 + 12 * h->cfg.max_ents;
  if (!h->vis_tris && alloc_arr(h, &h->vis_tris, (size_t)N * cap)) return fail(MWB_ECUDA, "scratch allocation failed");
  const bool host = !is_device_ptr(mask);
  uint32_t* d_mask = host ? reinterpret_cast<uint32_t*>(h->d_ids) : mask;   // d_ids: N x int32 staging, free between calls
#ifndef MWB_HOSTSIM
  switch (h->S.msaa) {
    case 1: visible_ents_kernel<1><<<N, 256, 0, s>>>(h->S, h->A, h->vis_tris, cap, box0, d_mask); break;
    case 4: visible_ents_kernel<4><<<N, 256, 0, s>>>(h->S, h->A, h->vis_tris, cap, box0, d_mask); break;
    case 16: visible_ents_kernel<16><<<N, 256, 0, s>>>(h->S, h->A, h->vis_tris, cap, box0, d_mask); break;
    default: visible_ents_kernel<8><<<N, 256, 0, s>>>(h->S, h->A, h->vis_tris, cap, box0, d_mask); break;
  }
  h->launches++;
  CK(cudaGetLastError());
#else
  const int W = h->S.obs_w, H = h->S.obs_h, M = h->S.msaa;
  for (int i = 0; i < N; ++i) {
    TriRec* tris = h->vis_tris + (size_t)i * cap;
    const Camera cam = make_camera(h->S, i);
    int ent_slot[32];
    const int n_query = queried_entities(h->S, i, ent_slot);
    int n_room = 0;
    const mwb_quad* quads = env_quads(h->S, i);
    const int nq = h->S.num_quads[geom_index(h->S, i)];
    TriInput in;
    TriRec rec;
    for (int task = 0; task < 2 * nq; ++task)
      if (room_triangle(h->S, h->A, quads, i, task >> 1, task & 1, in) && finish_triangle(cam, in, W, H, rec)) tris[n_room++] = rec;
    for (int j = 0; j < 12 * n_query; ++j) {
      query_box_triangle(entity_pose(h->S, i, ent_slot[j / 12]), j % 12, in);
      if (!finish_triangle(cam, in, W, H, rec)) empty_bbox(rec);
      tris[box0 + j] = rec;
    }
    uint32_t vis = 0;
    for (int py = 0; py < H; ++py)
      for (int px = 0; px < W; ++px)
        for (int sm = 0; sm < M; ++sm) {
          float ox, oy;
          if (M == 16) sample_xy_dyn<16>(sm, ox, oy);
          else if (M == 8) sample_xy_dyn<8>(sm, ox, oy);
          else if (M == 4) sample_xy_dyn<4>(sm, ox, oy);
          else sample_xy_dyn<1>(sm, ox, oy);
          vis |= visible_at_sample(tris, n_room, box0, n_query, ent_slot, px, py, (float)px + ox, (float)py + oy);
        }
    d_mask[i] = vis;
  }
#endif
  if (host && d2h(mask, d_mask, (size_t)N * sizeof(uint32_t), s) != 0) return fail(MWB_ECUDA, "readback failed");
  if (stream_leave(h, s)) return MWB_ECUDA;
  if (host) {
    if (sync_stream(s) != 0) return fail(MWB_ECUDA, "stream sync failed");
  } else if (!stream) {
    if (sync_stream(s) != 0) return fail(MWB_ECUDA, "stream sync failed");
  }
  return MWB_OK;
}

// ------------------------------------------------------------------ ABI: snapshot / restore
// Every array that changes while episodes run (entity lists, counters, camera / lighting parameters, RNG
// streams, pending-reset flags) plus the geometry currently on the device, in one fixed order.
struct SnapHeader {
  uint32_t magic, abi;
  int32_t N, E, R, Q, S, G;
  uint64_t bytes;
};

static void snapshot_arrays(mwb_handle* h, std::vector<std::pair<void*, size_t>>& v) {
  const DevState& S = h->S;
  const size_t N = S.N, E = S.E, G = S.shared_geom ? 1 : N;
#define SA(field, count) v.push_back(std::make_pair((void*)S.field, (size_t)(count) * sizeof(*S.field)))
  SA(ent_proto, E * N); SA(ent_px, E * N); SA(ent_py, E * N); SA(ent_pz, E * N); SA(ent_dir, E * N);
  SA(ent_col, E * 3 * N); SA(ent_size, E * N); SA(num_slots, N); SA(agent_slot, N); SA(carrying, N); SA(step_count, N);
  SA(num_picked, N); SA(needs_reset, N); SA(episodes_done, 1); SA(cam, 4 * N); SA(envp, 12 * N);
  SA(ghost_slot, N); SA(ghost_proto, N); SA(ghost_pose, 4 * N); SA(ghost_col, 3 * N);
  SA(rng_s_hi, N); SA(rng_s_lo, N); SA(rng_inc_hi, N); SA(rng_inc_lo, N); SA(rng_has32, N); SA(rng_cache, N);
  SA(num_rooms, G); SA(num_quads, G); SA(num_segs, G);
  SA(rooms, G * S.R); SA(quads, G * S.Q); SA(segs, G * S.S); SA(room_tex, N * S.R * 3);
#undef SA
}

static SnapHeader snapshot_header(mwb_handle* h) {
  std::vector<std::pair<void*, size_t>> v;
  snapshot_arrays(h, v);
  SnapHeader hd;
  hd.magic = 0x5342574du;   // "MWBS"
  hd.abi = MWB_ABI_VERSION;
  hd.N = h->S.N; hd.E = h->S.E; hd.R = h->S.R; hd.Q = h->S.Q; hd.S = h->S.S;
  hd.G = h->S.shared_geom ? 1 : h->S.N;
  hd.bytes = sizeof(SnapHeader);
  for (size_t k = 0; k < v.size(); ++k) hd.bytes += v[k].second;
  return hd;
}

extern "C" int mwb_snapshot_size(mwb_handle* h, size_t* bytes) {
  if (!h || !bytes) return fail(MWB_EINVAL, "null argument");
  *bytes = (size_t)snapshot_header(h).bytes;
  return MWB_OK;
}

extern "C" int mwb_snapshot(mwb_handle* h, void* blob, size_t bytes) {
  if (!h || !blob) return fail(MWB_EINVAL, "null argument");
  const SnapHeader hd = snapshot_header(h);
  if (bytes < hd.bytes) return fail(MWB_ECAPACITY, "snapshot buffer too small");
  std::vector<std::pair<void*, size_t>> v;
  snapshot_arrays(h, v);
  unsigned char* p = (unsigned char*)blob;
  memcpy(p, &hd, sizeof(hd));
  p += sizeof(hd);
  if (stream_enter(h, h->stream)) return MWB_ECUDA;
  for (size_t k = 0; k < v.size(); ++k) {
    if (d2h(p, v[k].first, v[k].second, h->stream) != 0) return fail(MWB_ECUDA, "readback failed");
    p += v[k].second;
  }
  if (sync_stream(h->stream) != 0) return fail(MWB_ECUDA, "sync failed");
  return MWB_OK;
}

extern "C" int mwb_restore(mwb_handle* h, const void* blob, size_t bytes) {
  if (!h || !blob) return fail(MWB_EINVAL, "null argument");
  const SnapHeader want = snapshot_header(h);
  SnapHeader hd;
  if (bytes < sizeof(hd)) return fail(MWB_EINVAL, "not a snapshot");
  memcpy(&hd, blob, sizeof(hd));
  if (hd.magic != want.magic || hd.abi != want.abi) return fail(MWB_EABI, "snapshot from another ABI version");
  if (hd.N != want.N || hd.E != want.E || hd.R != want.R || hd.Q != want.Q || hd.S != want.S || hd.G != want.G ||
      hd.bytes != want.bytes || bytes < hd.bytes)
    return fail(MWB_EINVAL, "snapshot does not match this handle's configuration");
  std::vector<std::pair<void*, size_t>> v;
  snapshot_arrays(h, v);
  const unsigned char* p = (const unsigned char*)blob + sizeof(hd);
  if (stream_enter(h, h->stream)) return MWB_ECUDA;
  for (size_t k = 0; k < v.size(); ++k) {
    if (h2d(v[k].first, p, v[k].second, h->stream) != 0) return fail(MWB_ECUDA, "upload failed");
    p += v[k].second;
  }
  if (sync_stream(h->stream) != 0) return fail(MWB_ECUDA, "sync failed");
  return MWB_OK;
}

// ------------------------------------------------------------------ ABI: camera read-back (parity tests)
#ifndef MWB_HOSTSIM
__global__ void camera_kernel(DevState S, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= S.N) return;
  const Camera c = make_camera(S, i);
  float* o = out + (size_t)i * 16;
  o[0] = c.ex; o[1] = c.ey; o[2] = c.ez; o[3] = c.sx; o[4] = c.sy; o[5] = c.sz; o[6] = c.ux; o[7] = c.uy; o[8] = c.uz;
  o[9] = c.fx; o[10] = c.fy; o[11] = c.fz; o[12] = c.px; o[13] = c.py; o[14] = c.za; o[15] = c.zb;
}
#endif

extern "C" int mwb_debug_camera(mwb_handle* h, float* out) {
  if (!h || !out) return fail(MWB_EINVAL, "null argument");
  const int N = h->S.N;
#ifndef MWB_HOSTSIM
  if (stream_enter(h, h->stream)) return MWB_ECUDA;
  float* d = nullptr;
  if (dev_alloc((void**)&d, (size_t)N * 16 * sizeof(float)) != 0) return fail(MWB_ECUDA, "device allocation failed");
  camera_kernel<<<(N + 127) / 128, 128, 0, h->stream>>>(h->S, d);
  h->launches++;
  int rc = d2h(out, d, (size_t)N * 16 * sizeof(float), h->stream);
  rc |= sync_stream(h->stream);
  dev_free(d);
  if (rc) return fail(MWB_ECUDA, "readback failed");
#else
  for (int i = 0; i < N; ++i) {
    const Camera c = make_camera(h->S, i);
    float* o = out + (size_t)i * 16;
    o[0] = c.ex; o[1] = c.ey; o[2] = c.ez; o[3] = c.sx; o[4] = c.sy; o[5] = c.sz; o[6] = c.ux; o[7] = c.uy; o[8] = c.uz;
    o[9] = c.fx; o[10] = c.fy; o[11] = c.fz; o[12] = c.px; o[13] = c.py; o[14] = c.za; o[15] = c.zb;
  }
#endif
  return MWB_OK;
}

// ------------------------------------------------------------------ ABI: state exchange
// Device address of one of the handle's per-env state arrays, so that a caller can read it in place (stream-ordered
// after mwb_step) instead of copying the whole state: what the levels' step() put into `info` --
// info["health"] (collecthealth.py:100) is the per-env counter, info["goal_pos"] (tmaze.py:89) three entity-pose rows.
extern "C" int mwb_state_array(mwb_handle* h, int which, void** dev_ptr, int64_t* count) {
  if (!h || !dev_ptr || !count) return fail(MWB_EINVAL, "null argument");
  const int64_t N = h->S.N, E = h->S.E;
  switch (which) {
    case MWB_ARRAY_COUNTER: *dev_ptr = h->S.num_picked; *count = N; break;       // int32 [N]
    case MWB_ARRAY_STEP_COUNT: *dev_ptr = h->S.step_count; *count = N; break;    // int32 [N]
    case MWB_ARRAY_ENT_X: *dev_ptr = h->S.ent_px; *count = E * N; break;         // float64 [E][N]
    case MWB_ARRAY_ENT_Y: *dev_ptr = h->S.ent_py; *count = E * N; break;
    case MWB_ARRAY_ENT_Z: *dev_ptr = h->S.ent_pz; *count = E * N; break;
    case MWB_ARRAY_ENT_DIR: *dev_ptr = h->S.ent_dir; *count = E * N; break;
    default: return fail(MWB_EINVAL, "unknown array");
  }
  return MWB_OK;
}

extern "C" int mwb_get_state(mwb_handle* h, const mwb_state_view* out) {
  if (!h || !out) return fail(MWB_EINVAL, "null argument");
  const int N = h->S.N;
  std::vector<WorldUpload> up(N);
  if (stream_enter(h, h->stream)) return MWB_ECUDA;
#ifndef MWB_HOSTSIM
  gather_kernel<<<(N + 127) / 128, 128, 0, h->stream>>>(h->S, h->d_upload);
  h->launches++;
  CK(cudaGetLastError());
#else
  for (int i = 0; i < N; ++i) gather_one(h->S, i, h->d_upload[i]);
#endif
  if (d2h(up.data(), h->d_upload, (size_t)N * sizeof(WorldUpload), h->stream) != 0) return fail(MWB_ECUDA, "readback failed");
  std::vector<int32_t> rtex;
  if (out->room_tex) {
    rtex.resize((size_t)N * h->S.R * 3);
    if (d2h(rtex.data(), h->S.room_tex, rtex.size() * sizeof(int32_t), h->stream) != 0) return fail(MWB_ECUDA, "readback failed");
  }
  if (sync_stream(h->stream) != 0) return fail(MWB_ECUDA, "sync failed");
  for (int i = 0; i < N; ++i) {
    const WorldUpload& u = up[i];
    const int as = u.agent_slot >= 0 && u.agent_slot < MWB_MAX_ENTS_CAP ? u.agent_slot : 0;
    if (out->agent_pos) for (int k = 0; k < 3; ++k) out->agent_pos[i * 3 + k] = u.ents[as].pos[k];
    if (out->agent_dir) out->agent_dir[i] = u.ents[as].dir;
    if (out->step_count) out->step_count[i] = u.step_count;
    if (out->carrying) out->carrying[i] = u.carrying;
    if (out->num_slots) out->num_slots[i] = u.num_slots;
    if (out->agent_slot) out->agent_slot[i] = u.agent_slot;
    if (out->num_picked_up) out->num_picked_up[i] = u.num_picked;
    if (out->ents) for (int e = 0; e < h->S.E; ++e) out->ents[(size_t)i * h->S.E + e] = u.ents[e];
    if (out->cam) for (int k = 0; k < 4; ++k) out->cam[i * 4 + k] = u.cam[k];
    if (out->env_params) for (int k = 0; k < 12; ++k) out->env_params[i * 12 + k] = u.envp[k];
    if (out->rng) out->rng[i] = u.rng;
  }
  if (out->room_tex) memcpy(out->room_tex, rtex.data(), rtex.size() * sizeof(int32_t));
  if (out->episodes_done) {
    unsigned long long v = 0;
    if (d2h(&v, h->S.episodes_done, sizeof(v), h->stream) != 0 || sync_stream(h->stream) != 0) return fail(MWB_ECUDA, "readback failed");
    *out->episodes_done = (int64_t)v;
  }
  return MWB_OK;
}
