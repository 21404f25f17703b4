// raster.cuh -- K2: tile-based first-person rasteriser, one thread block per environment.
//
// Replaces MiniWorldEnv.render_obs / _render_world / FrameBuffer.resolve / get_depth_map of
// the reference (miniworld.py:1064-1086, 1177-1236; opengl.py:339-435), i.e. the whole
// OpenGL draw + MSAA resolve + glReadPixels round trip, for N environments per launch.
//
// Structure of one block (env i, 10 warps; big frames are cut into several blocks per env):
//   A. a TMA bulk copy stages the env's static quads in shared memory while one thread builds the camera
//      from the glibc-exact cos / sin frame_trig_kernel evaluated and another lays out the frame's draw list.
//   B. geometry: one thread per triangle task (half of a static room quad or of a box face)
//      transforms, lights and sets up its triangle; survivors of frustum / back-face culling
//      are compacted IN DRAW ORDER into shared memory (shuffle prefix scan) -- the set-up
//      triangles of rooms and boxes never touch HBM.  They are ranked front to back and filed into
//      per-half-tile candidate lists.  Mesh entities (thousands of triangles) arrive as per-entity
//      lists prepared AND binned by half-tile by mesh_setup_kernel.
//   C. raster: warps claim 8x4 half-tiles from a shared counter (lane = pixel).  The hot path walks the
//      half-tile's candidate list; mesh lists and half-tiles whose list overflowed fall back to a scan in
//      chunks of 32 triangles, where every lane tests one triangle's bbox / edge functions / nearest depth
//      against the half-tile and a warp ballot yields the survivors.  Each triangle is classified per
//      pixel (lazy single-surface pixels, quad pairs), undecided (pixel, triangle) pairs go through an
//      exact sample-parallel phase on (depth16, slot) keys in shared memory.
//   D. resolve: each pixel shades the distinct triangles its samples see (perspective-
//      correct Gouraud x trilinear texture), box-filters, converts to unorm8; the half-tile is
//      transposed through shared memory and written as 8-byte row segments (or channel-first /
//      float64 greyscale: the reference's observation wrappers fused in); depth (sample 0's
//      16-bit code -> metres) goes out as 32-byte row segments.
// HBM traffic per env-step is the framebuffer written once (+ L2-resident template reads).
#pragma once
#include "raster_core.cuh"

#define MWB_TILE_CAP 16              // candidate triangles listed per half-tile; fuller half-tiles scan the lists

// K2's dynamic shared memory, in this order (host and kernel share the arithmetic):
//   [triangle records (small levels)]
//   [staged static quads  |  visit order u16 + depth keys f32 + slot of every record u16 + per-half-tile candidate
//    counts u16 + lists u16 x MWB_TILE_CAP]      <- one region: the TMA-staged quads are dead once the triangles are set up
//   [frame stage]
struct K2Layout {
  int order_off, zkey_off, slot_off, cnt_off, list_off, tmp_off, stage_off, end;
};
static inline
#ifdef __CUDACC__
__host__ __device__
#endif
K2Layout k2_layout(bool smem_tris, int tri_cap, int stage_bytes, int halves_per_part, int frame_stage_bytes) {
  K2Layout L;
  const int tri_bytes = smem_tris ? tri_cap * (int)sizeof(TriRec) : 0;
  const int cap2 = (tri_cap + 1) & ~1;
  L.order_off = tri_bytes;
  L.zkey_off = L.order_off + cap2 * 2;
  L.slot_off = L.zkey_off + tri_cap * 4;
  L.cnt_off = L.slot_off + cap2 * 2;
  L.list_off = L.cnt_off + ((halves_per_part + 1) & ~1) * 2;
  L.tmp_off = L.list_off + halves_per_part * MWB_TILE_CAP * 2;      // second builder thread's entries before the merge
  const int lists_end = L.tmp_off + halves_per_part * MWB_TILE_CAP * 2, quads_end = tri_bytes + stage_bytes;
  L.stage_off = ((lists_end > quads_end ? lists_end : quads_end) + 15) & ~15;
  L.end = L.stage_off + frame_stage_bytes;
  return L;
}
static inline
#ifdef __CUDACC__
__host__ __device__
#endif
int k2_halves_per_part(int W, int H, int parts) {
  const int tiles_x = (W + 7) >> 3, n_halves = tiles_x * ((H + 3) >> 2);
  int per = (n_halves + parts - 1) / parts;
  // frames cut into several blocks: every part covers whole rows of half-tiles, i.e. a contiguous band of the
  // frame in memory (what lets the band be staged and written out with ordered 16-byte stores)
  if (parts > 1) per = (per + tiles_x - 1) / tiles_x * tiles_x;
  return per;
}

#ifdef __CUDACC__

#define MWB_MAX_SEGS (2 + MWB_MAX_DRAWN)   // rooms, drawn entities, the top view's agent marker
#define MWB_EQ_CAP 96                // exact-phase queue entries per warp
#define MWB_SORT_LIMIT 512            // room triangle lists up to this length are depth-sorted
#define MWB_STAGE_QUAD_BYTES 16384   // static quads up to this size are staged in shared memory

// ---- TMA (bulk async copy) helpers: global -> shared, completion on an mbarrier -----------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

// ---- per-frame trigonometry: thread (env i, k): k < 6 the camera's cos / sin, else entity slot (k - 6) / 2 -----------
__global__ void frame_trig_kernel(DevState S) {
  const int per = 6 + 2 * S.E;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (long long)S.N * per) return;
  const int k = (int)(g / S.N), i = (int)(g % S.N);       // env index fastest: coalesced state reads and stores
  const size_t N = S.N;
  if (k < 6) {
    double ang[3];
    camera_angles(S, i, ang);
    S.cam_trig[(size_t)k * N + i] = (k & 1) ? mwb_libm::sin_glibc(ang[k >> 1]) : mwb_libm::cos_glibc(ang[k >> 1]);
    return;
  }
  const int e = (k - 6) >> 1, j = (k - 6) & 1;
  const int p = e == S.ghost_slot[i] ? S.ghost_proto[i] : (e < S.num_slots[i] ? S.ent_proto[e * N + i] : -1);
  if (p < 0) return;
  const double dir = entity_pose(S, i, e).dir;
  const double deg = S.protos[p].deg_form ? d_div(d_mul(dir, 180.0), 3.141592653589793) : d_mul(dir, 57.29577951308232);
  const double rad = d_div(d_mul((double)(float)deg, 3.141592653589793), 180.0);      // as model_rotation
  S.ent_cs[((size_t)e * 2 + j) * N + i] = (float)(j ? mwb_libm::sin_glibc(rad) : mwb_libm::cos_glibc(rad));
}

// ---- mesh pre-pass: block (env i, entity slot e) sets up that entity's triangles ----------
__global__ void __launch_bounds__(256) mesh_setup_kernel(DevState S, RenderAssets A, ViewSpec view) {
  const int i = blockIdx.x, e = blockIdx.y;
  const size_t N = S.N;
  __shared__ Camera cam;
  __shared__ int warp_tot[8];
  __shared__ int box[4];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  MeshSegInfo* info = S.mesh_seg + (size_t)i * S.E + e;
  const int p = e == S.ghost_slot[i] ? S.ghost_proto[i] : (e < S.num_slots[i] ? S.ent_proto[e * N + i] : -1);
  if (p < 0 || S.protos[p].kind != MWB_KIND_MESH) {
    if (tid == 0) info->count = 0;
    return;
  }
  if (tid == 0) {
    if (view.mode == 1) {
      cam = make_top_camera(S, i, view);
    } else {
      double trig[6];
      for (int k = 0; k < 6; ++k) trig[k] = S.cam_trig[(size_t)k * N + i];
      cam = make_camera(S, i, trig);
    }
    box[0] = box[1] = 0x7fffffff;
    box[2] = box[3] = -1;
  }
  __syncthreads();
  const mwb_proto& pr = S.protos[p];
  const EntPose P = entity_pose(S, i, e);
  const float c = S.ent_cs[((size_t)e * 2 + 0) * N + i], s = S.ent_cs[((size_t)e * 2 + 1) * N + i];   // frame_trig_kernel
  const int ntris = A.meshes[pr.mesh_id].count;
  TriRec* out = S.mesh_tris + ((size_t)i * S.E + e) * S.mesh_cap;
  uint2* out_bbox = S.mesh_bbox + ((size_t)i * S.E + e) * S.mesh_cap;
  int total = 0;
  int x0 = 0x7fffffff, y0 = 0x7fffffff, x1 = -1, y1 = -1;
  for (int start = 0; start < ntris; start += 256) {
    const int t = start + tid;
    TriRec rec;
    int keep = 0;
    if (t < ntris) {
      TriInput in;
      mesh_triangle(A, pr, P, c, s, t, in);
      keep = finish_triangle(cam, in, S.obs_w, S.obs_h, rec) ? 1 : 0;
    }
    int incl = keep;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int woff = 0, chunk = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      int v = warp_tot[w];
      if (w < warp) woff += v;
      chunk += v;
    }
    if (keep) {
      const int pos = total + woff + incl - 1;
      if (pos < S.mesh_cap) {
        out[pos] = rec;
        out_bbox[pos] = make_uint2((unsigned)rec.bx, (unsigned)rec.by);
      }
      x0 = min(x0, rec.bx & 0xFFFF); x1 = max(x1, rec.bx >> 16);
      y0 = min(y0, rec.by & 0xFFFF); y1 = max(y1, rec.by >> 16);
    }
    total += chunk;
    __syncthreads();
  }
  if (x1 >= 0) {
    atomicMin(&box[0], x0); atomicMin(&box[1], y0);
    atomicMax(&box[2], x1); atomicMax(&box[3], y1);
  }
  __syncthreads();
  const int count = total < S.mesh_cap ? total : S.mesh_cap;
  // ---- bin the listed triangles by half-tile (8 x 4 pixels) of the entity's screen box, so that a
  // rasteriser warp scans only the triangles that can touch its half-tile instead of the whole mesh
  __shared__ int bin_cnt[MWB_MAX_BINS + 1];
  __shared__ int scan_tot[8];
  int binned = 0;
  const int c0 = box[0] >> 3, c1 = box[2] >> 3, r0 = box[1] >> 2, r1 = box[3] >> 2;
  const int cols = c1 - c0 + 1, rows = r1 - r0 + 1, nbins = box[2] >= 0 ? cols * rows : 0;
  int* off = S.mesh_bin_off + ((size_t)i * S.E + e) * (MWB_MAX_BINS + 1);
  uint16_t* bidx = S.mesh_bin_idx + ((size_t)i * S.E + e) * ((size_t)MWB_BIN_REFS * S.mesh_cap);
  if (nbins > 0 && nbins <= MWB_MAX_BINS && count > 64 && count <= 65535) {   // bin entries are 16-bit triangle indices
    for (int b = tid; b <= nbins; b += 256) bin_cnt[b] = 0;
    __syncthreads();
    // pass 1: count.  A triangle is listed in a bin if its bbox meets the half-tile and no edge excludes it
    // (the same conservative tests the rasteriser applies per half-tile).
    for (int pass = 0; pass < 2; ++pass) {
      for (int t = tid; t < count; t += 256) {
        const uint2 bb = out_bbox[t];
        const int tc0 = max((int)(bb.x & 0xFFFF) >> 3, c0), tc1 = min((int)(bb.x >> 16) >> 3, c1);
        const int tr0 = max((int)(bb.y & 0xFFFF) >> 2, r0), tr1 = min((int)(bb.y >> 16) >> 2, r1);
        const TriRec& T = out[t];
        float A[3], B[3], K[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { A[k] = T.A[k]; B[k] = T.B[k]; K[k] = T.K[k]; }
        for (int r = tr0; r <= tr1; ++r)
          for (int c = tc0; c <= tc1; ++c) {
            const float fx0 = (float)(c << 3), fy0 = (float)(r << 2);
            if (A[0] * fx0 + B[0] * fy0 + K[0] < 0.0f || A[1] * fx0 + B[1] * fy0 + K[1] < 0.0f ||
                A[2] * fx0 + B[2] * fy0 + K[2] < 0.0f)
              continue;
            const int b = (r - r0) * cols + (c - c0);
            const int pos = atomicAdd(&bin_cnt[b], 1);
            if (pass == 1) bidx[pos] = (uint16_t)t;      // bin_cnt holds the running cursor in pass 2
          }
      }
      __syncthreads();
      if (pass == 0) {
        // exclusive scan of the counts -> offsets (also the cursors of pass 2)
        const int per = (nbins + 255) / 256, b0 = tid * per;
        int sum = 0;
        for (int k = 0; k < per; ++k)
          if (b0 + k < nbins) sum += bin_cnt[b0 + k];
        int incl = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          int v = __shfl_up_sync(0xffffffffu, incl, d);
          if (lane >= d) incl += v;
        }
        if (lane == 31) scan_tot[warp] = incl;
        __syncthreads();
        int base = incl - sum;
        for (int w = 0; w < warp; ++w) base += scan_tot[w];
        int refs = 0;
        for (int w = 0; w < 8; ++w) refs += scan_tot[w];
        __syncthreads();
        for (int k = 0; k < per; ++k)
          if (b0 + k < nbins) {
            const int cnt = bin_cnt[b0 + k];
            bin_cnt[b0 + k] = base;
            off[b0 + k] = base;
            base += cnt;
          }
        if (tid == 0) off[nbins] = refs;
        binned = refs <= MWB_BIN_REFS * S.mesh_cap ? 1 : 0;    // uniform across the block
        __syncthreads();
        if (!binned) break;
      }
    }
  }
  if (tid == 0) {
    info->count = count;
    info->bx = box[2] >= 0 ? (box[0] | (box[2] << 16)) : 0;
    info->by = box[3] >= 0 ? (box[1] | (box[3] << 16)) : 0;
    info->binned = binned;
  }
}

// ---- depth16 code -> metres table (65536 floats, built once per handle by the very function it replaces)
__global__ void depth_lut_kernel(float* __restrict__ lut) {
  const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < 65536u) lut[c] = depth_code_to_metres(c);
}

// ---- K2 --------------------------------------------------------------------------------
// Block size and resident blocks per SM K2 is compiled for (64 registers per thread): the measured default.
// 256 x 3 was slower; 512 x 2 was equal on config 3 and 6 % slower on config 4.
constexpr int MWB_K2_THREADS = 320, MWB_K2_MIN_BLOCKS = 3;
template <int MSAA>
__global__ void __launch_bounds__(MWB_K2_THREADS, MWB_K2_MIN_BLOCKS)
render_kernel(DevState S, RenderAssets A, ViewSpec view, int fmt, uint8_t* __restrict__ obs, float* __restrict__ depth, int env0,
              int parts, int tri_cap, int stage_bytes, int frame_stage_bytes, K2Layout lay, int* __restrict__ overflow) {
  constexpr int THREADS = MWB_K2_THREADS, WARPS = THREADS / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // large frames are cut into `parts` blocks per env (each redoes the cheap geometry phase and
  // rasterises its share of the half-tiles), which evens out the load when few envs are resident
  const int i = env0 + (int)blockIdx.x / parts, part = (int)blockIdx.x % parts;
  // set-up triangles of rooms + boxes: shared memory, or this env's HBM block for big levels
  const size_t tri_bytes = S.room_tris ? 0 : (size_t)tri_cap * sizeof(TriRec);
  TriRec* tris = S.room_tris ? S.room_tris + ((size_t)i * parts + part) * tri_cap : reinterpret_cast<TriRec*>(smem_raw);
  __shared__ Camera cam;
  __shared__ FrameMap fmap;
  __shared__ Segment segs[MWB_MAX_SEGS];
  __shared__ int seg_count[MWB_MAX_SEGS];
  __shared__ int warp_tot[WARPS];
  __shared__ __align__(8) uint64_t quad_bar;
  // everything a warp keeps in shared memory for its current half-tile sits in ONE record, so that a single base
  // register (+ immediate offsets) addresses all of it
  struct __align__(16) WarpScratch {
    uint32_t keys[MSAA][32];          // per-sample keys of explicit pixels: [sample][pixel lane] depth16 << 16 | slot
    uint32_t items[MWB_EQ_CAP];       // queued (pixel, triangle) exact items
    int chunk[32];                    // triangle tested by each lane in the current chunk
    uint8_t stage[4][24];             // RGB of the half-tile, row-major, for the 8-byte row-segment stores
  };
  __shared__ WarpScratch wscratch[WARPS];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = S.obs_w, H = S.obs_h;

  // static room quads of this env: staged into shared memory by one TMA bulk copy that overlaps
  // the camera set-up (fixed-layout levels: 56 quads = 7.6 KB); larger templates are read from L2
  const mwb_quad* gquads = env_quads(S, i);
  const int nq = S.num_quads[geom_index(S, i)];
  const uint32_t quad_bytes = ((uint32_t)nq * (uint32_t)sizeof(mwb_quad) + 15u) & ~15u;
  const bool staged = quad_bytes > 0 && quad_bytes <= (uint32_t)stage_bytes;
  mwb_quad* squads = reinterpret_cast<mwb_quad*>(smem_raw + tri_bytes);
  uint16_t* order = reinterpret_cast<uint16_t*>(smem_raw + lay.order_off);
  float* zkey = reinterpret_cast<float*>(smem_raw + lay.zkey_off);
  uint16_t* tri_slot = reinterpret_cast<uint16_t*>(smem_raw + lay.slot_off);     // record position -> slot (draw order)
  uint16_t* tile_cnt = reinterpret_cast<uint16_t*>(smem_raw + lay.cnt_off);      // candidates per half-tile of this part
  uint16_t* tile_list = reinterpret_cast<uint16_t*>(smem_raw + lay.list_off);    // [half-tile][MWB_TILE_CAP] record positions
  uint16_t* tile_tmp = reinterpret_cast<uint16_t*>(smem_raw + lay.tmp_off);
  // whole-frame RGB stage (frame_stage_bytes > 0): warps drop their pixels here and the block writes the frame
  // out at the end with 16-byte stores in address order
  uint8_t* fstage = smem_raw + lay.stage_off;
  __shared__ float ent_cs[MWB_MAX_DRAWN][2];   // (cos, sin) of every entity slot's model rotation (Box form of the angle)
  __shared__ int next_half;
  if (tid == 0) mbar_init(&quad_bar, 1);
  if (tid < MWB_MAX_SEGS) seg_count[tid] = 0;
  __syncthreads();
  if (tid == 0 && staged) tma_bulk_g2s(squads, gquads, quad_bytes, &quad_bar);
  if (tid == 0) {                      // the camera, from the glibc-exact cos / sin frame_trig_kernel evaluated
    if (view.mode == 1) {
      cam = make_top_camera(S, i, view);
    } else {
      double tr[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) tr[k] = S.cam_trig[(size_t)k * S.N + i];
      cam = make_camera(S, i, tr);
    }
  } else if (tid == 32) {
    fmap = build_frame_map(S, i, view.mode == 1 && view.render_agent != 0);   // meanwhile another warp lays out the draw list
  } else if (tid >= 64 && tid < 64 + 2 * MWB_MAX_DRAWN) {
    // ... and the (cos, sin) of every entity slot's model rotation, for the twelve triangle tasks of each Box
    const int e = (tid - 64) >> 1;
    if (e < S.num_slots[i] && e < S.E) ent_cs[e][tid & 1] = S.ent_cs[((size_t)e * 2 + (tid & 1)) * S.N + i];
  }
  __syncthreads();
  if (staged) mbar_wait(&quad_bar, 0);
  const mwb_quad* quads = staged ? squads : gquads;

  // half-tiles of this block (a frame is cut into `parts` bands of whole half-tile rows)
  const int tiles_x = (W + 7) >> 3;
  const float inv_tiles_x = 1.0f / (float)tiles_x;
  const int halves_y = (H + 3) >> 2;
  const int n_halves = tiles_x * halves_y, per_part = k2_halves_per_part(W, H, parts);
  const int h_begin = min(n_halves, part * per_part), h_end = min(n_halves, h_begin + per_part);
  const int band_row0 = (h_begin / tiles_x) << 2;         // first pixel row of this block's band (parts > 1: whole rows)

  // ---- B. room + box triangles -> shared memory, draw order preserved
  int ntris = 0;
  for (int start = 0; start < fmap.n_tasks; start += THREADS) {
    const int task = start + tid;
    TriRec rec;
    int keep = 0, seg = 0;
    if (task < fmap.n_tasks) keep = task_triangle(S, A, cam, fmap, quads, i, task, W, H, rec, seg, ent_cs) ? 1 : 0;
    // quads stay PAIRS: tasks (2k, 2k + 1) are the fan halves of one planar quad (room quad, box face; the map
    // view's marker pairs with nothing).  If either half survives both keep a record -- the culled one an empty record
    // -- so that records / slots (2k, 2k + 1) always belong together (classify_pixel's pair logic relies on it).
    const int keep_other = __shfl_xor_sync(0xffffffffu, keep, 1);
    const int seg_other = __shfl_xor_sync(0xffffffffu, seg, 1);
    if (!keep && keep_other) {
      empty_record(rec);
      seg = seg_other;
      keep = 1;
    }
    int incl = keep;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int woff = 0, total = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      int v = warp_tot[w];
      if (w < warp) woff += v;
      total += v;
    }
    if (keep) {
      const int pos = ntris + woff + incl - 1;
      if (pos < tri_cap) {
        tris[pos] = rec;
        atomicAdd(&seg_count[seg], 1);
      }
    }
    ntris += total;
    __syncthreads();
  }
  const int n_res = ntris < tri_cap ? ntris : tri_cap;
  // (while thread 0 fills the segment table, everybody computes the depth keys of the visiting order: neither needs the other)
  for (int t = tid; t < n_res; t += THREADS) {
    const TriRec& T = tris[t];
    const float x0 = (float)(T.bx & 0xFFFF), x1 = (float)((T.bx >> 16) + 1), y0 = (float)(T.by & 0xFFFF), y1 = (float)((T.by >> 16) + 1);
    zkey[t] = T.Zc + fminf(T.Za * x0, T.Za * x1) + fminf(T.Zb * y0, T.Zb * y1);
  }
  if (tid == 0) {
    next_half = h_begin + WARPS;
    if (ntris > tri_cap) atomicAdd(overflow, 1);
    // segment table: smem-resident lists are contiguous in draw order; mesh lists live in HBM
    int smem_pos = 0, slot = 0;
    const int last = fmap.n_ents + (fmap.agent_task >= 0 ? 1 : 0);
    for (int k = 0; k <= last; ++k) {
      Segment& sg = segs[k];
      if (k == 0 || k > fmap.n_ents || fmap.ent_kind[k - 1] == MWB_KIND_BOX) {
        sg.tris = tris + smem_pos;
        sg.bbox = nullptr;
        sg.bin_idx = nullptr;
        sg.bin_off = nullptr;
        sg.count = seg_count[k];
        smem_pos += sg.count;
        sg.bx = (W - 1) << 16;
        sg.by = (H - 1) << 16;
      } else {
        const int e = fmap.ent_slot[k - 1];
        const MeshSegInfo mi = S.mesh_seg[(size_t)i * S.E + e];
        sg.tris = S.mesh_tris + ((size_t)i * S.E + e) * S.mesh_cap;
        sg.bbox = S.mesh_bbox + ((size_t)i * S.E + e) * S.mesh_cap;
        sg.bin_idx = mi.binned ? S.mesh_bin_idx + ((size_t)i * S.E + e) * ((size_t)MWB_BIN_REFS * S.mesh_cap) : nullptr;
        sg.bin_off = mi.binned ? S.mesh_bin_off + ((size_t)i * S.E + e) * (MWB_MAX_BINS + 1) : nullptr;
        sg.count = mi.count;
        sg.bx = mi.bx;
        sg.by = mi.by;
      }
      sg.base = slot;
      slot += (sg.count + 1) & ~1;       // even bases: slot parity == record parity inside every list (quad pairs)
    }
  }
  __syncthreads();
  const int nsegs = 1 + fmap.n_ents + (fmap.agent_task >= 0 ? 1 : 0);
  bool has_mesh = false;                 // any list in HBM (mesh entity) in this frame?
  for (int k = 1; k <= fmap.n_ents; ++k) has_mesh = has_mesh || fmap.ent_kind[k - 1] == MWB_KIND_MESH;

  // ---- visiting order of the block-resident triangles (rooms, boxes, the map view's marker): front to back by
  // their nearest possible depth, so that the conservative occlusion tests fire early (the image does not depend
  // on the order: per sample the result is the minimum over (depth code, slot))
  {
    for (int t = tid; t < n_res; t += THREADS) {
      // slot of record t: the records of one list are contiguous, in draw order
      int slot = t;
      for (int k = 0; k < nsegs; ++k) {
        const Segment& sg = segs[k];
        if (sg.bbox != nullptr) continue;
        const int start = (int)(sg.tris - tris);
        if (t >= start && t < start + sg.count) slot = sg.base + (t - start);
      }
      tri_slot[t] = (uint16_t)slot;
    }
    if (n_res <= MWB_SORT_LIMIT) {
      for (int t = tid; t < n_res; t += THREADS) {
        const float z = zkey[t];
        int rank = 0;
        for (int q = 0; q < n_res; ++q) {
          const float zq = zkey[q];
          rank += (zq < z || (zq == z && q < t)) ? 1 : 0;
        }
        order[rank] = (uint16_t)t;
      }
    } else {
      for (int t = tid; t < n_res; t += THREADS) order[t] = (uint16_t)t;
    }
    __syncthreads();
  }

  // ---- candidate lists: one THREAD per half-tile walks the block-resident triangles in visiting order and files
  // those that can touch its half-tile (bbox + the three conservative edge bounds) -- the test every rasteriser warp
  // used to repeat per 32-triangle chunk is done once per (triangle, half-tile) pair here, lanes = half-tiles, the
  // triangle fields broadcast from shared memory.  A half-tile with more than MWB_TILE_CAP candidates keeps only
  // the count; its warp then scans the lists the old way.
  // Two threads (adjacent lanes) per half-tile: the first takes the nearer half of the ranked triangles, the second the
  // farther half (into a scratch list appended behind the first's), which halves this phase's critical path.
  {
    const int n_tiles = h_end - h_begin, mid = (n_res + 1) >> 1;
    for (int w0 = 0; w0 < 2 * n_tiles; w0 += THREADS) {
      const int w = w0 + tid, hl = w >> 1, j = w & 1;
      int cnt = 0;
      if (hl < n_tiles) {
        const int half = h_begin + hl;
        const int hrow = (int)(((float)half + 0.5f) * inv_tiles_x), hcol = half - hrow * tiles_x;
        const int tx0 = hcol << 3, ty0 = hrow << 2;
        const float fx0 = (float)tx0, fy0 = (float)ty0;
        uint16_t* dst = (j ? tile_tmp : tile_list) + hl * MWB_TILE_CAP;
        const int q1 = j ? n_res : mid;
        for (int q = j ? mid : 0; q < q1; ++q) {
          const int p = order[q];
          const TriRec& t = tris[p];
          const int bx = t.bx, by = t.by;
          if ((bx & 0xFFFF) > tx0 + 7 || (bx >> 16) < tx0 || (by & 0xFFFF) > ty0 + 3 || (by >> 16) < ty0) continue;
          if (t.A[0] * fx0 + t.B[0] * fy0 + t.K[0] < 0.0f || t.A[1] * fx0 + t.B[1] * fy0 + t.K[1] < 0.0f ||
              t.A[2] * fx0 + t.B[2] * fy0 + t.K[2] < 0.0f)
            continue;
          if (cnt < MWB_TILE_CAP) dst[cnt] = (uint16_t)p;
          ++cnt;
        }
      }
      const int other = __shfl_xor_sync(0xffffffffu, cnt, 1);      // (THREADS is a multiple of 32: whole warps get here)
      if (hl < n_tiles) {
        if (j) {                                  // append behind the first thread's entries
          uint16_t* lst = tile_list + hl * MWB_TILE_CAP;
          const uint16_t* src = tile_tmp + hl * MWB_TILE_CAP;
          for (int k = 0; k < cnt && other + k < MWB_TILE_CAP; ++k) lst[other + k] = src[k];
        } else {
          tile_cnt[hl] = (uint16_t)min(cnt + other, 0xFFFF);
        }
      }
    }
  }
  __syncthreads();

  // ---- C/D. one warp per 8x4 half-tile (lane = one pixel; an 8x8 tile is two of them)
  const int lx = lane & 7, ly = lane >> 3;
  const SegLookup fetch{segs, nsegs};
  // exact-phase work is done sample-parallel: lane -> (queued item lane / MSAA, sample lane % MSAA)
  constexpr int IPR = 32 / MSAA;                 // items per round
  const int my_s = lane % MSAA;
  float my_sx, my_sy;
  sample_xy_dyn<MSAA>(my_s, my_sx, my_sy);
  WarpScratch& ws = wscratch[warp];
  uint32_t(*skeys)[32] = ws.keys;
  uint32_t* equeue = ws.items;
  // half-tiles in row-major order of 8x4 blocks: index h -> column h % tiles_x, row h / tiles_x
  // the first WARPS half-tiles go one to each warp; after that warps claim half-tiles from next_half (set with the
  // segment table, several barriers ago), which evens out the per-warp work
  int half = h_begin + warp;
#pragma unroll 1
  while (half < h_end) {
    const int hrow = (int)(((float)half + 0.5f) * inv_tiles_x), hcol = half - hrow * tiles_x;   // exact: half < 2^20
    const int tx0 = hcol << 3, ty0 = hrow << 2;
    const int hl = half - h_begin;
    int nxt = 0;               // claim the next half-tile now; the atomic's latency hides behind this one
    if (lane == 0) nxt = atomicAdd(&next_half, 1);
    half = __shfl_sync(0xffffffffu, nxt, 0);
    const int px = tx0 + lx, py = ty0 + ly;
    PixelState<MSAA> P;
    pixel_init(P);
#pragma unroll
    for (int s = 0; s < MSAA; ++s) skeys[s][lane] = MWB_SKY_KEY;
    int qn = 0;                                  // queued exact items (warp-uniform)

    // Exact processing of the queued (pixel, triangle) items, MSAA lanes per item: every lane
    // evaluates one sample and folds it into the pixel's key with an integer atomicMin
    // (order-independent, hence deterministic).  Then explicit pixels refresh their bound.
    auto flush = [&]() {
      __syncwarp();
#pragma unroll 1
      for (int r = 0; r < qn; r += IPR) {
        const int qi = r + lane / MSAA;
        if (qi < qn) {
          const uint32_t it = equeue[qi];
          const int slot = (int)(it & 0xFFFFu), pl = (int)((it >> 16) & 31u);
          const HotTri t = load_hot(&fetch(slot));
          const float xs = (float)(tx0 + (pl & 7)) + my_sx, ys = (float)(ty0 + (pl >> 3)) + my_sy;
          const uint32_t key = sample_key(t, slot, xs, ys, (it >> 21) & 1u);
          if (key != 0xFFFFFFFFu) atomicMin(&skeys[my_s][pl], key);
        }
      }
      __syncwarp();
      if (P.mode == MWB_PX_EXPLICIT) {
        uint32_t km = skeys[0][lane];
#pragma unroll
        for (int s = 1; s < MSAA; ++s) km = max(km, skeys[s][lane]);
        P.bound = (float)(km >> 16);
      }
      qn = 0;
    };

    // Queue what this lane's pixel could not decide for the candidates flagged in `mine` (first the lazily held
    // triangle -- or both halves of a lazily held quad pair -- which must now be materialised); the queue is drained
    // sample-parallel by flush().  slot_of(b) = slot of candidate b.
    auto enqueue = [&](uint32_t mine, uint32_t mine_full, auto slot_of) {
      int need_mat = (mine != 0 && P.mode == MWB_PX_LAZY) ? (lazy_is_pair(P) ? 2 : 1) : 0;
      if (mine != 0 && P.mode != MWB_PX_EXPLICIT) {
        P.bound = P.mode == MWB_PX_LAZY ? P.lazy_chi : 65535.0f;   // still an upper bound after materialisation
        P.mode = MWB_PX_EXPLICIT;
      }
#pragma unroll 1
      for (;;) {
        const bool has = need_mat != 0 || mine != 0;
        const uint32_t bal = __ballot_sync(0xffffffffu, has);
        if (!bal) break;
        const int cnt = __popc(bal);
        if (qn + cnt > MWB_EQ_CAP) flush();
        if (has) {
          const int pos = qn + __popc(bal & ((1u << lane) - 1u));
          uint32_t item;
          if (need_mat == 2) {          // a pair: both halves, each with its edge tests (the diagonal decides)
            item = ((uint32_t)lane << 16) | (uint32_t)(P.lazy_slot ^ 1);
            need_mat = 3;
          } else if (need_mat) {
            item = (need_mat == 1 ? (1u << 21) : 0u) | ((uint32_t)lane << 16) | (uint32_t)P.lazy_slot;
            need_mat = 0;
          } else {
            const int b = __ffs(mine) - 1;
            mine &= mine - 1;
            item = (((mine_full >> b) & 1u) << 21) | ((uint32_t)lane << 16) | (uint32_t)slot_of(b);
          }
          equeue[pos] = item;
        }
        qn += cnt;
      }
    };

    // ---- hot path: this half-tile's list of block-resident triangles (already tested against the half-tile, in
    // front-to-back order); every listed triangle is triaged at each lane's pixel (warp-uniform loop)
    const int n_cand = tile_cnt[hl];
    const bool listed = n_cand <= MWB_TILE_CAP;
    if (listed) {
      const uint16_t* list = tile_list + hl * MWB_TILE_CAP;
      uint32_t mine = 0, mine_full = 0;
#pragma unroll 1
      for (int q = 0; q < n_cand; ++q) {
        const int p = list[q];
        const ClassTri ct = load_class(tris + p);
        const int cls = classify_pixel<MSAA>(ct, (int)tri_slot[p], px, py, P, tris + (p ^ 1), (p & 1) ? 1 : 2);
        if (cls) mine |= 1u << q;
        if (cls == 2) mine_full |= 1u << q;
      }
      enqueue(mine, mine_full, [&](int b) { return (int)tri_slot[list[b]]; });
    }

    // ---- generic path: the mesh lists in HBM (and, for a half-tile whose candidate list overflowed, the resident lists)
#pragma unroll 1
    for (int sgi = (listed && !has_mesh) ? nsegs : 0; sgi < nsegs; ++sgi) {
      const Segment sg = segs[sgi];
      if (sg.count == 0 || (listed && sg.bbox == nullptr)) continue;
      if ((sg.bx & 0xFFFF) > tx0 + 7 || (sg.bx >> 16) < tx0 || (sg.by & 0xFFFF) > ty0 + 3 || (sg.by >> 16) < ty0) continue;
      const bool pairable = sg.bbox == nullptr;   // resident lists hold quad pairs in adjacent records
      // which triangles to visit: a binned mesh list only the triangles filed under this half-tile; else the whole list
      const uint16_t* ord = nullptr;
      int lo = 0, hi = sg.count;
      if (sg.bin_off != nullptr) {
        const int cols = ((sg.bx >> 16) >> 3) - ((sg.bx & 0xFFFF) >> 3) + 1;
        const int bin = (hrow - ((sg.by & 0xFFFF) >> 2)) * cols + (hcol - ((sg.bx & 0xFFFF) >> 3));
        lo = sg.bin_off[bin];
        hi = sg.bin_off[bin + 1];
        ord = sg.bin_idx;
      }
#pragma unroll 1
      for (int cb = lo; cb < hi; cb += 32) {
        // largest depth code stored anywhere in this half-tile: a triangle that cannot beat it is dropped whole
        const float tile_bound = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(pixel_bound(P), 0.0f))));
        const int j = cb + lane;
        int idx = -1;
        if (j < hi) {
          idx = ord ? (int)ord[j] : j;
          bool hit;
          if (sg.bbox != nullptr) {          // mesh list: coalesced bbox test first, record only if it passes
            const uint2 bb = sg.bbox[idx];
            const int bx0 = bb.x & 0xFFFF, bx1 = bb.x >> 16, by0 = bb.y & 0xFFFF, by1 = bb.y >> 16;
            hit = bx0 <= tx0 + 7 && bx1 >= tx0 && by0 <= ty0 + 3 && by1 >= ty0;
          } else {
            const TriRec& t = sg.tris[idx];
            const int bx0 = t.bx & 0xFFFF, bx1 = t.bx >> 16, by0 = t.by & 0xFFFF, by1 = t.by >> 16;
            hit = bx0 <= tx0 + 7 && bx1 >= tx0 && by0 <= ty0 + 3 && by1 >= ty0;
          }
          if (hit) {
            const TriRec& t = sg.tris[idx];
            const float fx0 = (float)tx0, fy0 = (float)ty0;
#pragma unroll
            for (int k = 0; k < 3; ++k)   // half-tile entirely outside one edge?
              if (t.A[k] * fx0 + t.B[k] * fy0 + t.K[k] < 0.0f) hit = false;
            // nearest depth the triangle can have inside the half-tile vs everything already stored
            if ((t.Za * fx0 + t.Zb * fy0 + t.Kz) * 65535.0f - 1.0f > tile_bound) hit = false;
          }
          if (!hit) idx = -1;
        }
        uint32_t mask = __ballot_sync(0xffffffffu, idx >= 0);
        __syncwarp();
        ws.chunk[lane] = idx;
        __syncwarp();
        // phase 1 (warp-uniform): triage every surviving triangle at this lane's pixel
        uint32_t mine = 0, mine_full = 0;
#pragma unroll 1
        while (mask) {
          const int b = __ffs(mask) - 1;
          mask &= mask - 1;
          const int tb = ws.chunk[b];
          const ClassTri ct = load_class(sg.tris + tb);
          const int cls = classify_pixel<MSAA>(ct, sg.base + tb, px, py, P, pairable ? sg.tris + (tb ^ 1) : nullptr, (tb & 1) ? 1 : 2);
          if (cls) mine |= 1u << b;
          if (cls == 2) mine_full |= 1u << b;
        }
        // phase 2: queue what this pixel could not decide
        enqueue(mine, mine_full, [&](int b) { return sg.base + ws.chunk[b]; });
      }
    }
    if (qn) flush();

    // Lazy pixels join the common resolve path as "all samples see lazy_slot", so that the
    // (expensive) shading code runs once for the whole warp instead of once per mode.
    uint8_t rgb[3];
    uint32_t code0;
    int lazy_slot = -1;
    if (P.mode == MWB_PX_LAZY) {
      lazy_slot = P.lazy_slot;
      if (depth != nullptr) {              // only the depth map needs sample 0's exact code
        int owner = lazy_slot;
        if (lazy_is_pair(P)) {             // which half of the quad owns sample 0: its diagonal edge decides
          const float xs = (float)px + sample_x<MSAA>(0), ys = (float)py + sample_y<MSAA>(0);
          if (!pair_sample_in_first(fetch(lazy_slot), (lazy_slot & 1) ? 1 : 2, xs, ys)) owner = lazy_slot ^ 1;
        }
        code0 = sample0_code<MSAA>(fetch(owner), px, py);
      } else {
        code0 = 0u;
      }
    } else {
#pragma unroll
      for (int s = 0; s < MSAA; ++s) P.keys[s] = skeys[s][lane];
      code0 = P.keys[0] >> 16;
    }
    resolve_pixel<MSAA>(A, cam, fetch, P.keys, lazy_slot, px, py, rgb);
    if (obs != nullptr && fmt == MWB_OBS_GREY_F64) {
      // GreyscaleWrapper fused into the epilogue: float64 [N][H][W][1], eight consecutive doubles per tile row
      if (px < W && py < H) reinterpret_cast<double*>(obs)[((size_t)i * H + py) * W + px] = grey_f64(rgb[0], rgb[1], rgb[2]);
    } else if (obs != nullptr && frame_stage_bytes > 0) {
      if (px < W && py < H) {
        if (fmt == MWB_OBS_CWH_U8) {
#pragma unroll
          for (int c = 0; c < 3; ++c) fstage[((size_t)c * W + px) * H + py] = rgb[c];
        } else {
#pragma unroll
          for (int c = 0; c < 3; ++c) fstage[((size_t)(py - band_row0) * W + px) * 3 + c] = rgb[c];
        }
      }
    } else if (obs != nullptr) {
      __syncwarp();
#pragma unroll
      for (int c = 0; c < 3; ++c) ws.stage[ly][lx * 3 + c] = rgb[c];
      __syncwarp();
      if (fmt == MWB_OBS_CWH_U8) {
        // PyTorchObsWrapper's transpose(2, 1, 0) fused into the epilogue: [N][3][W][H]; a half-tile is, per channel
        // and column, four consecutive bytes
        if (lane < 24) {
          const int c = lane >> 3, x = tx0 + (lane & 7);
          if (x < W) {
            uint8_t* dst = obs + (((size_t)i * 3 + c) * W + x) * H + ty0;
            const uint8_t b0 = ws.stage[0][(lane & 7) * 3 + c], b1 = ws.stage[1][(lane & 7) * 3 + c];
            const uint8_t b2 = ws.stage[2][(lane & 7) * 3 + c], b3 = ws.stage[3][(lane & 7) * 3 + c];
            if (ty0 + 4 <= H && (H & 3) == 0) {
              *reinterpret_cast<uint32_t*>(dst) = (uint32_t)b0 | ((uint32_t)b1 << 8) | ((uint32_t)b2 << 16) | ((uint32_t)b3 << 24);
            } else {
              if (ty0 + 0 < H) dst[0] = b0;
              if (ty0 + 1 < H) dst[1] = b1;
              if (ty0 + 2 < H) dst[2] = b2;
              if (ty0 + 3 < H) dst[3] = b3;
            }
          }
        }
      } else if (lane < 12) {   // 4 rows x 3 segments of 8 bytes
        const int row = lane / 3, seg = lane % 3;
        const int y = ty0 + row;
        if (y < H && (W & 7) == 0) {    // rows start 8-byte aligned only when W is a multiple of 8
          uint2 v = *reinterpret_cast<const uint2*>(&ws.stage[row][seg * 8]);
          *reinterpret_cast<uint2*>(obs + ((size_t)i * H + y) * W * 3 + (size_t)tx0 * 3 + seg * 8) = v;
        } else if (y < H) {   // W not a multiple of 8 (ragged right edge, unaligned rows): byte stores
          for (int q = 0; q < 8; ++q) {
            int bcol = seg * 8 + q;
            if (tx0 + bcol / 3 < W) obs[((size_t)i * H + y) * W * 3 + (size_t)tx0 * 3 + bcol] = ws.stage[row][bcol];
          }
        }
      }
    }
    // FrameBuffer.get_depth_map's float32 formula (two IEEE divisions per pixel) tabulated once per handle
    if (depth != nullptr && px < W && py < H)
      depth[((size_t)i * H + py) * W + px] = S.depth_lut != nullptr ? __ldg(S.depth_lut + code0) : depth_code_to_metres(code0);
  }
  if (obs != nullptr && frame_stage_bytes > 0) {
    __syncthreads();
    // this block's band of the frame (the whole frame when parts == 1; channel-first frames are only staged whole)
    const int band_rows = min(H, ((h_end + tiles_x - 1) / tiles_x) << 2) - band_row0;
    const size_t frame = (size_t)W * H * 3, band = (size_t)max(band_rows, 0) * W * 3;
    uint8_t* dst = obs + (size_t)i * frame + (size_t)band_row0 * W * 3;
    const int vec = (int)(band >> 4);
    for (int o = tid; o < vec; o += THREADS) reinterpret_cast<uint4*>(dst)[o] = reinterpret_cast<const uint4*>(fstage)[o];
    for (int o = (vec << 4) + tid; o < (int)band; o += THREADS) dst[o] = fstage[o];
  }
}

#endif  // __CUDACC__
