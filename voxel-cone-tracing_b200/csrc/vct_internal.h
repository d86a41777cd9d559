// vct_internal.h -- context, parameter block and device helpers shared by the kernels of libvct_b200.
// Compiled with --fmad=false: every float expression below is a sequence of single IEEE binary32
// operations in source order, which is what makes coverage / depth-slice / shadow-compare decisions
// reproducible bit for bit against the CPU oracle (DESIGN.md "Defined semantics").
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/vct_c_api.h"

#define VCT_MAX_CONES 16
#define VCT_EVENT_GENS 4

namespace vct {

// Uniform block handed to every kernel by value (fits in constant bank param space).
struct Params {
  int V;                 // VoxelDimensions
  int levels;            // log2(V)+1
  float grid_world;      // VoxelGridWorldSize
  int S;                 // ShadowMapSize
  int W, H;              // screen_width, screen_height
  float model[16], model_view[16], proj[16], depth_mvp[16], projx[16], projy[16], projz[16];
  float cam[3], light[3];
  float ambient;
  int n_cones;
  float cone_dir[VCT_MAX_CONES * 3];
  float cone_w[VCT_MAX_CONES];
  float diffuse_tan, spec_tan, step_mult, max_dist, max_alpha;
  int pcf_radius;
  float shadow_bias;
  int coverage;          // 0 CENTER, 1 MSAA4_ANY, 2 CONSERVATIVE
  int bounces;
  int row_begin, row_end;   // rows of the frame this context renders (row-band sharding); row_end 0 = H
  // row sharding by INTERLEAVED strips of 8 rows (one cone_trace block row): this context renders the strips g with
  // g % row_il == row_ph.  Costs vary smoothly over the image (ceiling vs floor), so dealing thin strips round-robin
  // balances the ranks to a few per cent where contiguous bands differ by ~15 %.  row_il <= 1: off (bands apply).
  int row_il, row_ph;
};

struct MaterialDev {
  cudaTextureObject_t diffuse, specular, height;
  int dw, dh, sw, sh, hw, hh;   // level-0 sizes (for the implicit LOD and HeightTextureSize)
  float shininess;
  int alpha_test;               // diffuse texture has texels with alpha < 255
};

struct TextureEntry {
  cudaMipmappedArray_t array = nullptr;
  cudaTextureObject_t tex = 0;
  int w = 0, h = 0;
  bool has_alpha = false;
};

struct MaterialHost { int d = -1, s = -1, h = -1; float shininess = 20.0f; };

// Kernels that count their work, numbered as vct_debug_counter reads them: executed textureLod calls of cone_trace
// (vct_cone_samples), texels visited by the voxel view, textureLod calls of the probe bake, texels visited by ray casts
enum StepCounter { STEPS_CONE, STEPS_VIEW, STEPS_PROBES, STEPS_RAYS, N_STEP_COUNTERS };

// Device counters, one cache line each to keep unrelated atomics apart.
struct Counters {
  unsigned int n_fragments;   unsigned int pad0[31];
  // tile-item queue of the current raster pass: written by raster_small, consumed by raster_tiles (stream order), so
  // the three words share a line and are reset by ONE 12-byte memset per pass (reset_item_queue).  items_overflow is
  // the per-pass twin of the sticky `overflow`: when set, raster_tiles consumes nothing (the queue holds stale items).
  unsigned int n_items, next_item, items_overflow; unsigned int pad1[29];
  unsigned int n_touched;     unsigned int pad2[31];
  unsigned int overflow;      unsigned int pad3[31];   // sticky until read by check_overflow
  // the work of the last launch of each counting kernel (StepCounter) as 64 partial counters, one 32-byte sector each
  // (65 K warps adding into ONE address serialise in a single L2 atomic unit): count_steps adds, reset_steps clears,
  // read_steps sums them
  unsigned long long steps[N_STEP_COUNTERS][64 * 4];
};
static_assert(offsetof(Counters, steps) == 512, "the step counters start after the four counter lines");
static_assert(sizeof(Counters) == 8704, "Counters: four counter lines and four step counters");

// Per-vertex transform cache written once per frame by vertex_pass -- the vertex-shader stage of the three
// reference programs (Voxelization.vs:15-22, VoxelConeTracing.vs:23-37) evaluated once per vertex, as GL does,
// instead of once per triangle / tile / pixel.  Same arithmetic as the per-use form, so every consumer sees
// bit-identical values.
struct VertexCache {
  float4* world;   // ModelMatrix * (Position,1)
  float4* dc;      // DepthMVP * (Position,1), xyz*0.5+0.5
  float4* clip;    // window-homogeneous (X, Y, w, z_clip); w = NaN if any clip coordinate is not finite
  float4* nrm_u;   // (ModelMatrix*(Normal,0)).xyz, TexCoords.x
  float4* tan_v;   // (ModelMatrix*(Tangent,0)).xyz, TexCoords.y
  float4* bit;     // (ModelMatrix*(BiTangent,0)).xyz, 0
};

struct TileItem { uint32_t tri; uint32_t origin; };   // origin = tile_x | tile_y << 16 (in tiles)

}  // namespace vct

struct vct_context {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  vct::Params P{};
  bool profile = true;
  int dense_resolve = 0;
  int shard_shadow = 0;         // 1 (set before vct_comm_init): vct_draw_depth rasterises this rank's triangle share and
                                // min-reduces it into every rank's D24 image through the switch (multimem.red.min.u32)
  int grid_format = 0;
  size_t max_fragments = 16u << 20;
  size_t max_items = 4u << 20;

  // scene
  float* d_verts = nullptr; uint32_t* d_idx = nullptr; uint16_t* d_trimat = nullptr;
  size_t nv = 0, nt = 0;
  std::vector<vct::TextureEntry> textures;
  std::vector<vct::MaterialHost> materials;
  vct::MaterialDev* d_materials = nullptr; size_t n_materials_dev = 0; bool materials_dirty = true;
  cudaTextureObject_t white_tex = 0; cudaMipmappedArray_t white_arr = nullptr;

  // Two frame slots (grid pyramid + touched list, visibility buffer, vertex cache): vct_frame / vct_draw_voxels
  // build into the slot that the previous frame's cone_trace is NOT reading, so consecutive frames pipeline.
  int cur = 0;                                   // slot of the most recent voxelisation / the one vct_render reads
  vct::VertexCache vcache2[2]{}; size_t vcache_nv[2] = {0, 0}; bool vcache_valid[2] = {false, false};
  vct::Params vcache_params[2]{};
  cudaEvent_t slot_read_done[2] = {nullptr, nullptr};   // recorded on the main stream after the last reader of a slot
  bool slot_read_pending[2] = {false, false};
  cudaStream_t stream_vox = nullptr; cudaEvent_t ev_vox_done = nullptr, ev_vtx_done = nullptr;
  unsigned long long scene_epoch = 1, frame_epoch = 0;   // device-side inputs changed since the last vct_frame?
  int pipeline_frames = 1;

  // shadow map (u32 d24, linear)
  uint32_t* d_depth = nullptr; int depth_S = 0; bool depth_valid = false;
  cudaArray_t depth_array = nullptr; cudaTextureObject_t depth_tex = 0;   // same texels as a 2D array for tex2Dgather
  cudaSurfaceObject_t depth_surf = 0;                                     // ... written by depth_to_array, as floats

  // voxel grid
  int grid_V = 0; int grid_fmt_alloc = -1;       // format the slots were allocated with (0 RGBA8, 1 RGBA16F)
  unsigned long long* d_accum = nullptr;       // 2 x u64 per voxel: (r<<32|g), (b<<32|count)
  struct GridBuf {
    cudaMipmappedArray_t array = nullptr;
    std::vector<cudaSurfaceObject_t> surf;
    cudaTextureObject_t tex = 0;
    uint32_t* touched = nullptr;               // voxels whose level-0 texel may be non-zero (exact when list_valid)
    unsigned int* n_touched = nullptr;         // device counter
    bool list_valid = true;                    // false: level 0 was written densely, a dense clear is needed before reuse
    // sparse mip build: one flag per 32x8x8 brick of level 0 (= one mip_fused3 block).  dirty_now is set by the sparse
    // resolve for every brick that holds a non-zero texel (exact superset while occ_valid); dirty_prev is the same for
    // the content this slot held before the current voxelisation, i.e. the bricks the sparse clear zeroed.  While
    // dirty_valid, now | prev covers every brick that changed since the slot's pyramid was last built (mips_current),
    // and only those are re-filtered -- the cost follows the occupied surface, not V^3.
    unsigned char* dirty_now = nullptr; unsigned char* dirty_prev = nullptr;
    bool dirty_valid = false, occ_valid = false, mips_current = false;
  } grid[2];
  size_t touched_cap = 0;
  // first-touch bits of the voxelisation in flight (one bit per voxel, x-runs of 32 per word): vox_shade sets a bit for
  // every voxel it touches first, vox_compact_mask turns the bits into the touched list IN MEMORY ORDER and clears them
  uint32_t* d_occ_mask = nullptr;
  // fused sharded voxelisation: external symmetric accumulator + occupancy mask (local view and multicast view)
  unsigned long long* shared_local = nullptr; unsigned long long* shared_mc = nullptr;
  // library-owned multi-GPU state (vct_comm.cu): symmetric segments, multicast mapping, bootstrap sockets.  When the
  // segments are mapped without a multicast object, shared_peers + r * shared_seg is rank r's inbox (unicast stores).
  void* comm = nullptr; unsigned char* shared_peers = nullptr; size_t shared_seg = 0;
  uint32_t* mask_prev[2] = {nullptr, nullptr}; int mask_prev_V = 0;   // occupancy mask of what each slot's level 0 holds
  bool mask_valid[2] = {false, false};                                // ... and whether it is exact
  uint32_t* d_push_list = nullptr; unsigned int* d_push_count = nullptr; size_t push_cap = 0;   // voxels this rank touched
  // exchange flavour: 0 = inbox (records multicast with multimem.st, merged locally; default), 1 = in-switch reduction
  // (multimem.red into a dense symmetric accumulator + occupancy mask)
  int shared_exchange = 0, shared_world = 1, shared_rank = 0, exchange_parity = 0;
  bool shared_frame_open = false;                // vct_frame_shared_begin issued, vct_frame_shared_end pending
  int tri_interleave = 1, tri_phase = 0;         // voxelisation takes every tri_interleave-th block of 128 triangles
  size_t exchange_cap = 0, exchange_cap_user = 0; // records per rank and parity in the inbox (user 0 = auto: min(V^3, 32 V^2))
  int accum_list_slot = -1;                    // slot whose touched list describes the accumulator's non-zero cells;
                                               // -1 = dense dirty, -2 = all zero (left so by vox_push_shared)

  void* d_voxrec = nullptr; size_t voxrec_nt = 0;   // per-triangle voxelisation records (vct_voxelize.cu)

  // work queues
  uint2* d_frags = nullptr; size_t frags_cap = 0;
  vct::TileItem* d_items = nullptr; size_t items_cap = 0;
  vct::Counters* d_counters = nullptr;
  unsigned int* h_overflow = nullptr;           // pinned [VCT_ASYNC_FRAMES][2]: overflow words copied out behind each async frame

  // second stream: the visibility pass is independent of voxelisation + mip and runs beside them in vct_frame
  cudaStream_t stream2 = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  vct::TileItem* d_items_vis = nullptr; size_t items_vis_cap = 0; vct::Counters* d_counters_vis = nullptr;
  int overlap_visibility = 1;

  // frame
  unsigned long long* d_vis2[2] = {nullptr, nullptr}; uchar4* d_frame = nullptr; int frame_W = 0, frame_H = 0;
  uchar4* last_frame = nullptr;   // where the most recent cone_trace wrote (d_frame, an async ring slot or a sharded-frame slot)
  // ring of device frame buffers for vct_frame_async (up to VCT_ASYNC_FRAMES frames in flight)
  uchar4* d_frame2[3] = {nullptr, nullptr, nullptr}; int frame2_W = 0, frame2_H = 0;
  cudaStream_t copy_stream = nullptr; cudaEvent_t ev_rendered[3]{}, ev_copied[3]{}; bool in_flight[3] = {false, false, false};
  unsigned frame_seq = 0, frame_oldest = 0;
  uint8_t* h_frame_pinned = nullptr; size_t h_frame_bytes = 0;
  // device staging of the calls that run a kernel on host arrays (host_round_trip): their inputs and outputs, grown on
  // demand and kept.  Each such call ends in a stream synchronise, so the next one finds the buffer free.
  unsigned char* d_stage = nullptr; size_t stage_bytes = 0;

  // timing
  // pass events, VCT_EVENT_GENS generations deep: every frame call (vct_frame, vct_frame_shared_begin) moves to the
  // next generation, so that the passes of the last few frames can be placed on ONE time axis (vct_pass_timeline) --
  // how the streams of consecutive frames overlap is otherwise invisible without a system profiler
  cudaEvent_t ev_begin[4][VCT_PASS_COUNT]{}, ev_end[4][VCT_PASS_COUNT]{};
  bool ev_recorded[4][VCT_PASS_COUNT]{};
  int ev_gen = 0;
  cudaEvent_t ev_ref = nullptr;   // time zero of vct_pass_timeline (recorded when Profile is switched on)
  uint64_t launches = 0;

  std::string err;
};

namespace vct {

int set_error(vct_context* c, int code, const std::string& msg);
int check_cuda(vct_context* c, cudaError_t e, const char* what);
#define VCT_CUDA(c, call)                                              \
  do {                                                                 \
    int _rc = vct::check_cuda((c), (call), #call);                     \
    if (_rc) return _rc;                                               \
  } while (0)

struct PassTimer {
  vct_context* c; int pass, gen;
  // the shadow map is not part of a frame: its events live in generation 0 and survive the generation changes
  PassTimer(vct_context* c_, int p) : c(c_), pass(p), gen(p == VCT_PASS_DEPTH ? 0 : c_->ev_gen) {
    if (c->profile) { cudaEventRecord(c->ev_begin[gen][p], c->stream); }
  }
  ~PassTimer() {
    if (c->profile) { cudaEventRecord(c->ev_end[gen][pass], c->stream); c->ev_recorded[gen][pass] = true; }
  }
};

// pass entry points implemented in the kernel files
int ensure_grid(vct_context* c);
int ensure_shadow(vct_context* c);
int ensure_frame(vct_context* c);
int ensure_queues(vct_context* c);
int sync_materials(vct_context* c);
int ensure_vertex_cache(vct_context* c);
int launch_shadow(vct_context* c);
int launch_voxel_clear(vct_context* c);
int begin_voxel_slot(vct_context* c);     // flips c->cur to the other slot (after making it safe to overwrite)
void mark_slot_read(vct_context* c);
void next_event_generation(vct_context* c);   // pass events of the next frame go to the next generation       // records slot_read_done[c->cur] on the main stream
int launch_voxelize(vct_context* c, size_t tb, size_t te);
int launch_resolve(vct_context* c, bool dense);
int launch_voxelize_shared(vct_context* c, size_t tb, size_t te);
int launch_resolve_shared(vct_context* c);
int launch_voxelize_inbox_into_slot(vct_context* c, size_t tb, size_t te);   // inbox flavour, slot already chosen
int launch_mip(vct_context* c);
int launch_visibility(vct_context* c);
int launch_cone(vct_context* c);
int launch_reinject(vct_context* c);
int launch_voxel_view(vct_context* c, int level, const float inv_vp[16], uint32_t* d_voxel);   // vct_view.cu
// queries on the current pyramid, all pointers on the device
int launch_trace_cones(vct_context* c, size_t n, const float* starts, const float* dirs, const float* tans, float* out,
                       uint32_t* steps);
int launch_sample_voxels(vct_context* c, size_t n, const float* pos, const float* lod, float* out);
int launch_probes(vct_context* c, size_t n, const float* xyz, float* out, uint32_t* steps);
int launch_cast_rays(vct_context* c, int level, size_t n, const float* seg, uint32_t* voxel, float* t, uint8_t* face,
                     uint8_t* rgba, uint32_t* steps);                                           // vct_view.cu
int check_overflow(vct_context* c);
int comm_barrier(vct_context* c, int channel, cudaStream_t stream);   // device-side cross-rank barrier, in stream order
int comm_check(vct_context* c);                                        // barrier time-outs -> VCT_ERR_STATE
bool comm_depth_views(vct_context* c, uint32_t** local, uint32_t** mc, uint32_t** peers, size_t* seg_words, int* world, int* rank);
void comm_release_for_destroy(vct_context* c);
int sync_all_streams(vct_context* c);      // main + voxel + visibility + copy streams idle (before freeing what frames in flight read)
// launch shape of a grid-stride kernel of the voxel chain: `mult` blocks of 256 threads per SM
#define VCT_CHAIN(mult) (unsigned)(148 * (mult)), 256u
inline cudaError_t reset_item_queue(vct_context* c) { return cudaMemsetAsync(&c->d_counters->n_items, 0, 3 * sizeof(unsigned int), c->stream); }
inline cudaError_t reset_steps(vct_context* c, StepCounter k) {
  return cudaMemsetAsync(c->d_counters->steps[k], 0, sizeof(c->d_counters->steps[k]), c->stream);
}

// ------------------------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

struct F4 { float x, y, z, w; };

// ((m0*x + m1*y) + m2*z) + m3*w -- same order as the oracle (no FMA: the TU is built with --fmad=false)
__device__ __forceinline__ F4 mul_mat_vec(const float* __restrict__ m, float x, float y, float z, float w) {
  F4 r;
  r.x = ((m[0] * x + m[4] * y) + m[8] * z) + m[12] * w;
  r.y = ((m[1] * x + m[5] * y) + m[9] * z) + m[13] * w;
  r.z = ((m[2] * x + m[6] * y) + m[10] * z) + m[14] * w;
  r.w = ((m[3] * x + m[7] * y) + m[11] * z) + m[15] * w;
  return r;
}

// Adds the warp's sum of n to partial counter slot() (0..63) of step counter k: one atomic per warp, from lane 0.  The
// kernel passes the lane it computed itself, and the slot as a callable evaluated only where the atomic is issued:
// with threadIdx read in here, or the slot computed ahead of the reduction, nvcc 12.9 schedules the kernels and
// allocates their registers differently.
template <class Slot>
__device__ __forceinline__ void count_steps(Counters* __restrict__ ctr, StepCounter k, unsigned lane, unsigned n, Slot slot) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) n += __shfl_xor_sync(0xffffffffu, n, d);
  if (lane == 0 && n) atomicAdd(&ctr->steps[k][slot() * 4], (unsigned long long)n);
}

// does this context render frame row j?  (row-band or interleaved-strip sharding of visibility and cone_trace)
__device__ __forceinline__ bool row_owned(const Params& P, int j) {
  if (P.row_il > 1) return ((j >> 3) % P.row_il) == P.row_ph;
  return j >= P.row_begin && j < ((P.row_end > 0 && P.row_end < P.H) ? P.row_end : P.H);
}

// index of the 32x8x8 level-0 brick holding voxel (x, y, z)
__host__ __device__ inline uint32_t brick_of(int x, int y, int z, int V) {
  return ((uint32_t)(z >> 3) * (uint32_t)(V >> 3) + (uint32_t)(y >> 3)) * (uint32_t)(V >> 5) + (uint32_t)(x >> 5);
}

inline size_t dirty_bytes(int V) { size_t n = (size_t)(V >> 5) * (V >> 3) * (V >> 3); return n ? n : 1; }

constexpr int SUBPIX = 256;
constexpr float SNAP_LIMIT = 8388608.0f;

__device__ __forceinline__ bool snap(float v, long long* out) {
  float s = v * (float)SUBPIX;
  if (!(s == s)) return false;
  s = fminf(fmaxf(s, -SNAP_LIMIT), SNAP_LIMIT);
  *out = (long long)__float2int_rn(s);
  return true;
}

// Exact integer triangle in 24.8 window coordinates, counter-clockwise after set-up.
struct RasterTri {
  int X0, Y0, X1, Y1, X2, Y2;   // |coords| <= 2^23
  long long area;
  int flipped;

  // edge a->b evaluated at p: dx*(py-ay) - dy*(px-ax)
  __device__ __forceinline__ static long long ev(int ax, int ay, int bx, int by, int px, int py) {
    return (long long)(bx - ax) * (long long)(py - ay) - (long long)(by - ay) * (long long)(px - ax);
  }
  __device__ __forceinline__ static int bias(int ax, int ay, int bx, int by) {
    int dx = bx - ax, dy = by - ay;
    return ((dy < 0) || (dy == 0 && dx < 0)) ? 0 : -1;
  }
  __device__ __forceinline__ long long e01(int px, int py) const { return ev(X0, Y0, X1, Y1, px, py); }
  __device__ __forceinline__ long long e12(int px, int py) const { return ev(X1, Y1, X2, Y2, px, py); }
  __device__ __forceinline__ long long e20(int px, int py) const { return ev(X2, Y2, X0, Y0, px, py); }

  __device__ __forceinline__ bool sample_inside(int sx, int sy) const {
    return e01(sx, sy) + bias(X0, Y0, X1, Y1) >= 0 && e12(sx, sy) + bias(X1, Y1, X2, Y2) >= 0 &&
           e20(sx, sy) + bias(X2, Y2, X0, Y0) >= 0;
  }
  __device__ __forceinline__ static long long emax(int ax, int ay, int bx, int by, int x0, int y0) {
    int dx = bx - ax, dy = by - ay;
    int px = (-dy > 0) ? x0 + SUBPIX : x0;
    int py = (dx > 0) ? y0 + SUBPIX : y0;
    return ev(ax, ay, bx, by, px, py);
  }
  __device__ __forceinline__ bool covered(int i, int j, int policy) const {
    int x0 = i * SUBPIX, y0 = j * SUBPIX;
    if (policy == 0) return sample_inside(x0 + 128, y0 + 128);
    if (policy == 1) {
      return sample_inside(x0 + 96, y0 + 32) || sample_inside(x0 + 224, y0 + 96) ||
             sample_inside(x0 + 32, y0 + 160) || sample_inside(x0 + 160, y0 + 224);
    }
    return emax(X0, Y0, X1, Y1, x0, y0) > 0 && emax(X1, Y1, X2, Y2, x0, y0) > 0 &&
           emax(X2, Y2, X0, Y0, x0, y0) > 0;
  }
  __device__ __forceinline__ void lambdas(int i, int j, float* l1, float* l2) const {
    int sx = i * SUBPIX + 128, sy = j * SUBPIX + 128;
    float fa = (float)area;
    *l1 = (float)e20(sx, sy) / fa;
    *l2 = (float)e01(sx, sy) / fa;
  }
};

__device__ __forceinline__ bool setup_raster(const float wx[3], const float wy[3], RasterTri* t) {
  long long X[3], Y[3];
#pragma unroll
  for (int k = 0; k < 3; ++k)
    if (!snap(wx[k], &X[k]) || !snap(wy[k], &Y[k])) return false;
  long long area = (X[1] - X[0]) * (Y[2] - Y[0]) - (Y[1] - Y[0]) * (X[2] - X[0]);
  if (area == 0) return false;
  t->flipped = area < 0;
  t->X0 = (int)X[0]; t->Y0 = (int)Y[0];
  if (t->flipped) {
    t->X1 = (int)X[2]; t->Y1 = (int)Y[2]; t->X2 = (int)X[1]; t->Y2 = (int)Y[1];
    area = -area;
  } else {
    t->X1 = (int)X[1]; t->Y1 = (int)Y[1]; t->X2 = (int)X[2]; t->Y2 = (int)Y[2];
  }
  t->area = area;
  return true;
}

__device__ __forceinline__ int floor_div256(int a) { return a >> 8; }  // arithmetic shift == floor

// pixel bounding box clipped to [0,W)x[0,H); false if empty
__device__ __forceinline__ bool raster_bbox(const RasterTri& t, int policy, int W, int H, int* i0, int* i1,
                                            int* j0, int* j1) {
  int minx = min(t.X0, min(t.X1, t.X2)), maxx = max(t.X0, max(t.X1, t.X2));
  int miny = min(t.Y0, min(t.Y1, t.Y2)), maxy = max(t.Y0, max(t.Y1, t.Y2));
  int a0, a1, b0, b1;
  if (policy == 2) {
    a0 = floor_div256(minx); a1 = floor_div256(maxx - 1);
    b0 = floor_div256(miny); b1 = floor_div256(maxy - 1);
  } else {
    a0 = floor_div256(minx - (SUBPIX - 1)); a1 = floor_div256(maxx);
    b0 = floor_div256(miny - (SUBPIX - 1)); b1 = floor_div256(maxy);
  }
  a0 = max(a0, 0); b0 = max(b0, 0); a1 = min(a1, W - 1); b1 = min(b1, H - 1);
  if (a0 > a1 || b0 > b1) return false;
  *i0 = a0; *i1 = a1; *j0 = b0; *j1 = b1;
  return true;
}

__device__ __forceinline__ float interp3(float a0, float a1, float a2, float l1, float l2) {
  return (a0 + l1 * (a1 - a0)) + l2 * (a2 - a0);
}

// ---- shadow map sampling: PCF_Shadow_Mapping (Voxelization.fs:18-52, VoxelConeTracing.fs:132-163).
// Returns the number of lit taps; the caller applies /25 (voxelisation) or *0.111 (cone trace).
// Every tap is `texture(ShadowMap, DepthCoord.xy + offset).r` = one GL_LINEAR, CLAMP_TO_EDGE fetch of the
// D24 map (no compare mode, Voxel_Cone_Tracing.h:93-96), i.e. a 2x2 footprint and three lerps in the order
// top = t00 + a*(t10-t00); bot = t01 + a*(t11-t01); d = top + b*(bot-top).
__device__ __forceinline__ float depth_texel(const uint32_t* __restrict__ depth, int S, int i, int j) {
  i = min(max(i, 0), S - 1);
  j = min(max(j, 0), S - 1);
  return (float)__ldg(&depth[(size_t)j * S + i]) * (1.0f / 16777215.0f);
}

__device__ __forceinline__ float shadow_bilinear(const uint32_t* __restrict__ depth, int S, float u, float v) {
  const float fS = (float)S;
  float x = u * fS - 0.5f, y = v * fS - 0.5f;
  float fx = floorf(x), fy = floorf(y);
  float a = x - fx, b = y - fy;
  fx = fminf(fmaxf(fx, -2.0f), fS + 1.0f);
  fy = fminf(fmaxf(fy, -2.0f), fS + 1.0f);
  int i = (int)fx, j = (int)fy;
  float t00 = depth_texel(depth, S, i, j), t10 = depth_texel(depth, S, i + 1, j);
  float t01 = depth_texel(depth, S, i, j + 1), t11 = depth_texel(depth, S, i + 1, j + 1);
  float top = t00 + a * (t10 - t00);
  float bot = t01 + a * (t11 - t01);
  return top + b * (bot - top);
}

// reference form: every tap on its own (any radius)
static __device__ __noinline__ float pcf_lit_taps_generic(const uint32_t* __restrict__ depth, int S, int r, float bias,
                                                    float dcx, float dcy, float dcz, float dcw) {
  float cur = dcz / dcw;
  float inv = 1.0f / (float)S;
  float thr = cur - bias;
  float lit = 0.0f;
  for (int x = -r; x <= r; ++x)
    for (int y = -r; y <= r; ++y) {
      float ox = inv * (float)x, oy = inv * (float)y;
      float closest = shadow_bilinear(depth, S, dcx + ox, dcy + oy);
      if (thr <= closest) lit += 1.0f;
    }
  return lit;
}

// Footprint-sharing form for the reference's radius 2 (5x5 taps): the 25 taps read a 6x6 texel block, the
// horizontal lerp of a (texel row, tap column) pair is the `bot` of one tap and the `top` of the next, so 30
// horizontal + 25 vertical lerps replace 75.  Per-column fractions a[k] and per-row fractions b[k] are
// computed exactly as the per-tap form does, and every lerp has the same operands in the same order, so the
// result is bit-identical to pcf_lit_taps_generic; if the tap columns/rows are not consecutive texels
// (float rounding of `coord + k/S`, or far outside the map) the generic form is used.
template <int R>
__device__ __forceinline__ float pcf_lit_taps_block(const uint32_t* __restrict__ depth, int S, float bias, float dcx,
                                                    float dcy, float dcz, float dcw) {
  constexpr int T = 2 * R + 1;
  const float fS = (float)S;
  const float cur = dcz / dcw;
  const float inv = 1.0f / fS;
  const float thr = cur - bias;
  float ax[T], by[T];
  int ix0 = 0, iy0 = 0;
  bool regular = true;
#pragma unroll
  for (int k = 0; k < T; ++k) {
    float ox = inv * (float)(k - R);
    float x = (dcx + ox) * fS - 0.5f, y = (dcy + ox) * fS - 0.5f;
    float fx = floorf(x), fy = floorf(y);
    ax[k] = x - fx; by[k] = y - fy;
    int i = (int)fminf(fmaxf(fx, -2.0f), fS + 1.0f), j = (int)fminf(fmaxf(fy, -2.0f), fS + 1.0f);
    if (k == 0) { ix0 = i; iy0 = j; }
    else regular = regular && (i == ix0 + k) && (j == iy0 + k);
  }
  if (!regular) return pcf_lit_taps_generic(depth, S, R, bias, dcx, dcy, dcz, dcw);
  int cx[T + 1];
#pragma unroll
  for (int c = 0; c <= T; ++c) cx[c] = min(max(ix0 + c, 0), S - 1);
  float hprev[T];
  float lit = 0.0f;
#pragma unroll
  for (int r = 0; r <= T; ++r) {
    const uint32_t* row = depth + (size_t)min(max(iy0 + r, 0), S - 1) * S;
    float t[T + 1];
#pragma unroll
    for (int c = 0; c <= T; ++c) t[c] = (float)__ldg(row + cx[c]) * (1.0f / 16777215.0f);
    float h[T];
#pragma unroll
    for (int k = 0; k < T; ++k) h[k] = t[k] + ax[k] * (t[k + 1] - t[k]);
    if (r >= 1) {
#pragma unroll
      for (int k = 0; k < T; ++k) {
        float d = hprev[k] + by[r - 1] * (h[k] - hprev[k]);
        if (thr <= d) lit += 1.0f;
      }
    }
#pragma unroll
    for (int k = 0; k < T; ++k) hprev[k] = h[k];
  }
  return lit;
}

// Same arithmetic as pcf_lit_taps_block, but the 6x6 texel block is fetched with nine tex2Dgather operations from
// a cudaArray copy of the D24 map (clamp addressing == GL_CLAMP_TO_EDGE): 2D-local cache lines instead of six row
// segments per fragment, 9 instead of 36 load instructions.  Used where the texture pipe is otherwise idle
// (voxel shading); results are bit-identical (same texels, same lerps).
__device__ __forceinline__ float pcf_lit_taps_gather(cudaTextureObject_t dtex, const uint32_t* __restrict__ depth, int S,
                                                     float bias, float dcx, float dcy, float dcz, float dcw) {
  constexpr int R = 2, T = 5;
  const float fS = (float)S;
  const float cur = dcz / dcw;
  const float inv = 1.0f / fS;
  const float thr = cur - bias;
  float ax[T], by[T];
  int ix0 = 0, iy0 = 0;
  bool regular = true;
#pragma unroll
  for (int k = 0; k < T; ++k) {
    float ox = inv * (float)(k - R);
    float x = (dcx + ox) * fS - 0.5f, y = (dcy + ox) * fS - 0.5f;
    float fx = floorf(x), fy = floorf(y);
    ax[k] = x - fx; by[k] = y - fy;
    int i = (int)fminf(fmaxf(fx, -2.0f), fS + 1.0f), j = (int)fminf(fmaxf(fy, -2.0f), fS + 1.0f);
    if (k == 0) { ix0 = i; iy0 = j; }
    else regular = regular && (i == ix0 + k) && (j == iy0 + k);
  }
  if (!regular) return pcf_lit_taps_generic(depth, S, R, bias, dcx, dcy, dcz, dcw);
  float t[6][6];
#pragma unroll
  for (int gy = 0; gy < 3; ++gy)
#pragma unroll
    for (int gx = 0; gx < 3; ++gx) {
      // footprint texels (ix0+2gx .. +1, iy0+2gy .. +1); gather order: .w=(x,y) .z=(x+1,y) .x=(x,y+1) .y=(x+1,y+1)
      const float4 g = tex2Dgather<float4>(dtex, (float)(ix0 + 2 * gx + 1), (float)(iy0 + 2 * gy + 1), 0);
      t[2 * gy][2 * gx] = g.w;              // the array already holds float(d24) * (1/16777215) (depth_to_array)
      t[2 * gy][2 * gx + 1] = g.z;
      t[2 * gy + 1][2 * gx] = g.x;
      t[2 * gy + 1][2 * gx + 1] = g.y;
    }
  float lit = 0.0f;
  float hprev[T];
#pragma unroll
  for (int r = 0; r <= T; ++r) {
    float h[T];
#pragma unroll
    for (int k = 0; k < T; ++k) h[k] = t[r][k] + ax[k] * (t[r][k + 1] - t[r][k]);
    if (r >= 1) {
#pragma unroll
      for (int k = 0; k < T; ++k) {
        float d = hprev[k] + by[r - 1] * (h[k] - hprev[k]);
        if (thr <= d) lit += 1.0f;
      }
    }
#pragma unroll
    for (int k = 0; k < T; ++k) hprev[k] = h[k];
  }
  return lit;
}

__device__ __forceinline__ float pcf_lit_taps(const uint32_t* __restrict__ depth, int S, int r, float bias,
                                              float dcx, float dcy, float dcz, float dcw) {
  if (r == 2) return pcf_lit_taps_block<2>(depth, S, bias, dcx, dcy, dcz, dcw);
  return pcf_lit_taps_generic(depth, S, r, bias, dcx, dcy, dcz, dcw);
}

// GL 4.3 8.14: lambda = log2(max(|d(uv*size)/dx|, |d(uv*size)/dy|))
__device__ __forceinline__ float lod_from_derivs(float dudx, float dvdx, float dudy, float dvdy, int w, int h) {
  float ax = dudx * (float)w, bx = dvdx * (float)h;
  float ay = dudy * (float)w, by = dvdy * (float)h;
  // log2(max(sqrt(p), sqrt(q))) = 0.5 * log2(max(p, q)); MUFU.LG2 -- the hardware quantises lambda to 1/256 anyway
  float rho2 = fmaxf(ax * ax + bx * bx, ay * ay + by * by);
  if (!(rho2 > 0.0f)) return 0.0f;
  return 0.5f * __log2f(rho2);
}

// float colour -> unorm8 (GL's conversion of a fragment output to an RGBA8 attachment)
__device__ __forceinline__ unsigned char to_unorm8(float x) {
  x = fminf(fmaxf(x, 0.0f), 1.0f);
  if (!(x == x)) x = 0.0f;
  return (unsigned char)__float2int_rn(x * 255.0f);
}

__device__ __forceinline__ float4 sample_material(cudaTextureObject_t t, float u, float v, float lod) {
  if (!(lod > 0.0f)) lod = 0.0f;
  return tex2DLod<float4>(t, u, v, lod);
}

#endif  // __CUDACC__

}  // namespace vct
