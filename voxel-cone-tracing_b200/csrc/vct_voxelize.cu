// vct_voxelize.cu -- V1..V4: triangle voxelisation with shadow-mapped light injection.
// Replaces DrawVoxelTexture's draw (Voxel_Cone_Tracing.h:213-245) and Shader/Voxelization.{vs,gs,fs}.
//
//   vox_cover  (raster_small / raster_tiles): Voxelization.vs:15-22 + .gs:22-51 + the rasteriser.  Emits
//              one 8-byte fragment record (triangle, pixel) per covered pixel of the V x V viewport.
//   vox_shade  : Voxelization.fs:54-89, one thread per fragment: depth slice, axis un-swizzle, albedo
//              fetch, 5x5 PCF, then an order-independent integer accumulation
//                 accum[v].rg += (r<<32 | g) ;  accum[v].bc += (b<<32 | 1)
//              with lanes that hit the same voxel merged first (warp-aggregated atomics).  The first
//              fragment of a voxel (old count == 0) appends the voxel to the touched list.
//   vox_clear / vox_resolve : sparse, over the touched list only.
#include <cooperative_groups.h>
#include <cuda_fp16.h>
#include <cooperative_groups/reduce.h>

#include "vct_raster.cuh"

namespace cg = cooperative_groups;

namespace vct {

// ---------------------------------------------------------------------------------------------------
// Per-triangle set-up.  raster_small evaluates it once per triangle (Voxelization.vs + .gs) and stores a 128-byte
// record -- snapped window coordinates, depth, axis, material, texture LOD, uv and light-space coordinates in
// rasterisation order -- which the tile stage and the per-fragment shading stage reload instead of redoing the
// geometry-shader work per tile / per fragment.
struct VoxTri {
  RasterTri t;
  float z0, z1, z2;
  int axis;
};

template <bool WITH_ATTRS>
__device__ __forceinline__ bool vox_setup(const Params& P, const VertexCache& vc,
                                          const uint32_t* __restrict__ idx, uint32_t tri, VoxTri& s,
                                          float (*uv)[2], F4* dc) {
  const int V = P.V;
  F4 world[3];
  float tuv[3][2];
  F4 tdc[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const uint32_t vi = __ldg(&idx[tri * 3 + k]);
    const float4 w = __ldg(&vc.world[vi]);                                // Voxelization.vs:21 (vertex_pass)
    world[k].x = w.x; world[k].y = w.y; world[k].z = w.z; world[k].w = w.w;
    if (WITH_ATTRS) {
      const float4 d = __ldg(&vc.dc[vi]);                                  // Voxelization.vs:18-19
      tdc[k].x = d.x; tdc[k].y = d.y; tdc[k].z = d.z; tdc[k].w = d.w;
      tuv[k][0] = __ldg(&vc.nrm_u[vi].w); tuv[k][1] = __ldg(&vc.tan_v[vi].w);
    }
  }
  // Voxelization.gs:25-39 (decision on the un-normalised |cross|; zero / NaN -> axis 3)
  float e1x = world[0].x - world[1].x, e1y = world[0].y - world[1].y, e1z = world[0].z - world[1].z;
  float e2x = world[2].x - world[0].x, e2y = world[2].y - world[0].y, e2z = world[2].z - world[0].z;
  float nx = fabsf(e1y * e2z - e1z * e2y), ny = fabsf(e1z * e2x - e1x * e2z), nz = fabsf(e1x * e2y - e1y * e2x);
  int axis;
  if (!(nx == nx) || !(ny == ny) || !(nz == nz)) axis = 3;
  else if (nx == 0.0f && ny == 0.0f && nz == 0.0f) axis = 3;
  else if (nx >= ny && nx >= nz) axis = 1;
  else if (ny >= nx && ny >= nz) axis = 2;
  else axis = 3;
  const float* Pm = axis == 1 ? P.projx : axis == 2 ? P.projy : P.projz;    // Voxelization.gs:41
  float wx[3], wy[3], wz[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    F4 c = mul_mat_vec(Pm, world[k].x, world[k].y, world[k].z, world[k].w);
    if (!(c.w > 0.0f)) return false;
    float ndx = c.x / c.w, ndy = c.y / c.w, ndz = c.z / c.w;
    wx[k] = (ndx * 0.5f + 0.5f) * (float)V;       // glViewport(0,0,V,V), Voxel_Cone_Tracing.h:218
    wy[k] = (ndy * 0.5f + 0.5f) * (float)V;
    wz[k] = ndz * 0.5f + 0.5f;
  }
  if (!setup_raster(wx, wy, &s.t)) return false;
  const int a = s.t.flipped ? 2 : 1, b = s.t.flipped ? 1 : 2;
  s.z0 = wz[0]; s.z1 = wz[a]; s.z2 = wz[b];
  s.axis = axis;
  if (WITH_ATTRS) {
    uv[0][0] = tuv[0][0]; uv[0][1] = tuv[0][1];
    uv[1][0] = tuv[a][0]; uv[1][1] = tuv[a][1];
    uv[2][0] = tuv[b][0]; uv[2][1] = tuv[b][1];
    dc[0] = tdc[0]; dc[1] = tdc[a]; dc[2] = tdc[b];
  }
  return true;
}

// 8 x 16 B per triangle
struct VoxRecord {
  int4 a;      // X0 Y0 X1 Y1
  int4 b;      // X2 Y2 axis material
  float4 z;    // z0 z1 z2 lod
  float4 uv01; // uv0.xy uv1.xy
  float4 uv2;  // uv2.xy - -
  float4 dc0, dc1, dc2;
};

__device__ __forceinline__ void load_raster_tri(const VoxRecord* __restrict__ rec, uint32_t tri, VoxTri& s) {
  const int4 a = __ldg(&rec[tri].a), b = __ldg(&rec[tri].b);
  s.t.X0 = a.x; s.t.Y0 = a.y; s.t.X1 = a.z; s.t.Y1 = a.w; s.t.X2 = b.x; s.t.Y2 = b.y;
  s.t.area = (long long)(s.t.X1 - s.t.X0) * (long long)(s.t.Y2 - s.t.Y0) - (long long)(s.t.Y1 - s.t.Y0) * (long long)(s.t.X2 - s.t.X0);
  s.t.flipped = 0;
  s.axis = b.z;
}

// ---------------------------------------------------------------------------------------------------
struct VoxCoverPass {
  Params P;
  VertexCache vc; const uint32_t* idx;
  const uint16_t* trimat; const MaterialDev* mats;
  VoxRecord* rec;
  uint2* frags; uint32_t frags_cap;
  Counters* ctr;

  struct Setup { VoxTri v; };

  // raster_small: full set-up from the vertex cache + the per-triangle record
  __device__ __forceinline__ bool setup_full(uint32_t tri, Setup& s, int& i0, int& i1, int& j0, int& j1) const {
    float uv[3][2];
    F4 dc[3];
    if (!vox_setup<true>(P, vc, idx, tri, s.v, uv, dc)) return false;
    if (!raster_bbox(s.v.t, P.coverage, P.V, P.V, &i0, &i1, &j0, &j1)) return false;
    const int mat = trimat ? trimat[tri] : 0;
    // implicit LOD of texture(DiffuseTexture, TexCoord) (Voxelization.fs:56): uv is affine over the triangle
    const RasterTri& t = s.v.t;
    const float fa = (float)t.area;
    const float dl1dx = (float)(-(long long)(t.Y0 - t.Y2) * SUBPIX) / fa, dl1dy = (float)((long long)(t.X0 - t.X2) * SUBPIX) / fa;
    const float dl2dx = (float)(-(long long)(t.Y1 - t.Y0) * SUBPIX) / fa, dl2dy = (float)((long long)(t.X1 - t.X0) * SUBPIX) / fa;
    const float du1 = uv[1][0] - uv[0][0], du2 = uv[2][0] - uv[0][0];
    const float dv1 = uv[1][1] - uv[0][1], dv2 = uv[2][1] - uv[0][1];
    const float lod = lod_from_derivs(dl1dx * du1 + dl2dx * du2, dl1dx * dv1 + dl2dx * dv2,
                                      dl1dy * du1 + dl2dy * du2, dl1dy * dv1 + dl2dy * dv2, mats[mat].dw, mats[mat].dh);
    VoxRecord r;
    r.a = make_int4(t.X0, t.Y0, t.X1, t.Y1);
    r.b = make_int4(t.X2, t.Y2, s.v.axis, mat);
    r.z = make_float4(s.v.z0, s.v.z1, s.v.z2, lod);
    r.uv01 = make_float4(uv[0][0], uv[0][1], uv[1][0], uv[1][1]);
    r.uv2 = make_float4(uv[2][0], uv[2][1], 0.0f, 0.0f);
    r.dc0 = make_float4(dc[0].x, dc[0].y, dc[0].z, dc[0].w);
    r.dc1 = make_float4(dc[1].x, dc[1].y, dc[1].z, dc[1].w);
    r.dc2 = make_float4(dc[2].x, dc[2].y, dc[2].z, dc[2].w);
    rec[tri] = r;
    return true;
  }
  // raster_tiles: reload the snapped triangle
  __device__ __forceinline__ bool setup(uint32_t tri, Setup& s, int& i0, int& i1, int& j0, int& j1) const {
    load_raster_tri(rec, tri, s.v);
    return raster_bbox(s.v.t, P.coverage, P.V, P.V, &i0, &i1, &j0, &j1);
  }
  __device__ __forceinline__ bool tile_may_cover(const Setup& s, int x0, int y0, int x1, int y1) const {
    return tile_may_cover_exact(s.v.t, x0, y0, x1, y1);
  }
  __device__ __forceinline__ void tile_rows(int&, int&, int&) const {}      // every tile row of the box

  // thread-serial path: <= 16 pixels -> 16-bit coverage mask, one warp-wide reservation
  __device__ __forceinline__ void small(const Setup& s, uint32_t tri, bool active, int i0, int i1, int j0, int j1) const {
    unsigned mask = 0;
    const int w = i1 - i0 + 1;
    if (active) {
      int bit = 0;
      for (int j = j0; j <= j1; ++j)
        for (int i = i0; i <= i1; ++i, ++bit)
          if (s.v.t.covered(i, j, P.coverage)) mask |= 1u << bit;
    }
    unsigned n = __popc(mask);
    // inclusive warp scan of n
    unsigned lane = threadIdx.x & 31, incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      unsigned t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= (unsigned)d) incl += t;
    }
    unsigned total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned base = 0;
    if (lane == 31 && total) base = atomicAdd(&ctr->n_fragments, total);
    base = __shfl_sync(0xffffffffu, base, 31);
    if (!n) return;
    unsigned pos = base + incl - n;
    while (mask) {
      int bit = __ffs(mask) - 1;
      mask &= mask - 1;
      int i = i0 + bit % w, j = j0 + bit / w;
      if (pos < frags_cap) frags[pos] = make_uint2(tri, (unsigned)i | ((unsigned)j << 16));
      else ctr->overflow = 1;
      ++pos;
    }
  }

  // warp path (raster_tiles, kAppends protocol)
  static constexpr bool kAppends = true;
  static constexpr bool kWarpMedium = false;    // fragments are appended with warp-wide reservations: thread / tile paths only
  __device__ __forceinline__ bool covered(const Setup& s, int i, int j) const { return s.v.t.covered(i, j, P.coverage); }
  __device__ __forceinline__ uint32_t reserve(uint32_t n) const { return atomicAdd(&ctr->n_fragments, n); }
  __device__ __forceinline__ void emit(uint32_t tri, int i, int j, uint32_t pos) const {
    if (pos < frags_cap) frags[pos] = make_uint2(tri, (unsigned)i | ((unsigned)j << 16));
    else ctr->overflow = 1;
  }
  __device__ __forceinline__ void pixel(const Setup&, uint32_t, int, int, bool) const {}
};

// vox_shade: the first fragment of a voxel sets the voxel's bit; vox_compact_mask then emits the touched list in MEMORY
// ORDER (runs of x-adjacent voxels), so that the list-driven kernels behind it -- clear, resolve, push, merge -- touch
// the accumulator and level 0 in coalesced runs instead of at random (they are bound by scattered 32-byte DRAM
// transactions otherwise: a list in first-touch order cost 30-40 ps per voxel whatever the grid size).
__device__ __forceinline__ void mark_first_touch(bool& pending, unsigned long long old, uint32_t voxel,
                                                 uint32_t* __restrict__ occ_mask) {
  if (pending && (uint32_t)old == 0u) atomicOr(&occ_mask[voxel >> 5], 1u << (voxel & 31u));
  pending = false;
}

// The merge appends the voxels that are new to this rank directly to the list (one counter atomic per warp-step): its
// records arrive in the SENDER's memory order, so the appended tail is memory-ordered in chunks anyway, and going through
// the bit mask instead costs a second compaction pass (measured: merge 86 -> 104 us at eight ranks).
__device__ __forceinline__ void append_first_touch(unsigned long long old, uint32_t voxel, uint32_t* __restrict__ touched,
                                                   unsigned int* __restrict__ n_touched) {
  if ((uint32_t)old == 0u) {
    cg::coalesced_group firsts = cg::coalesced_threads();
    uint32_t base = 0;
    if (firsts.thread_rank() == 0) base = atomicAdd(n_touched, (uint32_t)firsts.size());
    base = firsts.shfl(base, 0);
    touched[base + firsts.thread_rank()] = voxel;
  }
}

// One thread per 32-voxel mask word; a warp covers 1024 consecutive voxels and reserves its output range with one
// atomic, so the list is a sequence of memory-ordered chunks.  The words are cleared on the way.
__global__ void __launch_bounds__(256) vox_compact_mask(uint32_t* __restrict__ occ_mask, uint32_t n_words,
                                                        uint32_t* __restrict__ list, unsigned int* __restrict__ n_list) {
  const unsigned lane = threadIdx.x & 31;
  const uint32_t n_round = (n_words + 31u) & ~31u;
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < n_round; w += gridDim.x * blockDim.x) {
    uint32_t bits = w < n_words ? occ_mask[w] : 0u;
    if (!__any_sync(0xffffffffu, bits != 0u)) continue;
    if (bits) occ_mask[w] = 0u;
    const unsigned cnt = __popc(bits);
    unsigned incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= (unsigned)d) incl += t;
    }
    unsigned base = 0;
    if (lane == 31) base = atomicAdd(n_list, incl);
    base = __shfl_sync(0xffffffffu, base, 31) + incl - cnt;
    while (bits) {
      const int b = __ffs(bits) - 1;
      bits &= bits - 1;
      list[base++] = (w << 5) + (uint32_t)b;
    }
  }
}

// multimem.red: one reduction instruction applied to the same offset of every rank's copy, performed in the NVSwitch
// The symmetric accumulator holds (r, g, b, count) as four fp32 per voxel: every value is an integer below 2^24
// (<= 65 793 fragments of 255 per voxel), so fp32 addition is exact and order independent, and one 16-byte vector
// reduction carries a whole voxel.
__device__ __forceinline__ void multimem_add_v4f32(float4* mc_addr, float4 v) {
  asm volatile("multimem.red.relaxed.sys.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void multimem_or_b32(uint32_t* mc_addr, uint32_t v) {
  asm volatile("multimem.red.relaxed.sys.global.or.b32 [%0], %1;" ::"l"(mc_addr), "r"(v) : "memory");
}
// multicast store: one 16-byte store lands at the same offset on every rank
__device__ __forceinline__ void multimem_st_v4(void* mc_addr, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc_addr), "f"(__uint_as_float(v.x)),
               "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w)) : "memory");
}
__device__ __forceinline__ void multimem_st_u32(uint32_t* mc_addr, uint32_t v) {
  asm volatile("multimem.st.relaxed.sys.global.u32 [%0], %1;" ::"l"(mc_addr), "r"(v) : "memory");
}

// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) vox_shade(Params P, const VoxRecord* __restrict__ rec,
                                                 const MaterialDev* __restrict__ mats,
                                                 const uint32_t* __restrict__ depth, cudaTextureObject_t depth_tex,
                                                 const uint2* __restrict__ frags, uint32_t frags_cap,
                                                 unsigned long long* __restrict__ accum,
                                                 uint32_t* __restrict__ occ_mask, Counters* __restrict__ ctr) {
  const uint32_t nfrag = min(ctr->n_fragments, frags_cap);
  const int V = P.V;
  bool pending = false;
  unsigned long long pend_old = 0ull;
  uint32_t pend_voxel = 0u;
  // software pipeline: the next fragment's queue entry is loaded one iteration ahead and its triangle record
  // (one 128-byte line) is prefetched, so the dependent chain queue -> record -> shadow texels starts warm
  const uint32_t stride = gridDim.x * blockDim.x;
  uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
  uint2 fr_next = f < nfrag ? frags[f] : make_uint2(0u, 0u);
  for (; f < nfrag; f += stride) {
    const uint2 fr = fr_next;
    if (f + stride < nfrag) {
      fr_next = frags[f + stride];
      asm volatile("prefetch.global.L1 [%0];" ::"l"(&rec[fr_next.x]));
    }
    mark_first_touch(pending, pend_old, pend_voxel, occ_mask);
    const uint32_t tri = fr.x;
    const int i = (int)(fr.y & 0xFFFFu), j = (int)(fr.y >> 16);
    VoxTri s;
    load_raster_tri(rec, tri, s);
    const float4 zl = __ldg(&rec[tri].z);
    float l1, l2;
    s.t.lambdas(i, j, &l1, &l2);
    float z = interp3(zl.x, zl.y, zl.z, l1, l2);
    if (P.coverage == 2) {
      float zmin = fminf(zl.x, fminf(zl.y, zl.z)), zmax = fmaxf(zl.x, fmaxf(zl.y, zl.z));
      z = fminf(fmaxf(z, zmin), zmax);
    }
    float tz = (float)V * z;                                  // Voxelization.fs:58
    if (!(tz >= 0.0f) || !(tz < (float)V)) continue;          // clipped / imageStore out of bounds
    const int cz = (int)tz;
    int vx, vy, vz;
    if (s.axis == 1) { vx = V - 1 - cz; vz = V - 1 - i; vy = j; }        // Voxelization.fs:70-75
    else if (s.axis == 2) { vz = V - 1 - j; vy = V - 1 - cz; vx = i; }   // :76-81
    else { vx = i; vy = j; vz = V - 1 - cz; }                            // :82-86
    if ((unsigned)vx >= (unsigned)V || (unsigned)vy >= (unsigned)V || (unsigned)vz >= (unsigned)V) continue;

    // texture(DiffuseTexture, TexCoord), Voxelization.fs:56
    const MaterialDev& m = mats[__ldg(&rec[tri].b.w)];
    const float4 uv01 = __ldg(&rec[tri].uv01), uv2 = __ldg(&rec[tri].uv2);
    const float u = interp3(uv01.x, uv01.z, uv2.x, l1, l2);
    const float vv = interp3(uv01.y, uv01.w, uv2.y, l1, l2);
    const float4 col = sample_material(m.diffuse, u, vv, zl.w);

    const float4 d0 = __ldg(&rec[tri].dc0), d1 = __ldg(&rec[tri].dc1), d2 = __ldg(&rec[tri].dc2);
    const float dx = interp3(d0.x, d1.x, d2.x, l1, l2);
    const float dy = interp3(d0.y, d1.y, d2.y, l1, l2);
    const float dz = interp3(d0.z, d1.z, d2.z, l1, l2);
    const float dw = interp3(d0.w, d1.w, d2.w, l1, l2);
    const int taps = (2 * P.pcf_radius + 1) * (2 * P.pcf_radius + 1);
    const float lit = P.pcf_radius == 2 ? pcf_lit_taps_gather(depth_tex, depth, P.S, P.shadow_bias, dx, dy, dz, dw)
                                        : pcf_lit_taps_generic(depth, P.S, P.pcf_radius, P.shadow_bias, dx, dy, dz, dw);
    const float shadow = lit / (float)taps;

    // imageStore(VoxelTexture, voxelPos, vec4(color.rgb * shadow, 1)): unorm8 conversion, Voxelization.fs:88
    unsigned r = (unsigned)__float2int_rn(fminf(fmaxf(col.x * shadow, 0.0f), 1.0f) * 255.0f);
    unsigned g = (unsigned)__float2int_rn(fminf(fmaxf(col.y * shadow, 0.0f), 1.0f) * 255.0f);
    unsigned b = (unsigned)__float2int_rn(fminf(fmaxf(col.z * shadow, 0.0f), 1.0f) * 255.0f);
    const uint32_t voxel = (uint32_t)(((size_t)vz * V + vy) * V + vx);

    // warp-aggregated atomics: lanes of this warp that hit the same voxel are summed first
    cg::coalesced_group active = cg::coalesced_threads();
    cg::coalesced_group same = cg::labeled_partition(active, voxel);
    unsigned long long rg = ((unsigned long long)r << 32) | g;
    unsigned long long bc = ((unsigned long long)b << 32) | 1ull;
    if (same.size() > 1) {
      rg = cg::reduce(same, rg, cg::plus<unsigned long long>());
      bc = cg::reduce(same, bc, cg::plus<unsigned long long>());
    }
    if (same.thread_rank() == 0) {
      atomicAdd(&accum[2 * (size_t)voxel], rg);
      // The returned old count is consumed one iteration later (mark_first_touch at the loop top), so the
      // warp does not sit on the L2 round trip of this atomic.
      pend_old = atomicAdd(&accum[2 * (size_t)voxel + 1], bc);
      pend_voxel = voxel;
      pending = true;
    }
  }
  mark_first_touch(pending, pend_old, pend_voxel, occ_mask);
}

// ---------------------------------------------------------------------------------------------------
// Sparse clear before a voxelisation into slot B: (1) zero the accumulator cells named by the list of the previous
// voxelisation (slot A), (2) zero the level-0 texels of slot B named by slot B's own old list (what the frame before
// last left there).  Cost is proportional to the occupied voxels, not to V^3.
// Thousands of voxels share a brick and neighbours in the touched list are neighbours in space: a lane stores only
// if its brick differs from the previous lane's (plain byte stores from every thread to the same few L2 sectors cost
// ~10 us per pass).  The leader and every lane's predecessor are derived from the active mask itself (independent
// thread scheduling does not promise that the callers' lanes are a converged prefix of the warp): the lowest active
// lane always stores, any other lane compares with the nearest active lane below it.
__device__ __forceinline__ void mark_dirty(unsigned char* dirty, uint32_t brick) {
  const unsigned active = __activemask();
  const unsigned lane = threadIdx.x & 31;
  const unsigned below = active & ((1u << lane) - 1u);
  const int prev = below ? 31 - __clz(below) : (int)lane;         // self for the leader: shuffle source stays in the mask
  const uint32_t up = __shfl_sync(active, brick, prev);
  if (!below || up != brick) dirty[brick] = 1;
}

__global__ void vox_clear_sparse(unsigned long long* __restrict__ accum, const uint32_t* __restrict__ listA,
                                 const unsigned int* __restrict__ nA, cudaSurfaceObject_t level0B,
                                 const uint32_t* __restrict__ listB, const unsigned int* __restrict__ nB, int V, int f16) {
  const uint32_t stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (listA) {
    const uint32_t n = *nA;
    for (uint32_t k = t0; k < n; k += stride) {
      uint32_t v = listA[k];
      *reinterpret_cast<ulonglong2*>(&accum[2 * (size_t)v]) = make_ulonglong2(0ull, 0ull);     // one 16-byte store per cell
    }
  }
  if (listB) {
    const uint32_t n = *nB;
    for (uint32_t k = t0; k < n; k += stride) {
      uint32_t v = listB[k];
      int x = v % V, y = (v / V) % V, z = v / (V * V);
      if (f16) surf3Dwrite(make_uint2(0u, 0u), level0B, x * 8, y, z);
      else surf3Dwrite(make_uchar4(0, 0, 0, 0), level0B, x * 4, y, z);
    }
  }
}

__global__ void zero_level0(cudaSurfaceObject_t level0, int V, int f16) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
  if (x >= V || y >= V) return;
  if (f16) surf3Dwrite(make_uint2(0u, 0u), level0, x * 8, y, z);
  else surf3Dwrite(make_uchar4(0, 0, 0, 0), level0, x * 4, y, z);
}

__device__ __forceinline__ uchar4 resolve_cell(unsigned long long rg, unsigned long long bc) {
  unsigned cnt = (unsigned)bc;
  if (!cnt) return make_uchar4(0, 0, 0, 0);
  unsigned r = (unsigned)(rg >> 32), g = (unsigned)rg, b = (unsigned)(bc >> 32);
  unsigned h = cnt >> 1;
  return make_uchar4((unsigned char)((r + h) / cnt), (unsigned char)((g + h) / cnt),
                     (unsigned char)((b + h) / cnt), 255);   // alpha written as 1.0, Voxelization.fs:88
}

// RGBA16F level 0: rgb = half(sum / (count * 255)), alpha = 1 (DESIGN.md "Defined semantics")
__device__ __forceinline__ uint2 resolve_cell16(unsigned long long rg, unsigned long long bc) {
  unsigned cnt = (unsigned)bc;
  if (!cnt) return make_uint2(0u, 0u);
  const float d = (float)cnt * 255.0f;
  const __half r = __float2half_rn((float)(unsigned)(rg >> 32) / d), g = __float2half_rn((float)(unsigned)rg / d),
               b = __float2half_rn((float)(unsigned)(bc >> 32) / d), a = __float2half_rn(1.0f);
  return make_uint2((unsigned)__half_as_ushort(r) | ((unsigned)__half_as_ushort(g) << 16),
                    (unsigned)__half_as_ushort(b) | ((unsigned)__half_as_ushort(a) << 16));
}

// Gather kernels over the touched list (resolve, push, merge) are bound by the latency of one scattered 16-byte access
// per voxel: every thread keeps ILP of them in flight (list entries first, then the cells, then the work).
constexpr int ILP = 4;

__global__ void vox_resolve_sparse(const unsigned long long* __restrict__ accum,
                                   const uint32_t* __restrict__ touched, const unsigned int* __restrict__ n_touched,
                                   cudaSurfaceObject_t level0, int V, int f16, unsigned char* __restrict__ dirty) {
  const uint32_t n = *n_touched;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t k0 = blockIdx.x * blockDim.x + threadIdx.x; k0 < n; k0 += ILP * stride) {
    uint32_t v[ILP];
    ulonglong2 a[ILP];
#pragma unroll
    for (int m = 0; m < ILP; ++m) v[m] = (k0 + m * stride < n) ? touched[k0 + m * stride] : 0xFFFFFFFFu;
#pragma unroll
    for (int m = 0; m < ILP; ++m)
      if (v[m] != 0xFFFFFFFFu) a[m] = *reinterpret_cast<const ulonglong2*>(&accum[2 * (size_t)v[m]]);
#pragma unroll
    for (int m = 0; m < ILP; ++m) {
      if (v[m] == 0xFFFFFFFFu) continue;
      int x = v[m] % V, y = (v[m] / V) % V, z = v[m] / (V * V);
      if (f16) surf3Dwrite(resolve_cell16(a[m].x, a[m].y), level0, x * 8, y, z);
      else surf3Dwrite(resolve_cell(a[m].x, a[m].y), level0, x * 4, y, z);
      mark_dirty(dirty, brick_of(x, y, z, V));
    }
  }
}

__global__ void vox_resolve_dense(const unsigned long long* __restrict__ accum, cudaSurfaceObject_t level0, int V, int f16) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
  if (x >= V || y >= V) return;
  size_t v = ((size_t)z * V + y) * V + x;
  const ulonglong2 a = *reinterpret_cast<const ulonglong2*>(&accum[2 * v]);
  if (f16) surf3Dwrite(resolve_cell16(a.x, a.y), level0, x * 8, y, z);
  else surf3Dwrite(resolve_cell(a.x, a.y), level0, x * 4, y, z);
}

__global__ void accum_to_counts(const unsigned long long* __restrict__ accum, size_t n, uint32_t* counts, uint32_t* sums) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long rg = accum[2 * i], bc = accum[2 * i + 1];
  if (counts) counts[i] = (uint32_t)bc;
  if (sums) { sums[3 * i] = (uint32_t)(rg >> 32); sums[3 * i + 1] = (uint32_t)rg; sums[3 * i + 2] = (uint32_t)(bc >> 32); }
}

// ---------------------------------------------------------------------------------------------------
// Prepares the CURRENT slot (c->cur, already switched by begin_voxel_slot) and the accumulator for a new
// voxelisation.
int launch_voxel_clear(vct_context* c) {
  int rc = ensure_grid(c); if (rc) return rc;
  PassTimer timer(c, VCT_PASS_VOX_CLEAR);
  const int V = c->P.V;
  vct_context::GridBuf& g = c->grid[c->cur];
  // accumulator: all zero already (vox_push_shared left it so), or described by a slot's touched list (sparse clear), or
  // unknown (dense memset)
  const bool accum_clean = c->accum_list_slot == -2 && !c->dense_resolve;
  const bool accum_sparse = c->accum_list_slot >= 0 && !c->dense_resolve;
  if (!accum_sparse && !accum_clean) VCT_CUDA(c, cudaMemsetAsync(c->d_accum, 0, (size_t)V * V * V * 16, c->stream));
  if (g.list_valid && g.occ_valid && g.mips_current) {
    // a new tracking period for the sparse mip build: the bricks of the content about to be zeroed become "prev"
    std::swap(g.dirty_now, g.dirty_prev);
    VCT_CUDA(c, cudaMemsetAsync(g.dirty_now, 0, dirty_bytes(V), c->stream));
    g.dirty_valid = true;
  } else if (g.list_valid && g.occ_valid && g.dirty_valid) {
    // level 0 changes again before its pyramid was built: keep accumulating into the same flags
  } else {
    VCT_CUDA(c, cudaMemsetAsync(g.dirty_now, 0, dirty_bytes(V), c->stream));
    g.dirty_valid = false;                   // which bricks differ from the pyramid is unknown: next build is dense
  }
  g.mips_current = false;
  if (!g.list_valid) {              // level 0 of this slot was written densely: zero all of it
    dim3 b(32, 8), gr((V + 31) / 32, (V + 7) / 8, V);
    zero_level0<<<gr, b, 0, c->stream>>>(g.surf[0], V, c->grid_format);
    c->launches += 1;
  }
  if (accum_sparse || g.list_valid) {
    const vct_context::GridBuf* a = accum_sparse ? &c->grid[c->accum_list_slot] : nullptr;
    vox_clear_sparse<<<VCT_CHAIN(8), 0, c->stream>>>(c->d_accum, a ? a->touched : nullptr, a ? a->n_touched : nullptr,
                                                  g.surf[0], g.list_valid ? g.touched : nullptr, g.n_touched, V, c->grid_format);
    c->launches += 1;
  }
  VCT_CUDA(c, cudaMemsetAsync(g.n_touched, 0, sizeof(unsigned int), c->stream));
  VCT_CUDA(c, cudaMemsetAsync(&c->d_counters->n_fragments, 0, sizeof(unsigned int), c->stream));
  g.list_valid = true;              // from here on the list (being rebuilt) describes this slot's level 0
  c->mask_valid[c->cur] = false;
  c->accum_list_slot = c->cur;
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

static int voxelize_impl(vct_context* c, size_t tb, size_t te, int shared) {
  if (!c->nt) return set_error(c, VCT_ERR_STATE, "voxelize: no mesh uploaded");
  if (!c->depth_valid) return set_error(c, VCT_ERR_STATE, "voxelize: call vct_draw_depth first (shadow map missing)");
  int rc = ensure_grid(c); if (rc) return rc;
  rc = ensure_queues(c); if (rc) return rc;
  rc = sync_materials(c); if (rc) return rc;
  rc = ensure_vertex_cache(c); if (rc) return rc;
  if (c->voxrec_nt != c->nt) {
    cudaFree(c->d_voxrec); c->d_voxrec = nullptr;
    VCT_CUDA(c, cudaMalloc(&c->d_voxrec, c->nt * sizeof(VoxRecord)));
    c->voxrec_nt = c->nt;
  }
  te = te < c->nt ? te : c->nt;
  if (tb >= te) return VCT_OK;
  {
    PassTimer timer(c, VCT_PASS_VOX_COVER);
    VCT_CUDA(c, reset_item_queue(c));
    VCT_CUDA(c, cudaMemsetAsync(&c->d_counters->n_fragments, 0, sizeof(unsigned int), c->stream));
    VoxCoverPass pass{c->P, c->vcache2[c->cur], c->d_idx, c->d_trimat, c->d_materials, (VoxRecord*)c->d_voxrec, c->d_frags, (uint32_t)c->frags_cap, c->d_counters};
    const uint32_t n = (uint32_t)(te - tb);
    const uint32_t n_blocks = (n + 127) / 128, il = (uint32_t)c->tri_interleave, ph = (uint32_t)c->tri_phase % il;
    const uint32_t own_blocks = n_blocks > ph ? (n_blocks - ph + il - 1) / il : 0;
    if (own_blocks)
      raster_small<VoxCoverPass><<<own_blocks, 128, 0, c->stream>>>(pass, (uint32_t)tb, (uint32_t)te, c->d_items,
                                                                     (uint32_t)c->items_cap, c->d_counters, il, ph);
    raster_tiles<VoxCoverPass><<<VCT_CHAIN(4), 0, c->stream>>>(pass, c->d_items, (uint32_t)c->items_cap, c->d_counters);
    c->launches += 2;
  }
  {
    PassTimer timer(c, VCT_PASS_VOX_SHADE);
    uint32_t* list = shared ? c->d_push_list : c->grid[c->cur].touched;
    unsigned int* n_list = shared ? c->d_push_count : c->grid[c->cur].n_touched;
    vox_shade<<<VCT_CHAIN(8), 0, c->stream>>>(c->P, (const VoxRecord*)c->d_voxrec, c->d_materials, c->d_depth,
                                           c->depth_tex, c->d_frags, (uint32_t)c->frags_cap, c->d_accum, c->d_occ_mask,
                                           c->d_counters);
    const uint32_t n_words = (uint32_t)(((size_t)c->P.V * c->P.V * c->P.V + 31) / 32);
    vox_compact_mask<<<VCT_CHAIN(4), 0, c->stream>>>(c->d_occ_mask, n_words, list, n_list);
    c->launches += 2;
  }
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

int launch_voxelize(vct_context* c, size_t tb, size_t te) { return voxelize_impl(c, tb, te, 0); }

// The exchange step of triangle-sharded voxelisation, fused over NVSwitch: every voxel this rank touched is added
// into the same cell of EVERY rank's symmetric accumulator (and its bit set in every rank's occupancy mask) by
// multimem.red on the multicast mapping -- three switch-side reductions per touched voxel, no all-reduce, no staging
// copy.  The private cells are zeroed on the way, so the private accumulator is clean for the next frame.
template <bool MULTICAST>
__global__ void vox_push_shared(unsigned long long* __restrict__ accum, const uint32_t* __restrict__ list,
                                const unsigned int* __restrict__ n_list, float4* shared, int V) {
  const uint32_t n = *n_list;
  uint32_t* mask = reinterpret_cast<uint32_t*>(shared + (size_t)V * V * V);
  const uint32_t n_round = (n + 31u) & ~31u;      // whole warps stay in the loop for the match below
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n_round; k += gridDim.x * blockDim.x) {
    const bool live = k < n;
    const uint32_t v = live ? list[k] : 0xFFFFFFFFu;
    if (live) {
      ulonglong2* cell = reinterpret_cast<ulonglong2*>(&accum[2 * (size_t)v]);
      const ulonglong2 a = *cell;
      *cell = make_ulonglong2(0ull, 0ull);
      const float4 f = make_float4((float)(unsigned)(a.x >> 32), (float)(unsigned)a.x, (float)(unsigned)(a.y >> 32),
                                   (float)(unsigned)a.y);
      if (MULTICAST) multimem_add_v4f32(&shared[v], f);
      else {
        atomicAdd(&shared[v].x, f.x); atomicAdd(&shared[v].y, f.y); atomicAdd(&shared[v].z, f.z); atomicAdd(&shared[v].w, f.w);
      }
    }
    // occupancy bits: lanes whose voxels share a 32-voxel mask word issue one OR
    const uint32_t word = live ? (v >> 5) : 0xFFFFFFFFu;
    const unsigned peers = __match_any_sync(0xffffffffu, word);
    uint32_t bits = live ? (1u << (v & 31)) : 0u;
    // OR-reduce the bits over the peer group (at most 32 lanes; groups are small in practice)
    uint32_t acc = 0;
    for (unsigned m = peers; m; m &= m - 1) acc |= __shfl_sync(peers, bits, __ffs(m) - 1);
    if (live && (int)(threadIdx.x & 31) == __ffs(peers) - 1) {
      if (MULTICAST) multimem_or_b32(&mask[word], acc);
      else atomicOr(&mask[word], acc);
    }
  }
}

// ---- inbox exchange -------------------------------------------------------------------------------------------
// Symmetric buffer: [4096 B header: count[parity][rank]] [records: (parity, rank, k) -> 16 B].  Every rank multicasts
// the voxels it touched (index + integer sums + count) into ITS row of every rank's inbox; after the barrier each
// rank adds the other rows into its private accumulator, which then equals a single-GPU voxelisation exactly, and
// the ordinary sparse resolve / mip / clear machinery applies unchanged.
// Record = uint4 {r | c0<<24, g | c1<<24, b | c2<<24, voxel}: 24-bit channel sums and a 24-bit count (bytes c0..c2).
// A sum of 2^24 or more (> 65 793 fragments in one voxel from one rank) does not fit and is reported as an overflow.
constexpr size_t EXCH_HEADER = 4096, EXCH_RECORD = 16;
__host__ __device__ inline size_t exch_record_offset(int parity, int world, int rank, size_t cap, size_t k) {
  return EXCH_HEADER + ((((size_t)parity * world + rank) * cap) + k) * EXCH_RECORD;
}

// MODE 0: plain store into one buffer (single GPU, or several handles sharing one buffer); 1: multimem.st through the
// multicast mapping (one store lands in every rank's inbox, replicated by the NVSwitch); 2: no multicast object --
// one peer store per rank into the mapped segments (dst + r * seg is rank r's inbox).
template <int MODE>
__global__ void vox_push_inbox(const unsigned long long* __restrict__ accum, const uint32_t* __restrict__ list,
                               const unsigned int* __restrict__ n_list, unsigned char* dst, size_t seg, int parity, int world,
                               int rank, uint32_t cap, Counters* __restrict__ ctr) {
  const uint32_t n = min(*n_list, cap);
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t k0 = blockIdx.x * blockDim.x + threadIdx.x; k0 < n; k0 += ILP * stride) {
    uint32_t vv[ILP];
    ulonglong2 aa[ILP];
#pragma unroll
    for (int m = 0; m < ILP; ++m) vv[m] = (k0 + m * stride < n) ? list[k0 + m * stride] : 0xFFFFFFFFu;
#pragma unroll
    for (int m = 0; m < ILP; ++m)
      if (vv[m] != 0xFFFFFFFFu) aa[m] = *reinterpret_cast<const ulonglong2*>(&accum[2 * (size_t)vv[m]]);
#pragma unroll
    for (int m = 0; m < ILP; ++m) {
      if (vv[m] == 0xFFFFFFFFu) continue;
      const uint32_t v = vv[m];
      const ulonglong2 a = aa[m];
      const size_t off = exch_record_offset(parity, world, rank, cap, k0 + m * stride);
      // accumulator cell: a.x = r << 32 | g, a.y = b << 32 | count
      const uint32_t r = (uint32_t)(a.x >> 32), g = (uint32_t)a.x, b = (uint32_t)(a.y >> 32), n_frag = (uint32_t)a.y;
      if ((r | g | b | n_frag) >> 24) ctr->overflow = 1;
      const uint4 q = make_uint4((r & 0xFFFFFFu) | (n_frag << 24), (g & 0xFFFFFFu) | ((n_frag >> 8) << 24),
                                 (b & 0xFFFFFFu) | ((n_frag >> 16) << 24), v);
      if (MODE == 1) multimem_st_v4(dst + off, q);
      else if (MODE == 2) { for (int p = 0; p < world; ++p) if (p != rank) *reinterpret_cast<uint4*>(dst + (size_t)p * seg + off) = q; }
      else *reinterpret_cast<uint4*>(dst + off) = q;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const size_t off = (size_t)(parity * 16 + rank) * 4;
    if (MODE == 1) multimem_st_u32(reinterpret_cast<uint32_t*>(dst + off), n);
    else if (MODE == 2) { for (int p = 0; p < world; ++p) *reinterpret_cast<uint32_t*>(dst + (size_t)p * seg + off) = n; }
    else *reinterpret_cast<uint32_t*>(dst + off) = n;
  }
}

// One launch per remote rank, in stream order.  A rank's records name distinct voxels and nothing else writes the
// accumulator between the barrier and the resolve, so each record is a plain 16-byte read-modify-write of its cell
// (no atomics); the cell read also tells whether the voxel is new to this rank's touched list.
__global__ void vox_merge_inbox(unsigned long long* __restrict__ accum, const unsigned char* __restrict__ inbox, int parity,
                                int world, int src_rank, uint32_t cap, uint32_t* __restrict__ touched,
                                unsigned int* __restrict__ n_touched, Counters* __restrict__ ctr, const unsigned int* own_n) {
  const uint32_t* counts = reinterpret_cast<const uint32_t*>(inbox) + parity * 16;
  if (blockIdx.x == 0 && threadIdx.x == 0 && *own_n > cap) ctr->overflow = 1;   // this rank touched more voxels than fit
  const uint32_t n = min(counts[src_rank], cap);
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t k0 = blockIdx.x * blockDim.x + threadIdx.x; k0 < n; k0 += ILP * stride) {
    uint4 q[ILP];
    ulonglong2 a[ILP];
#pragma unroll
    for (int m = 0; m < ILP; ++m) {
      q[m] = make_uint4(0u, 0u, 0u, 0xFFFFFFFFu);
      if (k0 + m * stride < n) q[m] = *reinterpret_cast<const uint4*>(inbox + exch_record_offset(parity, world, src_rank, cap, k0 + m * stride));
    }
#pragma unroll
    for (int m = 0; m < ILP; ++m)       // the records of one rank name distinct voxels: no hazard between the ILP cells
      if (q[m].w != 0xFFFFFFFFu) a[m] = *reinterpret_cast<const ulonglong2*>(&accum[2 * (size_t)q[m].w]);
#pragma unroll
    for (int m = 0; m < ILP; ++m) {
      if (q[m].w == 0xFFFFFFFFu) continue;
      const uint32_t v = q[m].w, n_frag = (q[m].x >> 24) | ((q[m].y >> 24) << 8) | ((q[m].z >> 24) << 16);
      const unsigned long long old = a[m].y;
      a[m].x += ((unsigned long long)(q[m].x & 0xFFFFFFu) << 32) | (q[m].y & 0xFFFFFFu);
      a[m].y += ((unsigned long long)(q[m].z & 0xFFFFFFu) << 32) | n_frag;
      *reinterpret_cast<ulonglong2*>(&accum[2 * (size_t)v]) = a[m];
      append_first_touch(old, v, touched, n_touched);
    }
  }
}

static int voxelize_inbox(vct_context* c, size_t tb, size_t te, bool slot_ready);
static int resolve_inbox(vct_context* c);

int launch_voxelize_shared(vct_context* c, size_t tb, size_t te) {
  if (c->shared_local && c->shared_exchange == 0) return voxelize_inbox(c, tb, te, false);
  if (!c->shared_local) return set_error(c, VCT_ERR_STATE, "vct_voxelize_shared: call vct_comm_init or vct_set_shared_accum first");
  if (c->comm && c->shared_world > 1 && !c->shared_mc)
    return set_error(c, VCT_ERR_STATE, "vct_voxelize_shared: SharedExchange = 1 (in-switch reduction) needs the multicast mapping");
  int rc = ensure_grid(c); if (rc) return rc;
  const size_t n = (size_t)c->P.V * c->P.V * c->P.V;
  if (c->push_cap != n) {
    cudaFree(c->d_push_list); cudaFree(c->d_push_count); c->d_push_list = nullptr; c->d_push_count = nullptr;
    VCT_CUDA(c, cudaMalloc(&c->d_push_list, n * 4));
    VCT_CUDA(c, cudaMalloc(&c->d_push_count, 128));
    c->push_cap = n;
  }
  if (c->accum_list_slot != -2)      // the private accumulator must start all zero; vox_push_shared leaves it that way
    VCT_CUDA(c, cudaMemsetAsync(c->d_accum, 0, n * 16, c->stream));
  c->accum_list_slot = -2;
  VCT_CUDA(c, cudaMemsetAsync(c->d_push_count, 0, 4, c->stream));
  rc = voxelize_impl(c, tb, te, 1); if (rc) return rc;
  {
    PassTimer timer(c, VCT_PASS_EXCHANGE_PUSH);
    if (c->shared_mc)
      vox_push_shared<true><<<VCT_CHAIN(8), 0, c->stream>>>(c->d_accum, c->d_push_list, c->d_push_count, (float4*)c->shared_mc, c->P.V);
    else
      vox_push_shared<false><<<VCT_CHAIN(8), 0, c->stream>>>(c->d_accum, c->d_push_list, c->d_push_count, (float4*)c->shared_local, c->P.V);
    c->launches += 1;
  }
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

// Mask-driven resolve of the symmetric accumulator into the current slot: one thread per 32-voxel mask word.
// Writes the resolved texel for every set bit, a zero texel for voxels that this slot held before and that are no
// longer occupied, and leaves accumulator cells and mask word zeroed for the next frame.
__global__ void vox_resolve_shared(unsigned long long* __restrict__ accum, uint32_t* __restrict__ mask,
                                   uint32_t* __restrict__ mask_prev, cudaSurfaceObject_t level0, int V, int f16) {
  // warp-cooperative: a warp loads 32 mask words at once, then walks only the non-zero ones with lane b handling
  // bit b of the word (a word is 32 consecutive voxels along x: one 128 B / 256 B run of level 0)
  const size_t n_words = ((size_t)V * V * V) >> 5;
  const unsigned lane = threadIdx.x & 31;
  const size_t warp0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t base = warp0 * 32; base < n_words; base += n_warps * 32) {
    const size_t w = base + lane;
    uint32_t now = 0, before = 0;
    if (w < n_words) { now = mask[w]; before = mask_prev[w]; }
    if (w < n_words && (now | before)) { mask_prev[w] = now; mask[w] = 0u; }
    unsigned todo = __ballot_sync(0xffffffffu, (now | before) != 0u);
    while (todo) {
      const int src = __ffs(todo) - 1;
      todo &= todo - 1;
      const uint32_t wn = __shfl_sync(0xffffffffu, now, src), wb = __shfl_sync(0xffffffffu, before, src);
      const size_t v = ((base + src) << 5) + lane;
      const int x = (int)(v % V), y = (int)((v / V) % V), z = (int)(v / ((size_t)V * V));
      if ((wn >> lane) & 1u) {
        float4* cell = reinterpret_cast<float4*>(accum) + v;
        const float4 f = *cell;                       // exact integers (see multimem_add_v4f32)
        *cell = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        const unsigned long long rg = ((unsigned long long)(unsigned)f.x << 32) | (unsigned)f.y;
        const unsigned long long bc = ((unsigned long long)(unsigned)f.z << 32) | (unsigned)f.w;
        if (f16) surf3Dwrite(resolve_cell16(rg, bc), level0, x * 8, y, z);
        else surf3Dwrite(resolve_cell(rg, bc), level0, x * 4, y, z);
      } else if ((wb >> lane) & 1u) {
        if (f16) surf3Dwrite(make_uint2(0u, 0u), level0, x * 8, y, z);
        else surf3Dwrite(make_uchar4(0, 0, 0, 0), level0, x * 4, y, z);
      }
    }
  }
}

int launch_resolve_shared(vct_context* c) {
  if (!c->shared_local) return set_error(c, VCT_ERR_STATE, "vct_resolve_shared: call vct_set_shared_accum first");
  if (c->shared_exchange == 0) return resolve_inbox(c);
  int rc = ensure_grid(c); if (rc) return rc;
  const int V = c->P.V;
  const size_t n_words = ((size_t)V * V * V) >> 5;
  if (c->mask_prev_V != V) {
    for (int k = 0; k < 2; ++k) {
      cudaFree(c->mask_prev[k]); c->mask_prev[k] = nullptr;
      VCT_CUDA(c, cudaMalloc(&c->mask_prev[k], n_words * 4));
    }
    c->mask_prev_V = V;
    c->mask_valid[0] = c->mask_valid[1] = false;
  }
  rc = begin_voxel_slot(c); if (rc) return rc;
  vct_context::GridBuf& g = c->grid[c->cur];
  PassTimer timer(c, VCT_PASS_RESOLVE);
  if (!c->mask_valid[c->cur]) {    // this slot's level 0 is not described by mask_prev: zero it densely once
    dim3 b(32, 8), gr((V + 31) / 32, (V + 7) / 8, V);
    zero_level0<<<gr, b, 0, c->stream>>>(g.surf[0], V, c->grid_format);
    VCT_CUDA(c, cudaMemsetAsync(c->mask_prev[c->cur], 0, n_words * 4, c->stream));
    c->launches += 1;
  }
  uint32_t* mask = reinterpret_cast<uint32_t*>(c->shared_local + 2 * (size_t)V * V * V);
  vox_resolve_shared<<<VCT_CHAIN(8), 0, c->stream>>>(c->shared_local, mask, c->mask_prev[c->cur], g.surf[0], V, c->grid_format);
  c->launches += 1;
  // the slot is now described by mask_prev, not by a touched list: a later private-accumulator voxelisation into
  // this slot must start from a dense zero, and mask_prev stays exact as long as only this path writes the slot
  g.list_valid = false;
  g.dirty_valid = false; g.occ_valid = false; g.mips_current = false;
  c->mask_valid[c->cur] = true;
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

// slot_ready: the caller (vct_frame_shared_begin) already switched to the slot to build into
int launch_voxelize_inbox_into_slot(vct_context* c, size_t tb, size_t te) { return voxelize_inbox(c, tb, te, true); }

static int voxelize_inbox(vct_context* c, size_t tb, size_t te, bool slot_ready) {
  int rc = ensure_grid(c); if (rc) return rc;
  if (!slot_ready) { rc = begin_voxel_slot(c); if (rc) return rc; }
  rc = launch_voxel_clear(c); if (rc) return rc;             // ordinary sparse clear (lists describe ALL voxels)
  rc = launch_voxelize(c, tb, te); if (rc) return rc;         // this rank's triangles -> private accumulator + list
  vct_context::GridBuf& g = c->grid[c->cur];
  const uint32_t cap = (uint32_t)c->exchange_cap;
  PassTimer timer(c, VCT_PASS_EXCHANGE_PUSH);
  if (c->shared_mc)
    vox_push_inbox<1><<<VCT_CHAIN(4), 0, c->stream>>>(c->d_accum, g.touched, g.n_touched, (unsigned char*)c->shared_mc, 0,
                                                   c->exchange_parity, c->shared_world, c->shared_rank, cap, c->d_counters);
  else if (c->shared_peers && c->shared_world > 1)
    vox_push_inbox<2><<<VCT_CHAIN(4), 0, c->stream>>>(c->d_accum, g.touched, g.n_touched, c->shared_peers, c->shared_seg,
                                                   c->exchange_parity, c->shared_world, c->shared_rank, cap, c->d_counters);
  else
    vox_push_inbox<0><<<VCT_CHAIN(4), 0, c->stream>>>(c->d_accum, g.touched, g.n_touched, (unsigned char*)c->shared_local, 0,
                                                   c->exchange_parity, c->shared_world, c->shared_rank, cap, c->d_counters);
  // own record count, needed by the merge for the overflow check (the list keeps growing during the merge)
  if (!c->d_push_count) VCT_CUDA(c, cudaMalloc(&c->d_push_count, 128));
  VCT_CUDA(c, cudaMemcpyAsync(c->d_push_count, g.n_touched, 4, cudaMemcpyDeviceToDevice, c->stream));
  c->launches += 1;
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

static int resolve_inbox(vct_context* c) {
  vct_context::GridBuf& g = c->grid[c->cur];
  {
    PassTimer timer(c, VCT_PASS_EXCHANGE_MERGE);
    // One launch per remote rank, in stream order: a rank's records name distinct voxels, so each is a plain 16-byte
    // read-modify-write.  (All ranks in one launch with atomic adds was measured: 185 us instead of 89 at four ranks.)
    for (int r = 0; r < c->shared_world; ++r) {
      if (r == c->shared_rank) continue;
      vox_merge_inbox<<<VCT_CHAIN(4), 0, c->stream>>>(c->d_accum, (const unsigned char*)c->shared_local, c->exchange_parity,
                                                   c->shared_world, r, (uint32_t)c->exchange_cap, g.touched, g.n_touched,
                                                   c->d_counters, c->d_push_count);
      c->launches += 1;
    }
  }
  c->exchange_parity ^= 1;
  int rc = launch_resolve(c, false); if (rc) return rc;
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

int launch_resolve(vct_context* c, bool dense) {
  int rc = ensure_grid(c); if (rc) return rc;
  PassTimer timer(c, VCT_PASS_RESOLVE);
  const int V = c->P.V;
  vct_context::GridBuf& g = c->grid[c->cur];
  if (dense) {
    dim3 b(32, 8), gr((V + 31) / 32, (V + 7) / 8, V);
    vox_resolve_dense<<<gr, b, 0, c->stream>>>(c->d_accum, g.surf[0], V, c->grid_format);
    g.list_valid = false;           // every texel was rewritten from the accumulator, the list was not maintained
    g.dirty_valid = false; g.occ_valid = false;
    c->mask_valid[c->cur] = false;
    c->accum_list_slot = -1;
  } else {
    vox_resolve_sparse<<<VCT_CHAIN(8), 0, c->stream>>>(c->d_accum, g.touched, g.n_touched, g.surf[0], V, c->grid_format, g.dirty_now);
    g.occ_valid = g.list_valid;
  }
  g.mips_current = false;
  c->launches += 1;
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

int readback_accum(vct_context* c, uint32_t* counts, uint32_t* sums) {
  int rc = ensure_grid(c); if (rc) return rc;
  const size_t n = (size_t)c->P.V * c->P.V * c->P.V;
  uint32_t *dc = nullptr, *ds = nullptr;
  if (counts) VCT_CUDA(c, cudaMalloc(&dc, n * 4));
  if (sums) VCT_CUDA(c, cudaMalloc(&ds, n * 12));
  accum_to_counts<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_accum, n, dc, ds);
  c->launches += 1;
  cudaError_t e = cudaSuccess;
  if (counts) e = cudaMemcpyAsync(counts, dc, n * 4, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess && sums) e = cudaMemcpyAsync(sums, ds, n * 12, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  cudaFree(dc); cudaFree(ds);
  return check_cuda(c, e, "readback_accum");
}

}  // namespace vct
