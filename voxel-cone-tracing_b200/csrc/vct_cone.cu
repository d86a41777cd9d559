// vct_cone.cu -- S2 + C1..C6: primary visibility and per-pixel cone tracing.
// Replaces Render() (Voxel_Cone_Tracing.h:146-190) and Shader/VoxelConeTracing.{vs,fs}.
//
// The reference is a forward renderer: the cone-trace fragment shader runs on rasterised scene geometry
// with the hardware depth test and `discard` on alpha < 0.5, and shades overdrawn fragments.  Here the
// work is split into
//   visibility (raster_small / raster_tiles): VoxelConeTracing.vs:25 + viewport + back-face cull + depth
//        LESS + alpha discard, as 2D homogeneous rasterisation (no clipping; the near plane is enforced
//        per fragment).  Output: 64-bit atomicMin of (depth bits << 32 | triangle id) per pixel.
//   cone_trace: one thread per pixel, one warp per 8x4 screen tile; rebuilds the interpolated varyings
//        of the winning triangle and evaluates VoxelConeTracing.fs:165-229 exactly once per pixel.
//        Voxel fetches are hardware trilinear tex3DLod on the mipmapped cudaArray (wrap = REPEAT).
#include <cuda_fp16.h>

#include "vct_raster.cuh"

namespace vct {

struct HVert { float X, Y, w, zc; };
struct HEdge { float A, B, C; };

__device__ __forceinline__ HEdge hcross(const HVert& a, const HVert& b) {
  HEdge e;
  e.A = a.Y * b.w - b.Y * a.w;
  e.B = b.X * a.w - a.X * b.w;
  e.C = a.X * b.Y - b.X * a.Y;
  return e;
}
__device__ __forceinline__ float heval(const HEdge& e, float px, float py) { return (e.A * px + e.B * py) + e.C; }
__device__ __forceinline__ bool hinside(const HEdge& e, float v) {
  return v > 0.0f || (v == 0.0f && (e.A > 0.0f || (e.A == 0.0f && e.B > 0.0f)));
}

struct HTri {
  HVert c[3];
  HEdge e[3];   // e[i] opposite vertex i
};

// VoxelConeTracing.vs:25 + viewport transform + GL_CULL_FACE(GL_BACK) as homogeneous set-up
template <bool WITH_BBOX>
__device__ __forceinline__ bool setup_htri(const Params& P, const VertexCache& vc,
                                           const uint32_t* __restrict__ idx, uint32_t tri, HTri& t, int& i0,
                                           int& i1, int& j0, int& j1) {
  const float W = (float)P.W, H = (float)P.H;
  bool in_near[3];
  bool any_near = false;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float4 c = __ldg(&vc.clip[__ldg(&idx[tri * 3 + k])]);       // VoxelConeTracing.vs:25 + viewport (vertex_pass)
    if (!(c.z == c.z)) return false;                                   // a clip coordinate was not finite
    t.c[k].X = c.x; t.c[k].Y = c.y; t.c[k].w = c.z; t.c[k].zc = c.w;
    in_near[k] = (c.w >= -c.z) && (c.z > 0.0f);
    any_near |= in_near[k];
  }
  if (!any_near) return false;
  t.e[0] = hcross(t.c[1], t.c[2]);
  t.e[1] = hcross(t.c[2], t.c[0]);
  t.e[2] = hcross(t.c[0], t.c[1]);
  float det = (t.c[0].X * t.e[0].A + t.c[0].Y * t.e[0].B) + t.c[0].w * t.e[0].C;
  if (!(det > 0.0f)) return false;
  if (!WITH_BBOX) return true;

  float minx = INFINITY, maxx = -INFINITY, miny = INFINITY, maxy = -INFINITY;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int n = (k + 1) % 3;
    if (in_near[k]) {
      float x = t.c[k].X / t.c[k].w, y = t.c[k].Y / t.c[k].w;
      minx = fminf(minx, x); maxx = fmaxf(maxx, x); miny = fminf(miny, y); maxy = fmaxf(maxy, y);
    }
    if (in_near[k] != in_near[n]) {
      float da = t.c[k].zc + t.c[k].w, db = t.c[n].zc + t.c[n].w;
      float s = da / (da - db);
      float X = t.c[k].X + s * (t.c[n].X - t.c[k].X);
      float Y = t.c[k].Y + s * (t.c[n].Y - t.c[k].Y);
      float w = t.c[k].w + s * (t.c[n].w - t.c[k].w);
      if (w > 0.0f) {
        float x = X / w, y = Y / w;
        minx = fminf(minx, x); maxx = fmaxf(maxx, x); miny = fminf(miny, y); maxy = fmaxf(maxy, y);
      } else {
        minx = miny = -1e30f; maxx = maxy = 1e30f;
      }
    }
  }
  if (!(minx <= maxx)) return false;
  float fx0 = fmaxf(floorf(minx) - 1.0f, 0.0f), fx1 = fminf(ceilf(maxx) + 1.0f, W - 1.0f);
  const bool strips = P.row_il > 1;      // interleaved strips: the box spans the frame, ownership is tested per row / tile
  const float rb = strips ? 0.0f : (float)P.row_begin, re = (float)((!strips && P.row_end > 0 && P.row_end < P.H) ? P.row_end : P.H);
  float fy0 = fmaxf(floorf(miny) - 1.0f, rb), fy1 = fminf(ceilf(maxy) + 1.0f, re - 1.0f);
  if (!(fx0 <= fx1) || !(fy0 <= fy1)) return false;
  i0 = (int)fx0; i1 = (int)fx1; j0 = (int)fy0; j1 = (int)fy1;
  return true;
}

template <bool TEST>
__device__ __forceinline__ bool hbary(const HTri& t, float px, float py, float b[3]) {
  float e0 = heval(t.e[0], px, py), e1 = heval(t.e[1], px, py), e2 = heval(t.e[2], px, py);
  if (TEST && !(hinside(t.e[0], e0) && hinside(t.e[1], e1) && hinside(t.e[2], e2))) return false;
  float s = (e0 + e1) + e2;
  if (TEST && !(s > 0.0f)) return false;
  b[0] = e0 / s; b[1] = e1 / s; b[2] = e2 / s;
  return true;
}

__device__ __forceinline__ float bary3(const float b[3], float a0, float a1, float a2) {
  return (b[0] * a0 + b[1] * a1) + b[2] * a2;
}

struct PixelUV { float u, v, dudx, dvdx, dudy, dvdy; };

__device__ __forceinline__ PixelUV pixel_uv(const VertexCache& vc, const uint32_t* __restrict__ idx,
                                            uint32_t tri, const HTri& t, float px, float py, const float b[3]) {
  const uint32_t i0 = __ldg(&idx[tri * 3 + 0]), i1 = __ldg(&idx[tri * 3 + 1]), i2 = __ldg(&idx[tri * 3 + 2]);
  const float u0 = __ldg(&vc.nrm_u[i0].w), u1 = __ldg(&vc.nrm_u[i1].w), u2 = __ldg(&vc.nrm_u[i2].w);
  const float w0 = __ldg(&vc.tan_v[i0].w), w1 = __ldg(&vc.tan_v[i1].w), w2 = __ldg(&vc.tan_v[i2].w);
  PixelUV r;
  r.u = bary3(b, u0, u1, u2);
  r.v = bary3(b, w0, w1, w2);
  float bx[3], by[3];
  hbary<false>(t, px + 1.0f, py, bx);
  hbary<false>(t, px, py + 1.0f, by);
  r.dudx = bary3(bx, u0, u1, u2) - r.u;
  r.dvdx = bary3(bx, w0, w1, w2) - r.v;
  r.dudy = bary3(by, u0, u1, u2) - r.u;
  r.dvdy = bary3(by, w0, w1, w2) - r.v;
  return r;
}

__device__ __forceinline__ float4 sample_mat(cudaTextureObject_t tex, int w, int h, const PixelUV& q, float du, float dv) {
  float lod = lod_from_derivs(q.dudx, q.dvdx, q.dudy, q.dvdy, w, h);
  return sample_material(tex, q.u + du, q.v + dv, lod);
}

// ---------------------------------------------------------------------------------------------------
struct VisibilityPass {
  Params P;
  VertexCache vc; const uint32_t* idx; const uint16_t* trimat; const MaterialDev* mats;
  unsigned long long* vis;

  static constexpr bool kAppends = false;
  static constexpr bool kWarpMedium = true;
  struct Setup { HTri t; };

  __device__ __forceinline__ bool setup(uint32_t tri, Setup& s, int& i0, int& i1, int& j0, int& j1) const {
    return setup_htri<true>(P, vc, idx, tri, s.t, i0, i1, j0, j1);
  }
  // Exact tile reject.  IEEE rounding is monotonic, so the COMPUTED value (A*px + B*py) + C is monotonic in px
  // and in py separately; its maximum over the pixel centres of a tile is the computed value at the corner
  // chosen by the signs of A and B.  If that maximum fails the inside test no pixel of the tile can pass.
  __device__ __forceinline__ bool setup_full(uint32_t tri, Setup& s, int& i0, int& i1, int& j0, int& j1) const {
    return setup(tri, s, i0, i1, j0, j1);
  }
  // interleaved strips: 8x8 tiles are aligned with the 8-row strips, so only every row_il-th tile row is walked
  __device__ __forceinline__ void tile_rows(int& ty0, int& ty1, int& step) const {
    if (P.row_il <= 1) return;
    step = P.row_il;
    ty0 += ((P.row_ph - ty0) % step + step) % step;          // first owned tile row >= ty0
    if (ty0 <= ty1) ty1 = ty0 + ((ty1 - ty0) / step) * step;  // last owned tile row <= ty1
  }
  __device__ __forceinline__ bool tile_may_cover(const Setup& s, int x0, int y0, int x1, int y1) const {
    if (P.row_il > 1 && !row_owned(P, y0)) return false;     // (cannot happen after tile_rows; kept as a guard)
    const float xa = (float)x0 + 0.5f, xb = (float)(x1 - 1) + 0.5f, ya = (float)y0 + 0.5f, yb = (float)(y1 - 1) + 0.5f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const HEdge& e = s.t.e[k];
      const float v = heval(e, e.A >= 0.0f ? xb : xa, e.B >= 0.0f ? yb : ya);
      if (!hinside(e, v)) return false;
    }
    return true;
  }

  __device__ __forceinline__ void shade(const Setup& s, uint32_t tri, int i, int j) const {
    const float px = (float)i + 0.5f, py = (float)j + 0.5f;
    const float e0 = heval(s.t.e[0], px, py), e1 = heval(s.t.e[1], px, py), e2 = heval(s.t.e[2], px, py);
    if (!(hinside(s.t.e[0], e0) && hinside(s.t.e[1], e1) && hinside(s.t.e[2], e2))) return;
    if (!((e0 + e1) + e2 > 0.0f)) return;
    // z_clip / w_clip: the common 1/(e0+e1+e2) cancels -> one division per fragment
    const float zc = (e0 * s.t.c[0].zc + e1 * s.t.c[1].zc) + e2 * s.t.c[2].zc;
    const float w = (e0 * s.t.c[0].w + e1 * s.t.c[1].w) + e2 * s.t.c[2].w;
    const float zw = (zc / w) * 0.5f + 0.5f;
    if (!(zw >= 0.0f) || zw > 1.0f) return;                 // near / far clip
    const unsigned long long key = ((unsigned long long)__float_as_uint(zw) << 32) | tri;
    unsigned long long* cell = &vis[(size_t)j * P.W + i];   // no early-z read: RED.MIN is fire-and-forget, a load is not
    const MaterialDev& m = mats[trimat ? trimat[tri] : 0];
    if (m.alpha_test) {                                     // discard, VoxelConeTracing.fs:167-172
      float b[3];
      hbary<false>(s.t, px, py, b);
      PixelUV q = pixel_uv(vc, idx, tri, s.t, px, py, b);
      float4 c = sample_mat(m.diffuse, m.dw, m.dh, q, 0.0f, 0.0f);
      if (c.w < 0.5f) return;
    }
    atomicMin(cell, key);
  }
  __device__ __forceinline__ void small(const Setup& s, uint32_t tri, bool active, int i0, int i1, int j0, int j1) const {
    if (!active) return;
    for (int j = j0; j <= j1; ++j) {
      if (P.row_il > 1 && !row_owned(P, j)) continue;
      for (int i = i0; i <= i1; ++i) shade(s, tri, i, j);
    }
  }
  __device__ __forceinline__ void pixel(const Setup& s, uint32_t tri, int i, int j, bool in_bbox) const {
    if (in_bbox && (P.row_il <= 1 || row_owned(P, j))) shade(s, tri, i, j);
  }
};

__global__ void fill_u64(unsigned long long* p, size_t n, unsigned long long v) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

int launch_visibility(vct_context* c) {
  if (!c->nt) return set_error(c, VCT_ERR_STATE, "vct_render: no mesh uploaded");
  int rc = ensure_frame(c); if (rc) return rc;
  rc = ensure_queues(c); if (rc) return rc;
  rc = sync_materials(c); if (rc) return rc;
  rc = ensure_vertex_cache(c); if (rc) return rc;
  PassTimer timer(c, VCT_PASS_VISIBILITY);
  const size_t n = (size_t)c->P.W * c->P.H;
  fill_u64<<<VCT_CHAIN(4), 0, c->stream>>>(c->d_vis2[c->cur], n, ~0ull);
  VCT_CUDA(c, reset_item_queue(c));
  VisibilityPass pass{c->P, c->vcache2[c->cur], c->d_idx, c->d_trimat, c->d_materials, c->d_vis2[c->cur]};
  const uint32_t nt = (uint32_t)c->nt;
  raster_small<VisibilityPass><<<(nt + 127) / 128, 128, 0, c->stream>>>(pass, 0, nt, c->d_items, (uint32_t)c->items_cap, c->d_counters);
  raster_tiles<VisibilityPass><<<VCT_CHAIN(4), 0, c->stream>>>(pass, c->d_items, (uint32_t)c->items_cap, c->d_counters);
  c->launches += 3;
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

// ---------------------------------------------------------------------------------------------------
struct V3 { float x, y, z; };
__device__ __forceinline__ V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ V3 vadd(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ V3 vsub(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ V3 vscale(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float vdot(V3 a, V3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }
__device__ __forceinline__ V3 vcross(V3 a, V3 b) {
  return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ V3 vnormalize(V3 a) {
  float l = sqrtf(vdot(a, a));
  return v3(a.x / l, a.y / l, a.z / l);
}

// tolerance-level normalisation (MUFU.RSQ, ~2 ulp) for shading vectors; anything that feeds a coverage or
// shadow-compare decision keeps IEEE division / sqrt.
__device__ __forceinline__ V3 vnormalize_fast(V3 a) {
  float r = rsqrtf(vdot(a, a));
  return v3(a.x * r, a.y * r, a.z * r);
}

struct ConeConsts { float vws, inv_vws, inv_grid; };

__device__ __forceinline__ ConeConsts cone_consts(const Params& P) {
  ConeConsts k;
  k.vws = P.grid_world / (float)P.V;      // voxelWorldSize, VoxelConeTracing.fs:90
  k.inv_vws = (float)P.V / P.grid_world;
  k.inv_grid = 1.0f / P.grid_world;
  return k;
}

// Voxel_Cone_Tracing(direction, tanHalfAngle), VoxelConeTracing.fs:82-107, with SampleVoxels (:59-66) folded in:
// uvw = pos / (G/2) * 0.5 + 0.5 = pos / G + 0.5, advanced along the ray with one FMA per axis; textureLod
// clamps lod to [0, log2 V] in hardware (maxMipmapLevelClamp).  This loop is tolerance-level arithmetic (its
// inputs already carry the 8-bit hardware filter weights), so it uses FMAs, MUFU log2 and MUFU reciprocal:
// ~25 instructions per sample instead of ~110 with IEEE division and libm log2f.
__device__ __forceinline__ float4 cone_march(cudaTextureObject_t grid, const Params& P, const ConeConsts& k,
                                             V3 start, V3 dir, float tanHalf, unsigned& samples) {
  float cr = 0.0f, cg = 0.0f, cb = 0.0f, alpha = 0.0f, occ = 0.0f;
  float dist = k.vws;
  const float two_tan = 2.0f * tanHalf;
  const float u0 = __fmaf_rn(start.x, k.inv_grid, 0.5f), v0 = __fmaf_rn(start.y, k.inv_grid, 0.5f),
              w0 = __fmaf_rn(start.z, k.inv_grid, 0.5f);
  const float du = dir.x * k.inv_grid, dv = dir.y * k.inv_grid, dw = dir.z * k.inv_grid;
  const float max_dist = P.max_dist, max_alpha = P.max_alpha, step_mult = P.step_mult;
  while (dist < max_dist && alpha < max_alpha) {
    const float diameter = fmaxf(k.vws, two_tan * dist);
    const float lod = __log2f(diameter * k.inv_vws);
    const float4 s = tex3DLod<float4>(grid, __fmaf_rn(dist, du, u0), __fmaf_rn(dist, dv, v0), __fmaf_rn(dist, dw, w0), lod);
    const float t = 1.0f - alpha;
    cr = __fmaf_rn(t, s.x, cr); cg = __fmaf_rn(t, s.y, cg); cb = __fmaf_rn(t, s.z, cb);
    const float ta = t * s.w;
    occ = __fmaf_rn(ta, __frcp_rn(__fmaf_rn(0.03f, diameter, 1.0f)), occ);
    alpha += ta;
    dist = __fmaf_rn(diameter, step_mult, dist);
    ++samples;
  }
  return make_float4(cr, cg, cb, occ);
}

// All diffuse cones of a pixel share tanHalfAngle and the start distance, hence the whole (dist, diameter,
// lod) sequence: they are marched in lockstep so that every step issues up to NC independent tex3DLod
// fetches (memory-level parallelism) instead of NC dependent chains, and the specular cone -- the longest
// chain, up to 29 steps at 256^3 -- advances in the same loop.  The per-cone weights (Cone_Weights,
// VoxelConeTracing.fs:48) are folded into the accumulation: sum_c w_c * sum_i (1-alpha_c,i) * s_c,i.
// Cone directions live in shared memory ([component][cone][thread], conflict free) so that the march loop
// keeps its register budget for the accumulators: 18 LDS per lockstep step on an otherwise idle LSU pipe.
template <int NC, int SU>
__device__ __forceinline__ void march_pixel(cudaTextureObject_t grid, const Params& P, const ConeConsts& k, V3 start,
                                            const float* __restrict__ sdir /* smem, stride blockDim.x */,
                                            V3 spec_dir, float4& diffuse, float4& specular, unsigned& samples) {
  const int n = min(P.n_cones, NC);
  const int stride = blockDim.x;
  const float u0 = __fmaf_rn(start.x, k.inv_grid, 0.5f), v0 = __fmaf_rn(start.y, k.inv_grid, 0.5f),
              w0 = __fmaf_rn(start.z, k.inv_grid, 0.5f);
  const float max_dist = P.max_dist, max_alpha = P.max_alpha, step_mult = P.step_mult;
  float alpha[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) alpha[c] = 0.0f;
  // diffuse state (shared distance sequence)
  float dr = 0.0f, dg = 0.0f, db = 0.0f, docc = 0.0f;
  float ddist = k.vws;
  const float d2t = 2.0f * P.diffuse_tan;
  bool d_any = n > 0;
  // specular state
  float sr = 0.0f, sg = 0.0f, sb = 0.0f, socc = 0.0f, salpha = 0.0f;
  float sdist = k.vws;
  const float s2t = 2.0f * P.spec_tan;
  const float su = spec_dir.x * k.inv_grid, sv = spec_dir.y * k.inv_grid, sw = spec_dir.z * k.inv_grid;
  bool s_on = true;
  // The sample positions of a cone depend only on the step index, never on the fetched values (only the
  // early exit does), so SU specular steps are fetched ahead per iteration and composited in order; fetches
  // past the exit are discarded (<= SU-1 per pixel) and not counted as samples.
  while (true) {
    d_any = d_any && (ddist < max_dist);
    s_on = s_on && (sdist < max_dist) && (salpha < max_alpha);
    if (!d_any && !s_on) break;
    float4 ss[SU];
    float sdiam[SU];
    if (s_on) {                                  // issue the specular fetches first: they head the longest chain
      float dk = sdist;
#pragma unroll
      for (int q = 0; q < SU; ++q) {
        sdiam[q] = fmaxf(k.vws, s2t * dk);
        // unconditional: a fetch past MAX_DISTANCE wraps like any other (GL_REPEAT) and is discarded below
        ss[q] = tex3DLod<float4>(grid, __fmaf_rn(dk, su, u0), __fmaf_rn(dk, sv, v0), __fmaf_rn(dk, sw, w0),
                                 __log2f(sdiam[q] * k.inv_vws));
        dk = __fmaf_rn(sdiam[q], step_mult, dk);
      }
    }
    if (d_any) {
      const float diam = fmaxf(k.vws, d2t * ddist);
      const float lod = __log2f(diam * k.inv_vws);
      const float rocc = __frcp_rn(__fmaf_rn(0.03f, diam, 1.0f));
      float4 s[NC];
      bool any = false;
      // (no array of predicates between the two loops: nvcc 12.9 miscompiled `bool on[NC]` carried across the texture
      // fetches in some register allocations -- wrong pixels with NC = 9 / SU = 2 -- so the condition is recomputed;
      // alpha[c] does not change in between)
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if ((c < n) && (alpha[c] < max_alpha)) {
          const float du = sdir[(0 * NC + c) * stride], dv = sdir[(1 * NC + c) * stride], dw = sdir[(2 * NC + c) * stride];
          s[c] = tex3DLod<float4>(grid, __fmaf_rn(ddist, du, u0), __fmaf_rn(ddist, dv, v0), __fmaf_rn(ddist, dw, w0), lod);
          ++samples;
        }
      }
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if ((c < n) && (alpha[c] < max_alpha)) {
          const float t = P.cone_w[c] * (1.0f - alpha[c]);
          dr = __fmaf_rn(t, s[c].x, dr); dg = __fmaf_rn(t, s[c].y, dg); db = __fmaf_rn(t, s[c].z, db);
          docc = __fmaf_rn(t * s[c].w, rocc, docc);
          alpha[c] = __fmaf_rn(1.0f - alpha[c], s[c].w, alpha[c]);
          any = any || (alpha[c] < max_alpha);
        }
      }
      d_any = any;
      ddist = __fmaf_rn(diam, step_mult, ddist);
    }
    if (s_on) {
#pragma unroll
      for (int q = 0; q < SU; ++q) {
        if (sdist < max_dist && salpha < max_alpha) {   // VoxelConeTracing.fs:94 loop condition, evaluated per step
          const float t = 1.0f - salpha;
          sr = __fmaf_rn(t, ss[q].x, sr); sg = __fmaf_rn(t, ss[q].y, sg); sb = __fmaf_rn(t, ss[q].z, sb);
          const float ta = t * ss[q].w;
          socc = __fmaf_rn(ta, __frcp_rn(__fmaf_rn(0.03f, sdiam[q], 1.0f)), socc);
          salpha += ta;
          sdist = __fmaf_rn(sdiam[q], step_mult, sdist);
          ++samples;
        }
      }
    }
  }
  diffuse = make_float4(dr, dg, db, docc);
  specular = make_float4(sr, sg, sb, socc);
}

// one warp = 8x4 pixels; block = 2 warps = 8x8 pixels (small blocks: the specular chain length varies a lot
// between warps and a block holds its registers until its slowest warp is done)
constexpr int BT = 64;
template <int NC, int SU, int MINB>
__global__ void __launch_bounds__(BT, MINB) cone_trace(Params P, VertexCache vc,
                                                  const uint32_t* __restrict__ idx,
                                                  const uint16_t* __restrict__ trimat,
                                                  const MaterialDev* __restrict__ mats,
                                                  const uint32_t* __restrict__ depth,
                                                  const unsigned long long* __restrict__ vis,
                                                  cudaTextureObject_t grid, uchar4* __restrict__ frame,
                                                  Counters* __restrict__ ctr, int y_begin, int y_end) {
  extern __shared__ float s_dirs[];   // [3][NC][blockDim.x]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lx = lane & 7, ly = lane >> 3;    // 8x4 pixel tile per warp (a 2x2-quad lane order measured the same)
  const int i = blockIdx.x * 8 + lx;
  // rows of this block: contiguous from y_begin, or (interleaved strips) the blockIdx.y-th owned group of 8 rows
  const int j = P.row_il > 1 ? ((int)blockIdx.y * P.row_il + P.row_ph) * 8 + warp * 4 + ly
                             : y_begin + (int)blockIdx.y * 8 + warp * 4 + ly;
  unsigned samples = 0;
  if (i < P.W && j < y_end) {
    const unsigned long long key = vis[(size_t)j * P.W + i];
    uchar4 out;
    if (key == ~0ull) {
      // glClearColor, Voxel_Cone_Tracing.h:156-159
      unsigned char bg = to_unorm8(P.ambient < 0.5f ? 0.5f : 1.0f);
      out = make_uchar4(bg, bg, bg, 255);
    } else {
      const uint32_t tri = (uint32_t)key;
      HTri t;
      int d0, d1, d2, d3;
      setup_htri<false>(P, vc, idx, tri, t, d0, d1, d2, d3);
      const float px = (float)i + 0.5f, py = (float)j + 0.5f;
      float b[3];
      hbary<false>(t, px, py, b);
      // vertex shader outputs (VoxelConeTracing.vs:27-34), then perspective-correct interpolation
      V3 Pw = v3(0, 0, 0), Nw = v3(0, 0, 0), Tw = v3(0, 0, 0), Bw = v3(0, 0, 0);
      float pdx = 0, pdy = 0, pdz = 0, pdw = 0;
      {
        float4 pw[3], pd[3], nw[3], tw[3], bw[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const uint32_t vi = __ldg(&idx[tri * 3 + k]);
          pw[k] = __ldg(&vc.world[vi]); pd[k] = __ldg(&vc.dc[vi]);
          nw[k] = __ldg(&vc.nrm_u[vi]); tw[k] = __ldg(&vc.tan_v[vi]); bw[k] = __ldg(&vc.bit[vi]);
        }
        Pw = v3(bary3(b, pw[0].x, pw[1].x, pw[2].x), bary3(b, pw[0].y, pw[1].y, pw[2].y), bary3(b, pw[0].z, pw[1].z, pw[2].z));
        Nw = v3(bary3(b, nw[0].x, nw[1].x, nw[2].x), bary3(b, nw[0].y, nw[1].y, nw[2].y), bary3(b, nw[0].z, nw[1].z, nw[2].z));
        Tw = v3(bary3(b, tw[0].x, tw[1].x, tw[2].x), bary3(b, tw[0].y, tw[1].y, tw[2].y), bary3(b, tw[0].z, tw[1].z, tw[2].z));
        Bw = v3(bary3(b, bw[0].x, bw[1].x, bw[2].x), bary3(b, bw[0].y, bw[1].y, bw[2].y), bary3(b, bw[0].z, bw[1].z, bw[2].z));
        pdx = bary3(b, pd[0].x, pd[1].x, pd[2].x); pdy = bary3(b, pd[0].y, pd[1].y, pd[2].y);
        pdz = bary3(b, pd[0].z, pd[1].z, pd[2].z); pdw = bary3(b, pd[0].w, pd[1].w, pd[2].w);
      }
      const V3 Cd = vsub(v3(P.cam[0], P.cam[1], P.cam[2]), Pw);       // VoxelConeTracing.vs:34

      const MaterialDev m = mats[trimat ? trimat[tri] : 0];
      const PixelUV q = pixel_uv(vc, idx, tri, t, px, py, b);
      const float4 mat = sample_mat(m.diffuse, m.dw, m.dh, q, 0.0f, 0.0f);    // :167

      // TBN = inverse(transpose(mat3(T,B,N))), :175 -- rows of the matrix being inverted are T, B, N
      const float c00 = Bw.y * Nw.z - Bw.z * Nw.y;
      const float c01 = Bw.z * Nw.x - Bw.x * Nw.z;
      const float c02 = Bw.x * Nw.y - Bw.y * Nw.x;
      const float det = (Tw.x * c00 + Tw.y * c01) + Tw.z * c02;
      const float id = __frcp_rn(det);
      float inv[3][3];
      inv[0][0] = c00 * id; inv[1][0] = c01 * id; inv[2][0] = c02 * id;
      inv[0][1] = (Tw.z * Nw.y - Tw.y * Nw.z) * id;
      inv[1][1] = (Tw.x * Nw.z - Tw.z * Nw.x) * id;
      inv[2][1] = (Tw.y * Nw.x - Tw.x * Nw.y) * id;
      inv[0][2] = (Tw.y * Bw.z - Tw.z * Bw.y) * id;
      inv[1][2] = (Tw.z * Bw.x - Tw.x * Bw.z) * id;
      inv[2][2] = (Tw.x * Bw.y - Tw.y * Bw.x) * id;
      auto tbn_mul = [&](V3 a) {
        return v3((inv[0][0] * a.x + inv[0][1] * a.y) + inv[0][2] * a.z,
                  (inv[1][0] * a.x + inv[1][1] * a.y) + inv[1][2] * a.z,
                  (inv[2][0] * a.x + inv[2][1] * a.y) + inv[2][2] * a.z);
      };

      // CalcBumpNormal, :110-128
      const float offx = 1.0f / (float)m.hw, offy = 1.0f / (float)m.hh;
      const float h0 = sample_mat(m.height, m.hw, m.hh, q, 0.0f, 0.0f).x;
      const float hx = sample_mat(m.height, m.hw, m.hh, q, offx, 0.0f).x;
      const float hy = sample_mat(m.height, m.hw, m.hh, q, 0.0f, offy).x;
      const V3 t1 = vnormalize_fast(v3(1.0f, 0.0f, hx - h0));
      const V3 t2 = vnormalize_fast(v3(0.0f, 1.0f, hy - h0));
      const V3 bump = vnormalize_fast(vcross(t1, t2));
      const V3 N = vnormalize_fast(tbn_mul(bump));
      const V3 L = vnormalize_fast(v3(P.light[0], P.light[1], P.light[2]));   // :179
      const V3 E = vnormalize_fast(Cd);                                         // :181

      // :186 with the *0.111 normalisation of :158
      const float shadow = pcf_lit_taps(depth, P.S, P.pcf_radius, P.shadow_bias, pdx, pdy, pdz, pdw) * 0.111f;
      const float directDiffuse = shadow * fmaxf(vdot(N, L), 0.0f);

      const ConeConsts kc = cone_consts(P);
      const V3 start = vadd(Pw, vscale(Nw, kc.vws));                       // :92
      float* sdir = s_dirs + threadIdx.x;
#pragma unroll
      for (int cidx = 0; cidx < NC; ++cidx) {                              // :196-199
        if (cidx < P.n_cones) {
          const V3 dir = vnormalize_fast(tbn_mul(v3(P.cone_dir[cidx * 3], P.cone_dir[cidx * 3 + 1], P.cone_dir[cidx * 3 + 2])));
          sdir[(0 * NC + cidx) * blockDim.x] = dir.x * kc.inv_grid;
          sdir[(1 * NC + cidx) * blockDim.x] = dir.y * kc.inv_grid;
          sdir[(2 * NC + cidx) * blockDim.x] = dir.z * kc.inv_grid;
        }
      }
      float4 sc = sample_mat(m.specular, m.sw, m.sh, q, 0.0f, 0.0f);      // :209
      if (!(sqrtf(sc.y * sc.y + sc.z * sc.z) > 0.0f)) { sc.y = sc.x; sc.z = sc.x; }   // .rrra, :210
      const V3 negL = v3(-L.x, -L.y, -L.z);
      const V3 R = vnormalize_fast(vsub(negL, vscale(N, 2.0f * vdot(N, negL))));      // :212
      const float spec = __powf(fmaxf(vdot(E, R), 0.0f), m.shininess);                // :213
      const float directSpec = spec * shadow;                                         // :214
      const V3 negE = v3(-E.x, -E.y, -E.z);
      const V3 refl = vnormalize_fast(vsub(negE, vscale(N, 2.0f * vdot(N, negE))));   // :217
      float4 idf, isp;
      march_pixel<NC, SU>(grid, P, kc, start, sdir, refl, idf, isp, samples);               // :196-199 and :218
      const float ir = idf.x, ig = idf.y, ib = idf.z, ia = idf.w;
      const float occlusion = 1.0f - ia;                                   // :201
      const float specOcc = 1.0f - isp.w;                                             // :221

      const float mr[3] = {mat.x, mat.y, mat.z}, ind[3] = {ir, ig, ib}, is3[3] = {isp.x, isp.y, isp.z};
      const float sc3[3] = {sc.x, sc.y, sc.z};
      unsigned char o8[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        float diff = (directDiffuse + occlusion * ind[k]) * mr[k];          // :205
        float specR = (is3[k] + specOcc * directSpec) * sc3[k];             // :223
        float amb = (P.ambient * mr[k]) * occlusion;                        // :225
        o8[k] = to_unorm8((amb + diff) + specR);                            // :227
      }
      out = make_uchar4(o8[0], o8[1], o8[2], to_unorm8(mat.w));
    }
    frame[(size_t)j * P.W + i] = out;
  }
  count_steps(ctr, STEPS_CONE, lane, samples, [] { return (blockIdx.x + blockIdx.y * 7u) & 63u; });   // Gcone-samples/s numerator
}

int launch_cone(vct_context* c) {
  int rc = ensure_frame(c); if (rc) return rc;
  rc = ensure_grid(c); if (rc) return rc;
  if (!c->depth_valid) return set_error(c, VCT_ERR_STATE, "vct_render: call vct_draw_depth first (shadow map missing)");
  rc = ensure_vertex_cache(c); if (rc) return rc;
  PassTimer timer(c, VCT_PASS_CONE);
  VCT_CUDA(c, reset_steps(c, STEPS_CONE));
  int y0 = c->P.row_begin, y1 = (c->P.row_end > 0 && c->P.row_end < c->P.H) ? c->P.row_end : c->P.H;
  const bool strips = c->P.row_il > 1;
  int own_groups = 0;                              // interleaved strips: how many groups of 8 rows this context owns
  if (strips) {
    const int groups = (c->P.H + 7) / 8;
    own_groups = groups > c->P.row_ph ? (groups - c->P.row_ph + c->P.row_il - 1) / c->P.row_il : 0;
    y0 = 0; y1 = c->P.H;
    if (!own_groups) return VCT_OK;
  }
  if (y0 >= y1) return VCT_OK;
  // one shape per cone table: specular fetch-ahead depth SU and register budget via MINB blocks per SM, the fastest
  // measured; <9, 2, 64, 8> and <9, 2, 32, 16> are miscompiled by nvcc 12.9 (profiles/r02_cone_variants.txt)
#define VCT_LAUNCH_CONE(NC, SU, MINB)                                                                                  \
  do {                                                                                                                 \
    dim3 b(BT), g((c->P.W + 7) / 8, strips ? own_groups : (y1 - y0 + 7) / 8);                                          \
    cone_trace<NC, SU, MINB><<<g, b, 3 * NC * BT * sizeof(float), c->stream>>>(c->P, c->vcache2[c->cur], c->d_idx,     \
        c->d_trimat, c->d_materials, c->d_depth, c->d_vis2[c->cur], c->grid[c->cur].tex, c->d_frame, c->d_counters, y0, y1); \
  } while (0)
  if (c->P.n_cones <= 6) VCT_LAUNCH_CONE(6, 4, 10);       // 96 registers, 10 blocks / SM: +2.4 % on config 2
  else if (c->P.n_cones <= 9) VCT_LAUNCH_CONE(9, 4, 8);   // BASELINE config 3: -10 % vs the 16-cone template
  else VCT_LAUNCH_CONE(16, 2, 8);
#undef VCT_LAUNCH_CONE
  c->launches += 1;
  c->last_frame = c->d_frame;
  mark_slot_read(c);
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

// ---------------------------------------------------------------------------------------------------
// Bounces >= 3 (extension; the reference has no re-injection pass, README.md:14 only claims one).
// For every occupied voxel: one diffuse-aperture cone along each of +-X, +-Y, +-Z starting one voxel
// out from the voxel centre, averaged; new = min(old + gathered * old, 1).  Reads the pyramid of the
// previous bounce through the texture, writes a staging buffer, then level 0 (no read/write hazard).
__global__ void __launch_bounds__(256) reinject_gather(Params P, cudaTextureObject_t grid, cudaSurfaceObject_t level0,
                                                       uint2* __restrict__ staged, int f16) {
  const int V = P.V;
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5), z = blockIdx.z;
  if (x >= V || y >= V) return;
  const size_t i = ((size_t)z * V + y) * V + x;
  float b0, b1, b2;
  uint2 raw;
  if (f16) {
    raw = surf3Dread<uint2>(level0, x * 8, y, z);
    if ((raw.y >> 16) == 0u) { staged[i] = make_uint2(0u, 0u); return; }
    b0 = __half2float(__ushort_as_half((unsigned short)(raw.x & 0xFFFFu)));
    b1 = __half2float(__ushort_as_half((unsigned short)(raw.x >> 16)));
    b2 = __half2float(__ushort_as_half((unsigned short)(raw.y & 0xFFFFu)));
  } else {
    const uchar4 old = surf3Dread<uchar4>(level0, x * 4, y, z);
    if (old.w == 0) { staged[i] = make_uint2(0u, 0u); return; }
    raw = make_uint2(0u, (unsigned)old.w);
    b0 = old.x * (1.0f / 255.0f); b1 = old.y * (1.0f / 255.0f); b2 = old.z * (1.0f / 255.0f);
  }
  const ConeConsts kc = cone_consts(P);
  const V3 c = v3(((float)x + 0.5f) * kc.vws - 0.5f * P.grid_world, ((float)y + 0.5f) * kc.vws - 0.5f * P.grid_world,
                  ((float)z + 0.5f) * kc.vws - 0.5f * P.grid_world);
  float acc[3] = {0.0f, 0.0f, 0.0f};
  unsigned dummy = 0;
#pragma unroll 1
  for (int a = 0; a < 6; ++a) {
    const float sgn = (a & 1) ? -1.0f : 1.0f;
    const V3 d = v3((a >> 1) == 0 ? sgn : 0.0f, (a >> 1) == 1 ? sgn : 0.0f, (a >> 1) == 2 ? sgn : 0.0f);
    const float4 r = cone_march(grid, P, kc, vadd(c, vscale(d, kc.vws)), d, P.diffuse_tan, dummy);
    acc[0] += r.x * (1.0f / 6.0f); acc[1] += r.y * (1.0f / 6.0f); acc[2] += r.z * (1.0f / 6.0f);
  }
  const float n0 = fminf(b0 + acc[0] * b0, 1.0f), n1 = fminf(b1 + acc[1] * b1, 1.0f), n2 = fminf(b2 + acc[2] * b2, 1.0f);
  if (f16) {
    staged[i] = make_uint2((unsigned)__half_as_ushort(__float2half_rn(n0)) | ((unsigned)__half_as_ushort(__float2half_rn(n1)) << 16),
                           (unsigned)__half_as_ushort(__float2half_rn(n2)) | (raw.y & 0xFFFF0000u));
  } else {
    uchar4 o;
    o.x = (unsigned char)__float2int_rn(n0 * 255.0f);
    o.y = (unsigned char)__float2int_rn(n1 * 255.0f);
    o.z = (unsigned char)__float2int_rn(n2 * 255.0f);
    o.w = (unsigned char)raw.y;
    staged[i] = make_uint2(*reinterpret_cast<uint32_t*>(&o), 1u);
  }
}

__global__ void reinject_commit(const uint2* __restrict__ staged, cudaSurfaceObject_t level0, int V, int f16) {
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5), z = blockIdx.z;
  if (x >= V || y >= V) return;
  const uint2 v = staged[((size_t)z * V + y) * V + x];
  if (!(v.x | v.y)) return;
  if (f16) surf3Dwrite(v, level0, x * 8, y, z);
  else surf3Dwrite(v.x, level0, x * 4, y, z);
}

int launch_reinject(vct_context* c) {
  int rc = ensure_grid(c); if (rc) return rc;
  PassTimer timer(c, VCT_PASS_REINJECT);
  const int V = c->P.V;
  uint2* staged = nullptr;
  VCT_CUDA(c, cudaMallocAsync(&staged, (size_t)V * V * V * 8, c->stream));
  dim3 b(256), g((V + 31) / 32, (V + 7) / 8, V);
  reinject_gather<<<g, b, 0, c->stream>>>(c->P, c->grid[c->cur].tex, c->grid[c->cur].surf[0], staged, c->grid_format);
  reinject_commit<<<g, b, 0, c->stream>>>(staged, c->grid[c->cur].surf[0], V, c->grid_format);
  c->launches += 2;
  c->grid[c->cur].mips_current = false;   // level 0 changed (occupied voxels only: inside the bricks already flagged)
  VCT_CUDA(c, cudaFreeAsync(staged, c->stream));
  VCT_CUDA(c, cudaGetLastError());
  return VCT_OK;
}

// ---------------------------------------------------------------------------------------------------
__global__ void trace_cones_kernel(Params P, cudaTextureObject_t grid, size_t n, const float* __restrict__ starts,
                                   const float* __restrict__ dirs, const float* __restrict__ tans,
                                   float4* __restrict__ out, uint32_t* __restrict__ steps) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const ConeConsts kc = cone_consts(P);
  unsigned cnt = 0;
  out[i] = cone_march(grid, P, kc, v3(starts[3 * i], starts[3 * i + 1], starts[3 * i + 2]),
                      v3(dirs[3 * i], dirs[3 * i + 1], dirs[3 * i + 2]), tans[i], cnt);
  if (steps) steps[i] = cnt;
}

int launch_trace_cones(vct_context* c, size_t n, const float* starts, const float* dirs, const float* tans, float* out,
                       uint32_t* steps) {
  trace_cones_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->P, c->grid[c->cur].tex, n, starts, dirs, tans,
                                                                         (float4*)out, steps);
  c->launches += 1;
  return check_cuda(c, cudaGetLastError(), "trace_cones");
}

// Irradiance probes (vct_bake_probes, no reference counterpart): the frame's diffuse term (VoxelConeTracing.fs:92,
// :196-201) at caller-supplied points, for a surface facing each of +X, -X, +Y, -Y, +Z, -Z (DESIGN.md section 3
// "Irradiance probes").  One thread per (probe, face); blockIdx.y is the face, so the block's rotated cone directions
// are computed once into shared memory, and consecutive threads take consecutive probes.  Every cone is cone_march, as
// in trace_cones_kernel: a probe equals the float32 composition of vct_trace_cones bit for bit.
constexpr int PROBE_BT = 128;
struct ProbeBasis { float tbn[6][9]; };   // per face: T, B, N

__global__ void __launch_bounds__(PROBE_BT) bake_probes_kernel(Params P, ProbeBasis basis, cudaTextureObject_t grid,
                                                               size_t n, const float* __restrict__ xyz,
                                                               float* __restrict__ out, uint32_t* __restrict__ steps,
                                                               Counters* __restrict__ ctr) {
  __shared__ float s_dir[VCT_MAX_CONES * 3];
  const int face = blockIdx.y;
  const float* tbn = basis.tbn[face];
  const int nc = min(P.n_cones, VCT_MAX_CONES);
  if ((int)threadIdx.x < nc) {
    // d.x T + d.y B + d.z N: one non-zero term per component (a signed permutation of d), so the sum is exact
    const float* d = &P.cone_dir[threadIdx.x * 3];
    const V3 dir = vnormalize(v3((d[0] * tbn[0] + d[1] * tbn[3]) + d[2] * tbn[6], (d[0] * tbn[1] + d[1] * tbn[4]) + d[2] * tbn[7],
                                 (d[0] * tbn[2] + d[1] * tbn[5]) + d[2] * tbn[8]));
    s_dir[threadIdx.x * 3] = dir.x; s_dir[threadIdx.x * 3 + 1] = dir.y; s_dir[threadIdx.x * 3 + 2] = dir.z;
  }
  __syncthreads();
  const size_t p = (size_t)blockIdx.x * PROBE_BT + threadIdx.x;
  unsigned cnt = 0;
  if (p < n) {
    const float x = xyz[3 * p], y = xyz[3 * p + 1], z = xyz[3 * p + 2];
    float4 r = make_float4(NAN, NAN, NAN, NAN);
    if (isfinite(x) && isfinite(y) && isfinite(z)) {
      const ConeConsts kc = cone_consts(P);
      const V3 start = vadd(v3(x, y, z), vscale(v3(tbn[6], tbn[7], tbn[8]), kc.vws));   // :92
      float ir = 0.0f, ig = 0.0f, ib = 0.0f, ia = 0.0f;
#pragma unroll 1
      for (int c = 0; c < nc; ++c) {
        const float4 s = cone_march(grid, P, kc, start, v3(s_dir[c * 3], s_dir[c * 3 + 1], s_dir[c * 3 + 2]), P.diffuse_tan, cnt);
        const float w = P.cone_w[c];
        ir = ir + w * s.x; ig = ig + w * s.y; ib = ib + w * s.z; ia = ia + w * s.w;
      }
      r = make_float4(ir, ig, ib, 1.0f - ia);                                              // ind.rgb, occlusion (:201)
    }
    float* o = out + (p * 6 + face) * 4;
    o[0] = r.x; o[1] = r.y; o[2] = r.z; o[3] = r.w;
    if (steps) steps[p * 6 + face] = cnt;
  }
  count_steps(ctr, STEPS_PROBES, threadIdx.x & 31, cnt, [] { return (blockIdx.x + blockIdx.y * 7u) & 63u; });
}

int launch_probes(vct_context* c, size_t n, const float* xyz, float* out, uint32_t* steps) {
  // DESIGN.md section 3: each row right-handed and orthonormal, faces +X, -X, +Y, -Y, +Z, -Z
  static const ProbeBasis basis = {{{0, 0, -1, 0, 1, 0, 1, 0, 0}, {0, 0, 1, 0, 1, 0, -1, 0, 0},
                                    {1, 0, 0, 0, 0, -1, 0, 1, 0}, {1, 0, 0, 0, 0, 1, 0, -1, 0},
                                    {1, 0, 0, 0, 1, 0, 0, 0, 1}, {-1, 0, 0, 0, 1, 0, 0, 0, -1}}};
  const size_t blocks = (n + PROBE_BT - 1) / PROBE_BT;
  if (blocks > 0x7fffffffu) return set_error(c, VCT_ERR_INVALID, "vct_bake_probes: too many probes for one launch");
  PassTimer timer(c, VCT_PASS_PROBES);
  VCT_CUDA(c, reset_steps(c, STEPS_PROBES));
  bake_probes_kernel<<<dim3((unsigned)blocks, 6), PROBE_BT, 0, c->stream>>>(c->P, basis, c->grid[c->cur].tex, n, xyz, out,
                                                                             steps, c->d_counters);
  c->launches += 1;
  mark_slot_read(c);
  return check_cuda(c, cudaGetLastError(), "bake_probes");
}

__global__ void sample_voxels_kernel(Params P, cudaTextureObject_t grid, size_t n, const float* __restrict__ pos,
                                     const float* __restrict__ lod, float4* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float half = P.grid_world * 0.5f;
  float u = (pos[3 * i] / half) * 0.5f + 0.5f, v = (pos[3 * i + 1] / half) * 0.5f + 0.5f, w = (pos[3 * i + 2] / half) * 0.5f + 0.5f;
  out[i] = tex3DLod<float4>(grid, u, v, w, lod[i]);
}

int launch_sample_voxels(vct_context* c, size_t n, const float* pos, const float* lod, float* out) {
  sample_voxels_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(c->P, c->grid[c->cur].tex, n, pos, lod, (float4*)out);
  c->launches += 1;
  return check_cuda(c, cudaGetLastError(), "sample_voxels");
}

}  // namespace vct
