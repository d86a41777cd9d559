// vct_view.cu -- walks through one mip level of the current pyramid: the voxel view (vct_render_voxels), one level drawn
// as cubes from the camera, and ray casts (vct_cast_rays) along caller-supplied world-space segments.  No reference
// counterpart.  Both walk their segment through the level's texels with the Amanatides-Woo traversal of walk_texels and
// stop at the first occupied one.  The arithmetic is the rule of DESIGN.md section 3 "Voxel view" and "Ray casts",
// written as single binary32 operations in source order (the TU is built with --fmad=false), so the CPU references of
// the tests (tests/voxel_view_ref.cpp for the view, tests/raycast_ref.cpp for casts) reproduce every byte, index, entry
// parameter and step count.
#include <cuda_fp16.h>

#include "vct_internal.h"

namespace vct {

struct Mat16 { float m[16]; };

// face shading weights /256: none and +-Y 256, +-X 218, +-Z 179
__device__ __forceinline__ unsigned shade8(unsigned c, int face) {
  const unsigned s = face == 1 ? 218u : face == 3 ? 179u : 256u;
  return (c * s + 128u) >> 8;
}

// DESIGN.md section 3 "Voxel view" steps 3-5 for the texel-space segment o -> e (t in [0, 1]) through the N^3 level:
// adds the texels it visits to `steps` and, at the first occupied one, calls
//   on_hit(idx, face, t, r, g, b, a)
// with its index (z N + y) N + x, the axis it was entered through (1, 2, 3 = X, Y, Z; 0 = none: the walk started in it),
// the segment parameter there (t_in, or the stepped axis's tMax), its colour un-premultiplied and its alpha as unorm8.
// The hit is reported where it is found and the counter is the caller's, so a caller that ignores an argument (the view:
// t and alpha) leaves its arithmetic dead and keeps no extra register live across the walk.
template <class OnHit>
__device__ __forceinline__ void walk_texels(const float o[3], const float e[3], int N, cudaSurfaceObject_t level, int f16,
                                            unsigned& steps, OnHit on_hit) {
  const float fN = (float)N;
  float d[3], iv[3];
  bool hit_box = true;
  float t_in = 0.0f, t_out = 1.0f;
  int face = 0;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    d[a] = e[a] - o[a];
    iv[a] = 0.0f;
    if (!isfinite(o[a]) || !isfinite(d[a])) hit_box = false;
    else if (d[a] == 0.0f) { if (!(o[a] >= 0.0f && o[a] <= fN)) hit_box = false; }
    else {
      iv[a] = 1.0f / d[a];
      const float t0 = (0.0f - o[a]) * iv[a], t1 = (fN - o[a]) * iv[a];
      const float lo = t1 < t0 ? t1 : t0, hi = t0 < t1 ? t1 : t0;
      if (lo > t_in) { t_in = lo; face = a + 1; }
      if (hi < t_out) t_out = hi;
    }
  }
  if (hit_box && t_in < t_out) {
    // scalar per-axis state: an array indexed by the chosen axis would live in local memory
    int v[3], st[3];
    float tm[3], td[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      v[a] = (int)fminf(fmaxf(floorf(o[a] + t_in * d[a]), 0.0f), (float)(N - 1));
      st[a] = d[a] > 0.0f ? 1 : d[a] < 0.0f ? -1 : 0;
      tm[a] = d[a] == 0.0f ? __int_as_float(0x7f800000) : ((float)(v[a] + (st[a] > 0)) - o[a]) * iv[a];
      td[a] = fabsf(iv[a]);
    }
    int vx = v[0], vy = v[1], vz = v[2];
    float tx = tm[0], ty = tm[1], tz = tm[2];
    float t_enter = t_in;
    for (;;) {
      ++steps;
      unsigned r = 0, g = 0, b = 0, al8 = 0;
      bool occ;
      if (f16) {
        const uint2 t = surf3Dread<uint2>(level, vx * 8, vy, vz);
        const float fa = __half2float(__ushort_as_half((unsigned short)(t.y >> 16)));
        occ = fa > 0.0f;
        if (occ) {
          r = to_unorm8(__half2float(__ushort_as_half((unsigned short)(t.x & 0xFFFFu))) / fa);
          g = to_unorm8(__half2float(__ushort_as_half((unsigned short)(t.x >> 16))) / fa);
          b = to_unorm8(__half2float(__ushort_as_half((unsigned short)(t.y & 0xFFFFu))) / fa);
          al8 = to_unorm8(fa);
        }
      } else {
        const uchar4 t = surf3Dread<uchar4>(level, vx * 4, vy, vz);
        const unsigned al = t.w;
        occ = al > 0u;
        if (occ) {   // un-premultiply: a coarse texel averages occupied and empty children
          r = min(255u, (t.x * 255u + al / 2u) / al);
          g = min(255u, (t.y * 255u + al / 2u) / al);
          b = min(255u, (t.z * 255u + al / 2u) / al);
          al8 = al;
        }
      }
      if (occ) {
        on_hit(((uint32_t)vz * (uint32_t)N + (uint32_t)vy) * (uint32_t)N + (uint32_t)vx, face, t_enter, r, g, b, al8);
        break;
      }
      // next voxel: the axis with the smallest tMax, ties X, Y, Z
      if (tx <= ty && tx <= tz) {
        if (tx >= t_out) break;
        vx += st[0];
        if (vx < 0 || vx >= N) break;
        t_enter = tx; tx += td[0]; face = 1;
      } else if (ty <= tz) {
        if (ty >= t_out) break;
        vy += st[1];
        if (vy < 0 || vy >= N) break;
        t_enter = ty; ty += td[1]; face = 2;
      } else {
        if (tz >= t_out) break;
        vz += st[2];
        if (vz < 0 || vz >= N) break;
        t_enter = tz; tz += td[2]; face = 3;
      }
    }
  }
}

// one warp = 8x4 pixels (as cone_trace); block = 8 warps = 32x8 pixels
__global__ void __launch_bounds__(256) voxel_view(Params P, Mat16 inv, int N, cudaSurfaceObject_t level, int f16,
                                                  uchar4* __restrict__ frame, uint32_t* __restrict__ voxel,
                                                  Counters* __restrict__ ctr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + (warp & 3) * 8 + (lane & 7);
  const int j = blockIdx.y * 8 + (warp >> 2) * 4 + (lane >> 3);
  unsigned steps = 0;
  if (i < P.W && j < P.H) {
    const float x = (float)(2 * i + 1) / (float)P.W - 1.0f, y = (float)(2 * j + 1) / (float)P.H - 1.0f;
    const F4 n = mul_mat_vec(inv.m, x, y, -1.0f, 1.0f), f = mul_mat_vec(inv.m, x, y, 1.0f, 1.0f);
    const float fN = (float)N, G = P.grid_world;
    const float o[3] = {(n.x / n.w / G + 0.5f) * fN, (n.y / n.w / G + 0.5f) * fN, (n.z / n.w / G + 0.5f) * fN};
    const float e[3] = {(f.x / f.w / G + 0.5f) * fN, (f.y / f.w / G + 0.5f) * fN, (f.z / f.w / G + 0.5f) * fN};
    uchar4 out;
    uint32_t idx = 0xFFFFFFFFu;
    bool hit = false;
    walk_texels(o, e, N, level, f16, steps, [&](uint32_t k, int face, float, unsigned r, unsigned g, unsigned b, unsigned) {
      out = make_uchar4(shade8(r, face), shade8(g, face), shade8(b, face), 255);
      idx = k;
      hit = true;
    });
    if (!hit) {   // the frame's clear colour, computed after the walk so that it holds no register during it
      const unsigned char bg = to_unorm8(P.ambient < 0.5f ? 0.5f : 1.0f);
      out = make_uchar4(bg, bg, bg, 255);
    }
    frame[(size_t)j * P.W + i] = out;
    if (voxel) voxel[(size_t)j * P.W + i] = idx;
  }
  count_steps(ctr, STEPS_VIEW, lane, steps, [] { return (blockIdx.x + blockIdx.y * 7u) & 63u; });
}

int launch_voxel_view(vct_context* c, int level, const float inv_vp[16], uint32_t* d_voxel) {
  PassTimer timer(c, VCT_PASS_VOXEL_VIEW);
  VCT_CUDA(c, reset_steps(c, STEPS_VIEW));
  Mat16 inv;
  for (int k = 0; k < 16; ++k) inv.m[k] = inv_vp[k];
  dim3 b(256), g((c->P.W + 31) / 32, (c->P.H + 7) / 8);
  voxel_view<<<g, b, 0, c->stream>>>(c->P, inv, c->P.V >> level, c->grid[c->cur].surf[level], c->grid_format == 1,
                                     c->d_frame, d_voxel, c->d_counters);
  c->launches += 1;
  c->last_frame = c->d_frame;
  mark_slot_read(c);
  return check_cuda(c, cudaGetLastError(), "voxel_view");
}

// Ray casts (DESIGN.md section 3 "Ray casts"): one thread per world-space segment a -> b (seg: a.xyz, b.xyz), the view's
// walk from (a/G + 0.5) N to (b/G + 0.5) N.  face: outward normal of the entry face, 1..6 = +X, -X, +Y, -Y, +Z, -Z.
__global__ void __launch_bounds__(256) cast_rays_kernel(float G, int N, cudaSurfaceObject_t level, int f16, size_t n,
                                                        const float* __restrict__ seg, uint32_t* __restrict__ voxel,
                                                        float* __restrict__ t, uint8_t* __restrict__ face,
                                                        uchar4* __restrict__ rgba, uint32_t* __restrict__ steps_out,
                                                        Counters* __restrict__ ctr) {
  const size_t k = (size_t)blockIdx.x * 256 + threadIdx.x;
  unsigned steps = 0;
  if (k < n) {
    const float* s = seg + 6 * k;
    const float fN = (float)N;
    const float o[3] = {(s[0] / G + 0.5f) * fN, (s[1] / G + 0.5f) * fN, (s[2] / G + 0.5f) * fN};
    const float e[3] = {(s[3] / G + 0.5f) * fN, (s[4] / G + 0.5f) * fN, (s[5] / G + 0.5f) * fN};
    uint32_t idx = 0xFFFFFFFFu;
    int axis = 0;
    float th = __int_as_float(0x7f800000);
    uchar4 c = make_uchar4(0, 0, 0, 0);
    walk_texels(o, e, N, level, f16, steps, [&](uint32_t hk, int hf, float ht, unsigned r, unsigned g, unsigned b, unsigned a) {
      idx = hk; axis = hf; th = ht; c = make_uchar4(r, g, b, a);
    });
    voxel[k] = idx;
    if (t) t[k] = th;
    if (face) {
      // the normal is -sign(d) along the entry axis, which the walk only takes where d != 0; axis 0: a miss, or the
      // segment started inside the hit texel
      const float da = axis == 1 ? e[0] - o[0] : axis == 2 ? e[1] - o[1] : e[2] - o[2];
      face[k] = (uint8_t)(axis ? 2 * axis - (da > 0.0f ? 0 : 1) : 0);
    }
    if (rgba) rgba[k] = c;
    if (steps_out) steps_out[k] = steps;
  }
  count_steps(ctr, STEPS_RAYS, threadIdx.x & 31, steps, [] { return blockIdx.x & 63u; });
}

int launch_cast_rays(vct_context* c, int level, size_t n, const float* seg, uint32_t* voxel, float* t, uint8_t* face,
                     uint8_t* rgba, uint32_t* steps) {
  const size_t blocks = (n + 255) / 256;
  if (blocks > 0x7fffffffu) return set_error(c, VCT_ERR_INVALID, "vct_cast_rays: too many segments for one launch");
  PassTimer timer(c, VCT_PASS_RAYS);
  VCT_CUDA(c, reset_steps(c, STEPS_RAYS));
  cast_rays_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(c->P.grid_world, c->P.V >> level, c->grid[c->cur].surf[level],
                                                            c->grid_format == 1, n, seg, voxel, t, face, (uchar4*)rgba,
                                                            steps, c->d_counters);
  c->launches += 1;
  mark_slot_read(c);
  return check_cuda(c, cudaGetLastError(), "cast_rays");
}

}  // namespace vct
