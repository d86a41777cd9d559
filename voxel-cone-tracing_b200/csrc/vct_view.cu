// vct_view.cu -- voxel view: one mip level of the current pyramid drawn as cubes from the camera (vct_render_voxels).
// No reference counterpart.  One thread per pixel walks its ray through the level's texels with the Amanatides-Woo
// traversal and stops at the first occupied one.  The arithmetic is the rule of DESIGN.md section 3 "Voxel view",
// written as single binary32 operations in source order (the TU is built with --fmad=false), so the CPU reference
// of the tests (tests/voxel_view_ref.cpp) reproduces every byte, index and step count.
#include <cuda_fp16.h>

#include "vct_internal.h"

namespace vct {

struct Mat16 { float m[16]; };

// face shading weights /256: none and +-Y 256, +-X 218, +-Z 179
__device__ __forceinline__ unsigned shade8(unsigned c, int face) {
  const unsigned s = face == 1 ? 218u : face == 3 ? 179u : 256u;
  return (c * s + 128u) >> 8;
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
    uchar4 out;
    uint32_t idx = 0xFFFFFFFFu;
    const unsigned char bg = to_unorm8(P.ambient < 0.5f ? 0.5f : 1.0f);   // the frame's clear colour
    out = make_uchar4(bg, bg, bg, 255);
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
      for (;;) {
        ++steps;
        unsigned r = 0, g = 0, b = 0;
        bool occ;
        if (f16) {
          const uint2 t = surf3Dread<uint2>(level, vx * 8, vy, vz);
          const float fa = __half2float(__ushort_as_half((unsigned short)(t.y >> 16)));
          occ = fa > 0.0f;
          if (occ) {
            r = to_unorm8(__half2float(__ushort_as_half((unsigned short)(t.x & 0xFFFFu))) / fa);
            g = to_unorm8(__half2float(__ushort_as_half((unsigned short)(t.x >> 16))) / fa);
            b = to_unorm8(__half2float(__ushort_as_half((unsigned short)(t.y & 0xFFFFu))) / fa);
          }
        } else {
          const uchar4 t = surf3Dread<uchar4>(level, vx * 4, vy, vz);
          const unsigned al = t.w;
          occ = al > 0u;
          if (occ) {   // un-premultiply: a coarse texel averages occupied and empty children
            r = min(255u, (t.x * 255u + al / 2u) / al);
            g = min(255u, (t.y * 255u + al / 2u) / al);
            b = min(255u, (t.z * 255u + al / 2u) / al);
          }
        }
        if (occ) {
          out = make_uchar4(shade8(r, face), shade8(g, face), shade8(b, face), 255);
          idx = ((uint32_t)vz * (uint32_t)N + (uint32_t)vy) * (uint32_t)N + (uint32_t)vx;
          break;
        }
        // next voxel: the axis with the smallest tMax, ties X, Y, Z
        if (tx <= ty && tx <= tz) {
          if (tx >= t_out) break;
          vx += st[0];
          if (vx < 0 || vx >= N) break;
          tx += td[0]; face = 1;
        } else if (ty <= tz) {
          if (ty >= t_out) break;
          vy += st[1];
          if (vy < 0 || vy >= N) break;
          ty += td[1]; face = 2;
        } else {
          if (tz >= t_out) break;
          vz += st[2];
          if (vz < 0 || vz >= N) break;
          tz += td[2]; face = 3;
        }
      }
    }
    frame[(size_t)j * P.W + i] = out;
    if (voxel) voxel[(size_t)j * P.W + i] = idx;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) steps += __shfl_xor_sync(0xffffffffu, steps, s);
  if (lane == 0 && steps) atomicAdd(&ctr->view_steps[((blockIdx.x + blockIdx.y * 7u) & 63u) * 4], (unsigned long long)steps);
}

int launch_voxel_view(vct_context* c, int level, const float inv_vp[16], uint32_t* d_voxel) {
  PassTimer timer(c, VCT_PASS_VOXEL_VIEW);
  VCT_CUDA(c, cudaMemsetAsync(c->d_counters->view_steps, 0, sizeof(c->d_counters->view_steps), c->stream));
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

}  // namespace vct
