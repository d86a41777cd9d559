/*
 * raycast_ref.cpp -- CPU reference of ray casts (vct_cast_rays), TEST INFRASTRUCTURE ONLY.
 *
 * A scalar restatement of the rule of DESIGN.md section 3 "Ray casts" (the voxel view's steps 3-5 along caller-supplied
 * world-space segments), written independently of csrc/vct_view.cu and of the view's reference tests/voxel_view_ref.cpp,
 * and fed with the CPU oracle's parameters and mip pyramid (tests/raycast_ref.py).  Every float operation is a single
 * IEEE binary32 operation in source order; it is compiled with -ffp-contract=off so that nothing is fused, and then
 * agrees with the device in every texel index, entry parameter, face, colour byte and step count.  That the view is a
 * special case of a cast is checked against the view's reference in tests/test_raycast.py.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>

extern "C" {
/* the uniforms a cast reads, in the layout of the oracle's orc_params fields of the same names */
typedef struct rc_params {
  int32_t VoxelDimensions, GridFormat;
  float VoxelGridWorldSize;
} rc_params;
}

namespace {

/* IEEE binary16 -> binary32 (exact) */
inline float half_to_float(uint16_t h) {
  uint32_t sign = (uint32_t)(h & 0x8000u) << 16, exp = (h >> 10) & 0x1F, mant = h & 0x3FFu, x;
  if (exp == 0) {
    if (!mant) x = sign;
    else { int e = -1; do { ++e; mant <<= 1; } while (!(mant & 0x400u)); x = sign | ((uint32_t)(127 - 15 - e) << 23) | ((mant & 0x3FFu) << 13); }
  } else if (exp == 31) x = sign | 0x7F800000u | (mant << 13);
  else x = sign | ((exp - 15 + 127) << 23) | (mant << 13);
  float f; std::memcpy(&f, &x, 4); return f;
}

inline uint8_t unorm8(float x) {
  x = std::fmin(std::fmax(x, 0.0f), 1.0f);
  if (!(x == x)) x = 0.0f;
  return (uint8_t)std::lrintf(x * 255.0f);
}

/* what walk() found: the first occupied texel of the segment, the axis it was entered through (0 none, 1 X, 2 Y, 3 Z),
 * the segment parameter there, its un-premultiplied colour and unorm8 alpha, and the texels visited */
struct Hit {
  bool hit = false;
  uint32_t idx = 0xFFFFFFFFu;
  int face = 0;
  float t = 0.0f;
  uint32_t c[3] = {0, 0, 0}, alpha = 0;
  uint32_t steps = 0;
};

/* rule steps 2 (the view's 3-5) for the texel-space segment org -> end (t in [0, 1]) through the N^3 level tex */
Hit walk(const float org[3], const float end[3], int N, const uint8_t* tex, bool f16) {
  Hit h;
  const float fN = (float)N;
  float d[3], iv[3] = {0.0f, 0.0f, 0.0f};
  bool in_box = true;
  float t_in = 0.0f, t_out = 1.0f;
  int face = 0;
  for (int a = 0; a < 3; ++a) {   /* slab test; entry face = first strict maximum in (none, X, Y, Z) */
    d[a] = end[a] - org[a];
    if (!std::isfinite(org[a]) || !std::isfinite(d[a])) in_box = false;
    else if (d[a] == 0.0f) { if (!(org[a] >= 0.0f && org[a] <= fN)) in_box = false; }
    else {
      iv[a] = 1.0f / d[a];
      const float t0 = (0.0f - org[a]) * iv[a], t1 = (fN - org[a]) * iv[a];
      const float lo = t1 < t0 ? t1 : t0, hi = t0 < t1 ? t1 : t0;
      if (lo > t_in) { t_in = lo; face = a + 1; }
      if (hi < t_out) t_out = hi;
    }
  }
  if (!(in_box && t_in < t_out)) return h;
  int v[3], st[3];   /* Amanatides-Woo */
  float tm[3], td[3];
  for (int a = 0; a < 3; ++a) {
    v[a] = (int)std::fmin(std::fmax(std::floor(org[a] + t_in * d[a]), 0.0f), (float)(N - 1));
    st[a] = d[a] > 0.0f ? 1 : d[a] < 0.0f ? -1 : 0;
    tm[a] = d[a] == 0.0f ? std::numeric_limits<float>::infinity() : ((float)(v[a] + (st[a] > 0)) - org[a]) * iv[a];
    td[a] = std::fabs(iv[a]);
  }
  float t_enter = t_in;
  for (;;) {
    ++h.steps;
    const size_t t = ((size_t)v[2] * N + v[1]) * N + v[0];
    uint32_t c[3] = {0, 0, 0}, alpha = 0;
    bool occ;
    if (f16) {
      uint16_t hx[4];
      std::memcpy(hx, tex + t * 8, 8);
      const float fa = half_to_float(hx[3]);
      occ = fa > 0.0f;
      if (occ) { for (int k = 0; k < 3; ++k) c[k] = unorm8(half_to_float(hx[k]) / fa); alpha = unorm8(fa); }
    } else {
      const uint32_t al = tex[t * 4 + 3];
      occ = al > 0;
      if (occ) { for (int k = 0; k < 3; ++k) c[k] = std::min(255u, ((uint32_t)tex[t * 4 + k] * 255u + al / 2u) / al); alpha = al; }
    }
    if (occ) {
      h.hit = true; h.idx = (uint32_t)t; h.face = face; h.t = t_enter;
      for (int k = 0; k < 3; ++k) h.c[k] = c[k];
      h.alpha = alpha;
      return h;
    }
    const int a = (tm[0] <= tm[1] && tm[0] <= tm[2]) ? 0 : (tm[1] <= tm[2]) ? 1 : 2;
    if (tm[a] >= t_out) return h;
    v[a] += st[a];
    if (v[a] < 0 || v[a] >= N) return h;
    t_enter = tm[a];
    tm[a] += td[a];
    face = a + 1;
  }
}

}  // namespace

/* n world-space segments seg[6k..6k+5] = a.xyz, b.xyz through mip `level` (tex, the level's texels); outputs may be NULL */
extern "C" int rc_cast_rays(const rc_params* pp, int level, const uint8_t* tex, size_t n, const float* seg, uint32_t* voxel,
                            float* t, uint8_t* face, uint8_t* rgba, uint32_t* steps) {
  const rc_params& p = *pp;
  if (level < 0 || (p.VoxelDimensions >> level) < 1) return -1;
  const int N = p.VoxelDimensions >> level;
  const bool f16 = p.GridFormat == 1;
  const float fN = (float)N, G = p.VoxelGridWorldSize;
#pragma omp parallel for schedule(dynamic, 4096)
  for (long long k = 0; k < (long long)n; ++k) {
    const float* s = seg + 6 * k;
    const float org[3] = {(s[0] / G + 0.5f) * fN, (s[1] / G + 0.5f) * fN, (s[2] / G + 0.5f) * fN};
    const float end[3] = {(s[3] / G + 0.5f) * fN, (s[4] / G + 0.5f) * fN, (s[5] / G + 0.5f) * fN};
    const Hit h = walk(org, end, N, tex, f16);
    if (voxel) voxel[k] = h.idx;
    if (t) t[k] = h.hit ? h.t : std::numeric_limits<float>::infinity();
    if (face) {   /* outward normal of the entry face: -sign(d) along the entry axis; 1..6 = +X, -X, +Y, -Y, +Z, -Z */
      uint8_t f = 0;
      if (h.hit && h.face) f = (uint8_t)(2 * h.face - (end[h.face - 1] - org[h.face - 1] > 0.0f ? 0 : 1));
      face[k] = f;
    }
    if (rgba) {
      const uint8_t px[4] = {(uint8_t)h.c[0], (uint8_t)h.c[1], (uint8_t)h.c[2], (uint8_t)h.alpha};
      std::memcpy(rgba + 4 * k, px, 4);
    }
    if (steps) steps[k] = h.steps;
  }
  return 0;
}
