/*
 * voxel_view_ref.cpp -- CPU reference of the voxel view (vct_render_voxels), TEST INFRASTRUCTURE ONLY.
 *
 * A scalar restatement of the rule of DESIGN.md section 3 "Voxel view", written independently of csrc/vct_view.cu and
 * fed with the CPU oracle's parameters and mip pyramid (tests/voxel_view_ref.py).  Every float operation is a single
 * IEEE binary32 (or, for the inverse camera matrix, binary64) operation in source order; it is compiled with
 * -ffp-contract=off so that nothing is fused, and then agrees with the device in every byte, texel index and step count.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>

extern "C" {
/* the uniforms the view reads, in the layout of the oracle's orc_params fields of the same names */
typedef struct vv_params {
  int32_t VoxelDimensions, GridFormat, screen_width, screen_height;
  float VoxelGridWorldSize, ambientFactor;
  float ModelMatrix[16], ModelViewMatrix[16], ProjectionMatrix[16];
} vv_params;
}

namespace {

struct V4 { float x, y, z, w; };

/* ((m0*x + m1*y) + m2*z) + m3*w, column-major */
inline V4 mul_mat_vec(const float* m, float x, float y, float z, float w) {
  V4 r;
  r.x = ((m[0] * x + m[4] * y) + m[8] * z) + m[12] * w;
  r.y = ((m[1] * x + m[5] * y) + m[9] * z) + m[13] * w;
  r.z = ((m[2] * x + m[6] * y) + m[10] * z) + m[14] * w;
  r.w = ((m[3] * x + m[7] * y) + m[11] * z) + m[15] * w;
  return r;
}

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

/* C = A * B, column-major, double, glm's operator* order */
void mat4_mul_d(const double* A, const double* B, double* C) {
  for (int j = 0; j < 4; ++j)
    for (int i = 0; i < 4; ++i)
      C[j * 4 + i] = ((A[0 * 4 + i] * B[j * 4 + 0] + A[1 * 4 + i] * B[j * 4 + 1]) + A[2 * 4 + i] * B[j * 4 + 2]) +
                     A[3 * 4 + i] * B[j * 4 + 3];
}

/* glm::inverse(mat4), compute_inverse<4, 4>: the 18 cofactors Coef00..Coef23, Fac0..Fac5, Vec0..Vec3, Inv0..Inv3, signs,
 * then every element times 1 / ((Dot0.x + Dot0.y) + (Dot0.z + Dot0.w)).  M(c, r) = column c, row r. */
void mat4_inverse_glm_d(const double* a, double* out) {
#define M(c, r) a[(c) * 4 + (r)]
  const double Coef00 = M(2, 2) * M(3, 3) - M(3, 2) * M(2, 3);
  const double Coef02 = M(1, 2) * M(3, 3) - M(3, 2) * M(1, 3);
  const double Coef03 = M(1, 2) * M(2, 3) - M(2, 2) * M(1, 3);
  const double Coef04 = M(2, 1) * M(3, 3) - M(3, 1) * M(2, 3);
  const double Coef06 = M(1, 1) * M(3, 3) - M(3, 1) * M(1, 3);
  const double Coef07 = M(1, 1) * M(2, 3) - M(2, 1) * M(1, 3);
  const double Coef08 = M(2, 1) * M(3, 2) - M(3, 1) * M(2, 2);
  const double Coef10 = M(1, 1) * M(3, 2) - M(3, 1) * M(1, 2);
  const double Coef11 = M(1, 1) * M(2, 2) - M(2, 1) * M(1, 2);
  const double Coef12 = M(2, 0) * M(3, 3) - M(3, 0) * M(2, 3);
  const double Coef14 = M(1, 0) * M(3, 3) - M(3, 0) * M(1, 3);
  const double Coef15 = M(1, 0) * M(2, 3) - M(2, 0) * M(1, 3);
  const double Coef16 = M(2, 0) * M(3, 2) - M(3, 0) * M(2, 2);
  const double Coef18 = M(1, 0) * M(3, 2) - M(3, 0) * M(1, 2);
  const double Coef19 = M(1, 0) * M(2, 2) - M(2, 0) * M(1, 2);
  const double Coef20 = M(2, 0) * M(3, 1) - M(3, 0) * M(2, 1);
  const double Coef22 = M(1, 0) * M(3, 1) - M(3, 0) * M(1, 1);
  const double Coef23 = M(1, 0) * M(2, 1) - M(2, 0) * M(1, 1);
  const double Fac0[4] = {Coef00, Coef00, Coef02, Coef03}, Fac1[4] = {Coef04, Coef04, Coef06, Coef07};
  const double Fac2[4] = {Coef08, Coef08, Coef10, Coef11}, Fac3[4] = {Coef12, Coef12, Coef14, Coef15};
  const double Fac4[4] = {Coef16, Coef16, Coef18, Coef19}, Fac5[4] = {Coef20, Coef20, Coef22, Coef23};
  const double Vec0[4] = {M(1, 0), M(0, 0), M(0, 0), M(0, 0)}, Vec1[4] = {M(1, 1), M(0, 1), M(0, 1), M(0, 1)};
  const double Vec2[4] = {M(1, 2), M(0, 2), M(0, 2), M(0, 2)}, Vec3[4] = {M(1, 3), M(0, 3), M(0, 3), M(0, 3)};
  const double SignA[4] = {+1, -1, +1, -1}, SignB[4] = {-1, +1, -1, +1};
  double inv[16];
  for (int k = 0; k < 4; ++k) {
    inv[0 * 4 + k] = ((Vec1[k] * Fac0[k] - Vec2[k] * Fac1[k]) + Vec3[k] * Fac2[k]) * SignA[k];
    inv[1 * 4 + k] = ((Vec0[k] * Fac0[k] - Vec2[k] * Fac3[k]) + Vec3[k] * Fac4[k]) * SignB[k];
    inv[2 * 4 + k] = ((Vec0[k] * Fac1[k] - Vec1[k] * Fac3[k]) + Vec3[k] * Fac5[k]) * SignA[k];
    inv[3 * 4 + k] = ((Vec0[k] * Fac2[k] - Vec1[k] * Fac4[k]) + Vec2[k] * Fac5[k]) * SignB[k];
  }
  const double Dot0[4] = {M(0, 0) * inv[0], M(0, 1) * inv[4], M(0, 2) * inv[8], M(0, 3) * inv[12]};
  const double OneOverDeterminant = 1.0 / ((Dot0[0] + Dot0[1]) + (Dot0[2] + Dot0[3]));
  for (int k = 0; k < 16; ++k) out[k] = inv[k] * OneOverDeterminant;
#undef M
}

inline uint8_t unorm8(float x) {
  x = std::fmin(std::fmax(x, 0.0f), 1.0f);
  if (!(x == x)) x = 0.0f;
  return (uint8_t)std::lrintf(x * 255.0f);
}

inline uint32_t shade8(uint32_t c, int face) {   /* face 0 none, 1 X, 2 Y, 3 Z */
  const uint32_t s = face == 1 ? 218u : face == 3 ? 179u : 256u;
  return (c * s + 128u) >> 8;
}

}  // namespace

extern "C" int vv_render_voxels(const vv_params* pp, int level, const uint8_t* tex, uint8_t* rgba, uint32_t* voxel,
                                uint64_t* steps_out) {
  const vv_params& p = *pp;
  if (level < 0 || (p.VoxelDimensions >> level) < 1) return -1;
  const int W = p.screen_width, H = p.screen_height, N = p.VoxelDimensions >> level;
  /* InvVP = ModelMatrix * inverse(ProjectionMatrix * ModelViewMatrix), double, rounded to float once */
  double model[16], mv[16], proj[16], pmv[16], ipmv[16], r[16];
  for (int k = 0; k < 16; ++k) { model[k] = p.ModelMatrix[k]; mv[k] = p.ModelViewMatrix[k]; proj[k] = p.ProjectionMatrix[k]; }
  mat4_mul_d(proj, mv, pmv);
  mat4_inverse_glm_d(pmv, ipmv);
  mat4_mul_d(model, ipmv, r);
  float inv[16];
  for (int k = 0; k < 16; ++k) inv[k] = (float)r[k];
  const uint8_t bg = unorm8(p.ambientFactor < 0.5f ? 0.5f : 1.0f);
  const bool f16 = p.GridFormat == 1;
  const float fN = (float)N, G = p.VoxelGridWorldSize;
  uint64_t total = 0;
#pragma omp parallel for schedule(dynamic, 4) reduction(+ : total)
  for (int j = 0; j < H; ++j)
    for (int i = 0; i < W; ++i) {
      const float x = (float)(2 * i + 1) / (float)W - 1.0f, y = (float)(2 * j + 1) / (float)H - 1.0f;
      const V4 n = mul_mat_vec(inv, x, y, -1.0f, 1.0f), f = mul_mat_vec(inv, x, y, 1.0f, 1.0f);
      const float org[3] = {(n.x / n.w / G + 0.5f) * fN, (n.y / n.w / G + 0.5f) * fN, (n.z / n.w / G + 0.5f) * fN};
      const float end[3] = {(f.x / f.w / G + 0.5f) * fN, (f.y / f.w / G + 0.5f) * fN, (f.z / f.w / G + 0.5f) * fN};
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
      uint8_t px[4] = {bg, bg, bg, 255};
      uint32_t hit = 0xFFFFFFFFu;
      if (in_box && t_in < t_out) {   /* Amanatides-Woo */
        int v[3], st[3];
        float tm[3], td[3];
        for (int a = 0; a < 3; ++a) {
          v[a] = (int)std::fmin(std::fmax(std::floor(org[a] + t_in * d[a]), 0.0f), (float)(N - 1));
          st[a] = d[a] > 0.0f ? 1 : d[a] < 0.0f ? -1 : 0;
          tm[a] = d[a] == 0.0f ? std::numeric_limits<float>::infinity() : ((float)(v[a] + (st[a] > 0)) - org[a]) * iv[a];
          td[a] = std::fabs(iv[a]);
        }
        for (;;) {
          ++total;
          const size_t t = ((size_t)v[2] * N + v[1]) * N + v[0];
          uint32_t c[3] = {0, 0, 0};
          bool occ;
          if (f16) {
            uint16_t h[4];
            std::memcpy(h, tex + t * 8, 8);
            const float fa = half_to_float(h[3]);
            occ = fa > 0.0f;
            if (occ) for (int k = 0; k < 3; ++k) c[k] = unorm8(half_to_float(h[k]) / fa);
          } else {
            const uint32_t al = tex[t * 4 + 3];
            occ = al > 0;
            if (occ) for (int k = 0; k < 3; ++k) c[k] = std::min(255u, ((uint32_t)tex[t * 4 + k] * 255u + al / 2u) / al);
          }
          if (occ) {
            for (int k = 0; k < 3; ++k) px[k] = (uint8_t)shade8(c[k], face);
            hit = (uint32_t)t;
            break;
          }
          const int a = (tm[0] <= tm[1] && tm[0] <= tm[2]) ? 0 : (tm[1] <= tm[2]) ? 1 : 2;
          if (tm[a] >= t_out) break;
          v[a] += st[a];
          if (v[a] < 0 || v[a] >= N) break;
          tm[a] += td[a];
          face = a + 1;
        }
      }
      const size_t q = (size_t)j * W + i;
      if (rgba) std::memcpy(rgba + q * 4, px, 4);
      if (voxel) voxel[q] = hit;
    }
  if (steps_out) *steps_out = total;
  return 0;
}

