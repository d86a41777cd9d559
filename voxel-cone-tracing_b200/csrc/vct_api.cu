// vct_api.cu -- the C ABI of include/vct_c_api.h: context, uniforms, scene upload, resources, read-back.
#include <cstdio>
#include <cstring>

#include <cuda_fp16.h>

#include "vct_internal.h"

namespace vct {

static thread_local std::string g_create_error;

int set_error(vct_context* c, int code, const std::string& msg) {
  if (c) c->err = msg; else g_create_error = msg;
  return code;
}

int check_cuda(vct_context* c, cudaError_t e, const char* what) {
  if (e == cudaSuccess) return VCT_OK;
  return set_error(c, VCT_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

int readback_accum(vct_context* c, uint32_t* counts, uint32_t* sums);

// ------------------------------------------------------------------------------------------ helpers
static int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

static void set_identity(float* m) {
  std::memset(m, 0, 16 * sizeof(float));
  m[0] = m[5] = m[10] = m[15] = 1.0f;
}

static void default_params(Params& P) {
  std::memset(&P, 0, sizeof(P));
  P.V = 128; P.levels = 8; P.grid_world = 150.0f; P.S = 4096; P.W = 1280; P.H = 720;   // Voxel_Cone_Tracing.h:16-17,24-25,35
  float* mats[] = {P.model, P.model_view, P.proj, P.depth_mvp, P.projx, P.projy, P.projz};
  for (float* m : mats) set_identity(m);
  P.cam[1] = 4.0f;                                       // Voxel_Cone_Tracing.h:8
  P.light[1] = 1.0f; P.light[2] = 0.25f;                 // :14
  P.ambient = 0.1f;                                      // :53
  static const float dirs[18] = {0, 0, 1, 0, 0.866025f, 0.5f, 0.823639f, 0.267617f, 0.5f,
                                 0.509037f, -0.700629f, 0.5f, -0.509037f, -0.700629f, 0.5f,
                                 -0.823639f, 0.267617f, 0.5f};           // VoxelConeTracing.fs:49-57
  static const float wts[6] = {0.25f, 0.15f, 0.15f, 0.15f, 0.15f, 0.15f};  // :48
  P.n_cones = 6;
  std::memcpy(P.cone_dir, dirs, sizeof(dirs));
  std::memcpy(P.cone_w, wts, sizeof(wts));
  P.diffuse_tan = 0.577f; P.spec_tan = 0.07f; P.step_mult = 1.0f;   // :198, :218
  P.max_dist = 75.0f; P.max_alpha = 0.95f;                          // :43-44
  P.pcf_radius = 2; P.shadow_bias = 0.002f;                         // Voxelization.fs:26,88
  P.coverage = 1;                                                   // 4x MSAA window, main.cpp:30
  P.bounces = 2;
}

// ------------------------------------------------------------------------------------------ resources
__global__ void zero_u64(unsigned long long* p, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, st = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += st) p[i] = 0ull;
}

static void free_grid(vct_context* c) {
  for (auto& g : c->grid) {
    if (g.tex) cudaDestroyTextureObject(g.tex);
    for (auto s : g.surf) cudaDestroySurfaceObject(s);
    g.surf.clear();
    if (g.array) cudaFreeMipmappedArray(g.array);
    cudaFree(g.touched); cudaFree(g.n_touched); cudaFree(g.dirty_now); cudaFree(g.dirty_prev);
    g = vct_context::GridBuf();
  }
  cudaFree(c->d_accum); cudaFree(c->d_occ_mask);
  c->d_accum = nullptr; c->d_occ_mask = nullptr; c->grid_V = 0; c->accum_list_slot = -1;
  c->mask_valid[0] = c->mask_valid[1] = false;
}

int ensure_grid(vct_context* c) {
  const int V = c->P.V;
  if (c->grid_V == V && c->grid_fmt_alloc == c->grid_format) return VCT_OK;
  cudaStreamSynchronize(c->stream);
  if (c->stream_vox) cudaStreamSynchronize(c->stream_vox);
  free_grid(c);
  c->grid_fmt_alloc = c->grid_format;
  const size_t n = (size_t)V * V * V;
  VCT_CUDA(c, cudaMalloc(&c->d_accum, n * 16));
  VCT_CUDA(c, cudaMalloc(&c->d_occ_mask, (n + 31) / 32 * 4));
  VCT_CUDA(c, cudaMemsetAsync(c->d_occ_mask, 0, (n + 31) / 32 * 4, c->stream));
  c->touched_cap = n;
  // RGBA8 is the reference's format (GL_RGBA8, Voxel_Cone_Tracing.h:119); RGBA16F is BASELINE config 3
  cudaChannelFormatDesc desc = c->grid_format == 1 ? cudaCreateChannelDescHalf4() : cudaCreateChannelDesc<uchar4>();
  for (auto& g : c->grid) {
    VCT_CUDA(c, cudaMalloc(&g.touched, n * 4));
    VCT_CUDA(c, cudaMalloc(&g.n_touched, 128));
    VCT_CUDA(c, cudaMemsetAsync(g.n_touched, 0, 128, c->stream));
    VCT_CUDA(c, cudaMalloc(&g.dirty_now, dirty_bytes(V)));
    VCT_CUDA(c, cudaMalloc(&g.dirty_prev, dirty_bytes(V)));
    VCT_CUDA(c, cudaMemsetAsync(g.dirty_now, 0, dirty_bytes(V), c->stream));
    VCT_CUDA(c, cudaMemsetAsync(g.dirty_prev, 0, dirty_bytes(V), c->stream));
    VCT_CUDA(c, cudaMallocMipmappedArray(&g.array, &desc, make_cudaExtent(V, V, V), c->P.levels, cudaArraySurfaceLoadStore));
    for (int l = 0; l < c->P.levels; ++l) {
      cudaArray_t lvl;
      VCT_CUDA(c, cudaGetMipmappedArrayLevel(&lvl, g.array, l));
      cudaResourceDesc rd{};
      rd.resType = cudaResourceTypeArray;
      rd.res.array.array = lvl;
      cudaSurfaceObject_t s;
      VCT_CUDA(c, cudaCreateSurfaceObject(&s, &rd));
      g.surf.push_back(s);
    }
    // sampler state of the reference's voxel texture: MIN = LINEAR_MIPMAP_LINEAR, MAG = LINEAR
    // (Voxel_Cone_Tracing.h:112-113), wrap never set => GL_REPEAT on s,t,r.
    cudaResourceDesc rd{};
    rd.resType = cudaResourceTypeMipmappedArray;
    rd.res.mipmap.mipmap = g.array;
    cudaTextureDesc td{};
    td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeWrap;
    td.filterMode = cudaFilterModeLinear;
    td.mipmapFilterMode = cudaFilterModeLinear;
    td.readMode = c->grid_format == 1 ? cudaReadModeElementType : cudaReadModeNormalizedFloat;   // half texels read as float
    td.normalizedCoords = 1;
    td.minMipmapLevelClamp = 0.0f;
    td.maxMipmapLevelClamp = (float)(c->P.levels - 1);
    VCT_CUDA(c, cudaCreateTextureObject(&g.tex, &rd, &td, nullptr));
    g.list_valid = true;
  }
  c->grid_V = V;
  // zero everything: accumulator and all mip levels of both slots (the reference uploads a zeroed texture and
  // calls glGenerateMipmap, Voxel_Cone_Tracing.h:115-126)
  VCT_CUDA(c, cudaMemsetAsync(c->d_accum, 0, n * 16, c->stream));
  for (int k = 0; k < 2; ++k) {
    c->cur = k;
    int rc = launch_resolve(c, true); if (rc) return rc;
    rc = launch_mip(c); if (rc) return rc;
    c->grid[k].list_valid = true;     // all zero: the (empty) list is exact
    c->grid[k].dirty_valid = true;    // ... no brick differs from the pyramid just built
    c->grid[k].occ_valid = true;      // ... and no brick holds a non-zero texel (flags all zero)
  }
  c->cur = 0;
  c->accum_list_slot = 0;             // accumulator all zero, slot 0's empty list describes it
  return VCT_OK;
}

int ensure_shadow(vct_context* c) {
  if (c->depth_S == c->P.S && c->d_depth) return VCT_OK;
  cudaFree(c->d_depth); c->d_depth = nullptr; c->depth_valid = false;
  if (c->depth_tex) { cudaDestroyTextureObject(c->depth_tex); c->depth_tex = 0; }
  if (c->depth_surf) { cudaDestroySurfaceObject(c->depth_surf); c->depth_surf = 0; }
  if (c->depth_array) { cudaFreeArray(c->depth_array); c->depth_array = nullptr; }
  VCT_CUDA(c, cudaMalloc(&c->d_depth, (size_t)c->P.S * c->P.S * 4));
  cudaChannelFormatDesc dd = cudaCreateChannelDesc<float>();
  VCT_CUDA(c, cudaMallocArray(&c->depth_array, &dd, c->P.S, c->P.S, cudaArrayTextureGather | cudaArraySurfaceLoadStore));
  cudaResourceDesc rd{};
  rd.resType = cudaResourceTypeArray;
  rd.res.array.array = c->depth_array;
  VCT_CUDA(c, cudaCreateSurfaceObject(&c->depth_surf, &rd));
  cudaTextureDesc td{};
  td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;    // GL_CLAMP_TO_EDGE, Voxel_Cone_Tracing.h:95-96
  td.filterMode = cudaFilterModePoint;
  td.readMode = cudaReadModeElementType;
  td.normalizedCoords = 0;
  VCT_CUDA(c, cudaCreateTextureObject(&c->depth_tex, &rd, &td, nullptr));
  c->depth_S = c->P.S;
  return VCT_OK;
}

int ensure_frame(vct_context* c) {
  if (c->frame_W == c->P.W && c->frame_H == c->P.H && c->d_frame) return VCT_OK;
  cudaStreamSynchronize(c->stream);
  cudaFree(c->d_vis2[0]); cudaFree(c->d_vis2[1]); cudaFree(c->d_frame);
  c->d_vis2[0] = c->d_vis2[1] = nullptr; c->d_frame = nullptr;
  const size_t n = (size_t)c->P.W * c->P.H;
  VCT_CUDA(c, cudaMalloc(&c->d_vis2[0], n * 8));
  VCT_CUDA(c, cudaMalloc(&c->d_vis2[1], n * 8));
  VCT_CUDA(c, cudaMalloc(&c->d_frame, n * 4));
  c->frame_W = c->P.W; c->frame_H = c->P.H;
  c->last_frame = nullptr;
  return VCT_OK;
}

int ensure_queues(vct_context* c) {
  if (c->frags_cap != c->max_fragments || !c->d_frags) {
    cudaFree(c->d_frags); c->d_frags = nullptr;
    VCT_CUDA(c, cudaMalloc(&c->d_frags, c->max_fragments * sizeof(uint2)));
    c->frags_cap = c->max_fragments;
  }
  if (c->items_cap != c->max_items || !c->d_items) {
    cudaFree(c->d_items); c->d_items = nullptr;
    VCT_CUDA(c, cudaMalloc(&c->d_items, c->max_items * sizeof(TileItem)));
    c->items_cap = c->max_items;
  }
  return VCT_OK;
}

int sync_all_streams(vct_context* c) {
  VCT_CUDA(c, cudaStreamSynchronize(c->stream));
  if (c->stream_vox) VCT_CUDA(c, cudaStreamSynchronize(c->stream_vox));
  if (c->stream2) VCT_CUDA(c, cudaStreamSynchronize(c->stream2));
  if (c->copy_stream) VCT_CUDA(c, cudaStreamSynchronize(c->copy_stream));
  return VCT_OK;
}

int check_overflow(vct_context* c) {
  unsigned int ov = 0, ov2 = 0;
  VCT_CUDA(c, cudaMemcpyAsync(&ov, &c->d_counters->overflow, 4, cudaMemcpyDeviceToHost, c->stream));
  VCT_CUDA(c, cudaStreamSynchronize(c->stream));
  if (c->d_counters_vis) {
    VCT_CUDA(c, cudaStreamSynchronize(c->stream_vox));
    VCT_CUDA(c, cudaStreamSynchronize(c->stream2));
    VCT_CUDA(c, cudaMemcpy(&ov2, &c->d_counters_vis->overflow, 4, cudaMemcpyDeviceToHost));
  }
  if (ov || ov2) {
    cudaMemsetAsync(&c->d_counters->overflow, 0, 4, c->stream);
    if (c->d_counters_vis) cudaMemset(&c->d_counters_vis->overflow, 0, 4);
    return set_error(c, VCT_ERR_OVERFLOW, "device work queue overflow: raise MaxFragments / MaxTileItems (or MaxExchangeVoxels for vct_voxelize_shared)");
  }
  return VCT_OK;
}

// ---- material textures: glTexImage2D + glGenerateMipmap(GL_TEXTURE_2D), Model.h:159-175
__global__ void expand_rgba(const uint8_t* __restrict__ src, uchar4* __restrict__ dst, size_t n, int ch,
                            unsigned int* has_alpha) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uchar4 o;
  o.x = src[i * ch];
  o.y = ch >= 3 ? src[i * ch + 1] : 0;     // GL_RED samples (r,0,0,1); GL_RGB samples alpha 1
  o.z = ch >= 3 ? src[i * ch + 2] : 0;
  o.w = ch == 4 ? src[i * ch + 3] : 255;
  dst[i] = o;
  if (o.w != 255) *has_alpha = 1u;
}

__global__ void mip2d(const uchar4* __restrict__ src, int pw, int ph, uchar4* __restrict__ dst, int nw, int nh) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= nw || y >= nh) return;
  int x0 = min(2 * x, pw - 1), x1 = min(2 * x + 1, pw - 1), y0 = min(2 * y, ph - 1), y1 = min(2 * y + 1, ph - 1);
  uchar4 a = src[(size_t)y0 * pw + x0], b = src[(size_t)y0 * pw + x1], c = src[(size_t)y1 * pw + x0], d = src[(size_t)y1 * pw + x1];
  uchar4 o;
  o.x = (unsigned char)((a.x + b.x + c.x + d.x + 2) >> 2);
  o.y = (unsigned char)((a.y + b.y + c.y + d.y + 2) >> 2);
  o.z = (unsigned char)((a.z + b.z + c.z + d.z + 2) >> 2);
  o.w = (unsigned char)((a.w + b.w + c.w + d.w + 2) >> 2);
  dst[(size_t)y * nw + x] = o;
}

static void free_texture(TextureEntry& t) {
  if (t.tex) cudaDestroyTextureObject(t.tex);
  if (t.array) cudaFreeMipmappedArray(t.array);
  t = TextureEntry();
}

static int make_texture(vct_context* c, TextureEntry& out, int w, int h, int ch, const uint8_t* pixels) {
  int levels = 1;
  for (int a = w, b = h; a > 1 || b > 1; a = a > 1 ? a / 2 : 1, b = b > 1 ? b / 2 : 1) ++levels;
  const size_t n = (size_t)w * h;
  uint8_t* d_src = nullptr; uchar4 *d_a = nullptr, *d_b = nullptr; unsigned int* d_flag = nullptr;
  VCT_CUDA(c, cudaMalloc(&d_src, n * ch));
  VCT_CUDA(c, cudaMalloc(&d_a, n * 4));
  VCT_CUDA(c, cudaMalloc(&d_b, (n / 2 + 4) * 4));
  VCT_CUDA(c, cudaMalloc(&d_flag, 4));
  VCT_CUDA(c, cudaMemsetAsync(d_flag, 0, 4, c->stream));
  VCT_CUDA(c, cudaMemcpyAsync(d_src, pixels, n * ch, cudaMemcpyHostToDevice, c->stream));
  expand_rgba<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(d_src, d_a, n, ch, d_flag);
  cudaChannelFormatDesc desc = cudaCreateChannelDesc<uchar4>();
  VCT_CUDA(c, cudaMallocMipmappedArray(&out.array, &desc, make_cudaExtent(w, h, 0), levels));
  int pw = w, ph = h;
  uchar4 *cur = d_a, *nxt = d_b;
  for (int l = 0; l < levels; ++l) {
    cudaArray_t lvl;
    VCT_CUDA(c, cudaGetMipmappedArrayLevel(&lvl, out.array, l));
    VCT_CUDA(c, cudaMemcpy2DToArrayAsync(lvl, 0, 0, cur, (size_t)pw * 4, (size_t)pw * 4, ph, cudaMemcpyDeviceToDevice, c->stream));
    if (l + 1 < levels) {
      int nw = pw > 1 ? pw / 2 : 1, nh = ph > 1 ? ph / 2 : 1;
      dim3 b(16, 16), g((nw + 15) / 16, (nh + 15) / 16);
      mip2d<<<g, b, 0, c->stream>>>(cur, pw, ph, nxt, nw, nh);
      uchar4* t = cur; cur = nxt; nxt = t;
      pw = nw; ph = nh;
    }
  }
  c->launches += levels;
  unsigned int flag = 0;
  VCT_CUDA(c, cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, c->stream));
  VCT_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaFree(d_src); cudaFree(d_a); cudaFree(d_b); cudaFree(d_flag);
  // sampler state: REPEAT, MIN = LINEAR_MIPMAP_LINEAR, MAG = LINEAR (Model.h:172-175)
  cudaResourceDesc rd{};
  rd.resType = cudaResourceTypeMipmappedArray;
  rd.res.mipmap.mipmap = out.array;
  cudaTextureDesc td{};
  td.addressMode[0] = td.addressMode[1] = cudaAddressModeWrap;
  td.filterMode = cudaFilterModeLinear;
  td.mipmapFilterMode = cudaFilterModeLinear;
  td.readMode = cudaReadModeNormalizedFloat;
  td.normalizedCoords = 1;
  td.maxMipmapLevelClamp = (float)(levels - 1);
  VCT_CUDA(c, cudaCreateTextureObject(&out.tex, &rd, &td, nullptr));
  out.w = w; out.h = h; out.has_alpha = flag != 0;
  return VCT_OK;
}

int sync_materials(vct_context* c) {
  if (!c->materials_dirty && c->d_materials) return VCT_OK;
  if (!c->white_tex) {
    TextureEntry t;
    const uint8_t white[4] = {255, 255, 255, 255};
    int rc = make_texture(c, t, 1, 1, 4, white); if (rc) return rc;
    c->white_tex = t.tex; c->white_arr = t.array;
  }
  size_t n = c->materials.size();
  if (n == 0) { c->materials.resize(1); n = 1; }
  std::vector<MaterialDev> host(n);
  for (size_t i = 0; i < n; ++i) {
    const MaterialHost& m = c->materials[i];
    auto pick = [&](int id, cudaTextureObject_t& t, int& w, int& h, bool* alpha) {
      if (id >= 0 && id < (int)c->textures.size() && c->textures[id].tex) {
        t = c->textures[id].tex; w = c->textures[id].w; h = c->textures[id].h;
        if (alpha) *alpha = c->textures[id].has_alpha;
      } else { t = c->white_tex; w = 1; h = 1; if (alpha) *alpha = false; }
    };
    bool alpha = false;
    pick(m.d, host[i].diffuse, host[i].dw, host[i].dh, &alpha);
    pick(m.s, host[i].specular, host[i].sw, host[i].sh, nullptr);
    pick(m.h, host[i].height, host[i].hw, host[i].hh, nullptr);
    host[i].shininess = m.shininess;
    host[i].alpha_test = alpha ? 1 : 0;
  }
  if (c->d_materials) { int rc = sync_all_streams(c); if (rc) return rc; }   // in-flight kernels read the table
  if (c->n_materials_dev < n) {
    cudaFree(c->d_materials); c->d_materials = nullptr;
    VCT_CUDA(c, cudaMalloc(&c->d_materials, n * sizeof(MaterialDev)));
    c->n_materials_dev = n;
  }
  VCT_CUDA(c, cudaMemcpyAsync(c->d_materials, host.data(), n * sizeof(MaterialDev), cudaMemcpyHostToDevice, c->stream));
  VCT_CUDA(c, cudaStreamSynchronize(c->stream));   // `host` goes out of scope
  c->materials_dirty = false;
  return VCT_OK;
}

// ---- vertex pass
__global__ void vertex_pass(Params P, const float* __restrict__ verts, size_t nv, VertexCache vc) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nv) return;
  const float* v = verts + i * 14;
  const float px = v[0], py = v[1], pz = v[2];
  F4 w = mul_mat_vec(P.model, px, py, pz, 1.0f);                         // Voxelization.vs:21, VoxelConeTracing.vs:27
  vc.world[i] = make_float4(w.x, w.y, w.z, w.w);
  F4 d = mul_mat_vec(P.depth_mvp, px, py, pz, 1.0f);                     // Voxelization.vs:18-19, VoxelConeTracing.vs:28-29
  vc.dc[i] = make_float4(d.x * 0.5f + 0.5f, d.y * 0.5f + 0.5f, d.z * 0.5f + 0.5f, d.w);
  F4 e = mul_mat_vec(P.model_view, px, py, pz, 1.0f);                    // VoxelConeTracing.vs:25
  F4 c = mul_mat_vec(P.proj, e.x, e.y, e.z, e.w);
  const bool finite = isfinite(c.x) && isfinite(c.y) && isfinite(c.z) && isfinite(c.w);
  vc.clip[i] = make_float4((c.x + c.w) * (0.5f * (float)P.W), (c.y + c.w) * (0.5f * (float)P.H),
                           finite ? c.w : __int_as_float(0x7fc00000), c.z);
  F4 n = mul_mat_vec(P.model, v[3], v[4], v[5], 0.0f);                   // VoxelConeTracing.vs:31-33
  F4 t = mul_mat_vec(P.model, v[8], v[9], v[10], 0.0f);
  F4 b = mul_mat_vec(P.model, v[11], v[12], v[13], 0.0f);
  vc.nrm_u[i] = make_float4(n.x, n.y, n.z, v[6]);
  vc.tan_v[i] = make_float4(t.x, t.y, t.z, v[7]);
  vc.bit[i] = make_float4(b.x, b.y, b.z, 0.0f);
}

static void free_vertex_cache(vct_context* c) {
  for (int k = 0; k < 2; ++k) {
    VertexCache& vc = c->vcache2[k];
    cudaFree(vc.world); cudaFree(vc.dc); cudaFree(vc.clip); cudaFree(vc.nrm_u); cudaFree(vc.tan_v); cudaFree(vc.bit);
    vc = VertexCache{}; c->vcache_nv[k] = 0; c->vcache_valid[k] = false;
  }
}

// (re)computes the vertex cache of the CURRENT slot if the mesh or any matrix it depends on changed
int ensure_vertex_cache(vct_context* c) {
  if (!c->nv) return set_error(c, VCT_ERR_STATE, "no mesh uploaded");
  const int k = c->cur;
  VertexCache& vc = c->vcache2[k];
  if (c->vcache_nv[k] != c->nv) {
    cudaStreamSynchronize(c->stream);
    float4** arr[] = {&vc.world, &vc.dc, &vc.clip, &vc.nrm_u, &vc.tan_v, &vc.bit};
    for (float4** a : arr) { cudaFree(*a); *a = nullptr; VCT_CUDA(c, cudaMalloc(a, c->nv * sizeof(float4))); }
    c->vcache_nv[k] = c->nv;
    c->vcache_valid[k] = false;
  }
  const Params& P = c->P; const Params& Q = c->vcache_params[k];
  const bool same = c->vcache_valid[k] && P.W == Q.W && P.H == Q.H && !std::memcmp(P.model, Q.model, sizeof(P.model)) &&
                    !std::memcmp(P.model_view, Q.model_view, sizeof(P.model_view)) && !std::memcmp(P.proj, Q.proj, sizeof(P.proj)) &&
                    !std::memcmp(P.depth_mvp, Q.depth_mvp, sizeof(P.depth_mvp));
  if (same) return VCT_OK;
  vertex_pass<<<(unsigned)((c->nv + 127) / 128), 128, 0, c->stream>>>(c->P, c->d_verts, c->nv, vc);
  c->launches += 1;
  c->vcache_params[k] = c->P;
  c->vcache_valid[k] = true;
  return check_cuda(c, cudaGetLastError(), "vertex_pass");
}

void next_event_generation(vct_context* c) {
  c->ev_gen = (c->ev_gen + 1) % VCT_EVENT_GENS;
  for (int p = 0; p < VCT_PASS_COUNT; ++p)
    if (p != VCT_PASS_DEPTH) c->ev_recorded[c->ev_gen][p] = false;
}

// ---- frame slots
void mark_slot_read(vct_context* c) {
  if (!c->slot_read_done[0]) {
    cudaEventCreateWithFlags(&c->slot_read_done[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->slot_read_done[1], cudaEventDisableTiming);
  }
  cudaEventRecord(c->slot_read_done[c->cur], c->stream);
  c->slot_read_pending[c->cur] = true;
}

// Switch to the other slot.  Whatever stream c->stream currently is (main, or the voxel stream inside a pipelined
// vct_frame) first waits for the last reader of that slot.
int begin_voxel_slot(vct_context* c) {
  const int nxt = c->cur ^ 1;
  if (c->slot_read_pending[nxt]) {
    VCT_CUDA(c, cudaStreamWaitEvent(c->stream, c->slot_read_done[nxt], 0));
  }
  c->cur = nxt;
  return VCT_OK;
}

// ---- queries on the pyramid
// The pyramid of a query that reads levels 0..top: allocated, and its levels above 0 built from level 0 if it reads any.
static int need_pyramid(vct_context* c, const char* what, int top) {
  int rc = ensure_grid(c); if (rc) return rc;
  if (top > 0 && !c->grid[c->cur].mips_current)
    return set_error(c, VCT_ERR_STATE, std::string(what) + ": the mip levels are stale (call vct_build_mips after vct_upload_grid_level0)");
  return VCT_OK;
}

// One host array of a call: `in` is copied to the device before the launch, `out` back after it.  Neither: the array
// is absent.
struct HostArray { const void* in; void* out; size_t bytes; };

// The host form of a device call.  Lays out the arrays in c->d_stage (grown on demand), each present one in its own
// 256-byte-aligned region, copies the inputs there on c->stream, runs launch(d) with d[k] the device pointer of a[k]
// (NULL for an absent array), copies the outputs back and synchronises c->stream once, error paths included, so that
// the buffer is free for the next call when this returns.  Returns the launch's own error code if it failed, else the
// first copy error, else the synchronise's.
template <size_t N, class Launch>
static int host_round_trip(vct_context* c, const char* what, const HostArray (&a)[N], Launch launch) {
  auto up256 = [](size_t b) { return (b + 255) & ~(size_t)255; };
  size_t bytes = 0;
  for (const HostArray& x : a) if (x.in || x.out) bytes += up256(x.bytes);
  if (c->stage_bytes < bytes) {
    cudaFree(c->d_stage);
    c->d_stage = nullptr; c->stage_bytes = 0;
    VCT_CUDA(c, cudaMalloc(&c->d_stage, bytes));
    c->stage_bytes = bytes;
  }
  void* d[N];
  unsigned char* p = c->d_stage;
  for (size_t k = 0; k < N; ++k) {
    d[k] = a[k].in || a[k].out ? p : nullptr;
    if (d[k]) p += up256(a[k].bytes);
  }
  cudaError_t e = cudaSuccess;
  for (size_t k = 0; k < N; ++k)
    if (a[k].in && e == cudaSuccess) e = cudaMemcpyAsync(d[k], a[k].in, a[k].bytes, cudaMemcpyHostToDevice, c->stream);
  const int rc = e == cudaSuccess ? launch(d) : VCT_OK;
  for (size_t k = 0; k < N; ++k)
    if (!rc && a[k].out && e == cudaSuccess) e = cudaMemcpyAsync(a[k].out, d[k], a[k].bytes, cudaMemcpyDeviceToHost, c->stream);
  const cudaError_t es = cudaStreamSynchronize(c->stream);
  if (rc) return rc;
  return check_cuda(c, e != cudaSuccess ? e : es, what);
}

// ------------------------------------------------------------------------------------------ tex bench
__global__ void fill_level_random(cudaSurfaceObject_t s, int n, unsigned seed, int f16) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
  if (x >= n || y >= n) return;
  unsigned h = (unsigned)(x * 73856093) ^ (unsigned)(y * 19349663) ^ (unsigned)(z * 83492791) ^ seed;
  h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
  if (f16) surf3Dwrite(make_uint2(h & 0x3BFF3BFFu, (h >> 3) & 0x3BFF3BFFu), s, x * 8, y, z);   // four finite halves in [0, 1)
  else surf3Dwrite(h, s, x * 4, y, z);
}

// Atomics micro-benchmark (roofline denominator of vox_shade's accumulation): the same two 64-bit atomicAdds per
// fragment, on the voxel population of the last voxelisation (touched list), `mult` consecutive fragments per voxel --
// the measured mean multiplicity -- so that the warp-level and L2-level collision profile resembles the real pass.
__global__ void __launch_bounds__(256) atomics_bench(unsigned long long* __restrict__ accum, const uint32_t* __restrict__ touched,
                                                     uint32_t n_touched, uint32_t n_frag, uint32_t mult) {
  for (uint32_t f = blockIdx.x * blockDim.x + threadIdx.x; f < n_frag; f += gridDim.x * blockDim.x) {
    const uint32_t v = touched[(f / mult) % n_touched];
    atomicAdd(&accum[2 * (size_t)v], 0x0000000100000001ull);
    atomicAdd(&accum[2 * (size_t)v + 1], 0x0000000100000001ull);
  }
}

// each thread marches `steps` samples; a warp covers an 8x4 patch of start points (as cone_trace does)
__global__ void __launch_bounds__(256) tex3d_bench(cudaTextureObject_t tex, int steps, float lod, int pattern,
                                                   float step_len, float4* sink, int W) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + (warp & 3) * 8 + (lane & 7);
  const int j = blockIdx.y * 8 + (warp >> 2) * 4 + (lane >> 3);
  float u = (i + 0.5f) / (float)W, v = (j + 0.5f) / (float)W, w = 0.37f;
  float du = 0.57f * step_len, dv = 0.31f * step_len, dw = 0.76f * step_len;
  unsigned rng = (unsigned)(i * 9781 + j * 6271) | 1u;
  float4 acc = make_float4(0, 0, 0, 0);
  for (int s = 0; s < steps; ++s) {
    if (pattern == 1) {
      rng ^= rng << 13; rng ^= rng >> 17; rng ^= rng << 5;
      u = (rng & 0xFFFF) * (1.0f / 65536.0f); v = ((rng >> 8) & 0xFFFF) * (1.0f / 65536.0f); w = (rng >> 16) * (1.0f / 65536.0f);
    } else { u += du; v += dv; w += dw; }
    float4 t = tex3DLod<float4>(tex, u, v, w, lod);
    acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
  }
  if (acc.x == -1.0f) sink[0] = acc;   // never true: keeps the loop alive
}

}  // namespace vct

using namespace vct;

// =========================================================================================== C ABI
extern "C" {

const char* vct_version(void) { return "vct_b200 0.1 (sm_100a)"; }

int vct_create(int device, vct_handle* out) {
  if (!out) return VCT_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    return set_error(nullptr, VCT_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") +
                                                (e == cudaSuccess ? "device count 0" : cudaGetErrorString(e)));
  if (device < 0 || device >= n) return set_error(nullptr, VCT_ERR_INVALID, "bad device index");
  vct_context* c = new vct_context();
  c->device = device;
  default_params(c->P);
  c->materials.resize(1);
  auto fail = [&](int rc) { g_create_error = c->err; delete c; return rc; };
  if (int rc = check_cuda(c, cudaSetDevice(device), "cudaSetDevice")) return fail(rc);
  if (int rc = check_cuda(c, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking), "cudaStreamCreate")) return fail(rc);
  for (int p = 0; p < VCT_PASS_COUNT; ++p) {
    for (int g = 0; g < VCT_EVENT_GENS; ++g) { cudaEventCreate(&c->ev_begin[g][p]); cudaEventCreate(&c->ev_end[g][p]); }
  }
  if (int rc = check_cuda(c, cudaMalloc(&c->d_counters, sizeof(Counters)), "cudaMalloc counters")) return fail(rc);
  cudaMemset(c->d_counters, 0, sizeof(Counters));
  *out = c;
  return VCT_OK;
}

int vct_destroy(vct_handle c) {
  if (!c) return VCT_ERR_INVALID;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  comm_release_for_destroy(c);
  free_grid(c);
  free_vertex_cache(c);
  for (auto& t : c->textures) free_texture(t);
  if (c->white_tex) cudaDestroyTextureObject(c->white_tex);
  if (c->white_arr) cudaFreeMipmappedArray(c->white_arr);
  cudaFree(c->d_verts); cudaFree(c->d_idx); cudaFree(c->d_trimat); cudaFree(c->d_materials);
  if (c->depth_tex) cudaDestroyTextureObject(c->depth_tex);
  if (c->depth_surf) cudaDestroySurfaceObject(c->depth_surf);
  if (c->depth_array) cudaFreeArray(c->depth_array);
  cudaFree(c->mask_prev[0]); cudaFree(c->mask_prev[1]); cudaFree(c->d_push_list); cudaFree(c->d_push_count);
  cudaFree(c->d_voxrec); cudaFree(c->d_depth); cudaFree(c->d_frags); cudaFree(c->d_items); cudaFree(c->d_counters);
  cudaFree(c->d_vis2[0]); cudaFree(c->d_vis2[1]); cudaFree(c->d_frame);
  cudaFree(c->d_stage);
  for (int k = 0; k < 2; ++k) if (c->slot_read_done[k]) cudaEventDestroy(c->slot_read_done[k]);
  if (c->stream_vox) { cudaStreamDestroy(c->stream_vox); cudaEventDestroy(c->ev_vox_done); cudaEventDestroy(c->ev_vtx_done); }
  for (int k = 0; k < 3; ++k) { cudaFree(c->d_frame2[k]); if (c->ev_rendered[k]) cudaEventDestroy(c->ev_rendered[k]); if (c->ev_copied[k]) cudaEventDestroy(c->ev_copied[k]); }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->h_overflow) cudaFreeHost(c->h_overflow);
  if (c->stream2) { cudaStreamDestroy(c->stream2); cudaEventDestroy(c->ev_fork); cudaEventDestroy(c->ev_join); }
  cudaFree(c->d_items_vis); cudaFree(c->d_counters_vis);
  for (int p = 0; p < VCT_PASS_COUNT; ++p)
    for (int g = 0; g < VCT_EVENT_GENS; ++g) { cudaEventDestroy(c->ev_begin[g][p]); cudaEventDestroy(c->ev_end[g][p]); }
  if (c->ev_ref) cudaEventDestroy(c->ev_ref);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return VCT_OK;
}

const char* vct_last_error(vct_handle c) { return c ? c->err.c_str() : g_create_error.c_str(); }

#define NEED(c) do { if (!(c)) return VCT_ERR_INVALID; cudaSetDevice((c)->device); } while (0)

int vct_set_i(vct_handle c, const char* name, int v) {
  NEED(c);
  if (!name) return set_error(c, VCT_ERR_INVALID, "null uniform name");
  std::string k(name);
  Params& P = c->P;
  if (k == "VoxelDimensions") {
    if (v < 2 || v > 1024 || (v & (v - 1))) return set_error(c, VCT_ERR_INVALID, "VoxelDimensions must be a power of two in [2,1024]");
    P.V = v; P.levels = ilog2(v) + 1;
  } else if (k == "ShadowMapSize") {
    if (v < 1 || v > 16384) return set_error(c, VCT_ERR_INVALID, "ShadowMapSize out of range");
    if (v != P.S) c->depth_valid = false;
    P.S = v;
  } else if (k == "screen_width") { if (v < 1 || v > 16384) return set_error(c, VCT_ERR_INVALID, "screen_width out of range"); P.W = v; }
  else if (k == "screen_height") { if (v < 1 || v > 16384) return set_error(c, VCT_ERR_INVALID, "screen_height out of range"); P.H = v; }
  else if (k == "PcfRadius") { if (v < 0 || v > 8) return set_error(c, VCT_ERR_INVALID, "PcfRadius out of range"); P.pcf_radius = v; }
  else if (k == "CoveragePolicy") { if (v < 0 || v > 2) return set_error(c, VCT_ERR_INVALID, "CoveragePolicy must be 0,1,2"); P.coverage = v; }
  else if (k == "Bounces") { if (v < 1 || v > 8) return set_error(c, VCT_ERR_INVALID, "Bounces out of range"); P.bounces = v; }
  else if (k == "NumDiffuseCones") { if (v < 0 || v > VCT_MAX_CONES) return set_error(c, VCT_ERR_INVALID, "NumDiffuseCones out of range"); P.n_cones = v; }
  else if (k == "GridFormat") { if (v != 0 && v != 1) return set_error(c, VCT_ERR_INVALID, "GridFormat: 0 = RGBA8, 1 = RGBA16F"); if (v != c->grid_format) c->scene_epoch++; c->grid_format = v; }
  else if (k == "MaxFragments") { if (v < 1024) return set_error(c, VCT_ERR_INVALID, "MaxFragments too small"); c->max_fragments = (size_t)v; }
  else if (k == "MaxTileItems") { if (v < 1024) return set_error(c, VCT_ERR_INVALID, "MaxTileItems too small"); c->max_items = (size_t)v; }
  else if (k == "RowBegin") { if (v < 0) return set_error(c, VCT_ERR_INVALID, "RowBegin < 0"); P.row_begin = v; }
  else if (k == "RowEnd") { if (v < 0) return set_error(c, VCT_ERR_INVALID, "RowEnd < 0"); P.row_end = v; }
  else if (k == "RowInterleave") { if (v < 0 || v > 64) return set_error(c, VCT_ERR_INVALID, "RowInterleave out of range"); P.row_il = v; }
  else if (k == "RowPhase") { if (v < 0 || v > 63) return set_error(c, VCT_ERR_INVALID, "RowPhase out of range"); P.row_ph = v; }
  else if (k == "OverlapVisibility") c->overlap_visibility = v != 0;
  else if (k == "SharedExchange") { if (v != 0 && v != 1) return set_error(c, VCT_ERR_INVALID, "SharedExchange: 0 inbox, 1 in-switch reduction"); c->shared_exchange = v; }
  else if (k == "TriangleInterleave") { if (v < 1) return set_error(c, VCT_ERR_INVALID, "TriangleInterleave < 1"); c->tri_interleave = v; c->scene_epoch++; }
  else if (k == "TrianglePhase") { if (v < 0) return set_error(c, VCT_ERR_INVALID, "TrianglePhase < 0"); c->tri_phase = v; c->scene_epoch++; }
  else if (k == "SharedWorld") { if (v < 1 || v > 16) return set_error(c, VCT_ERR_INVALID, "SharedWorld out of range"); c->shared_world = v; }
  else if (k == "SharedRank") { if (v < 0 || v > 15) return set_error(c, VCT_ERR_INVALID, "SharedRank out of range"); c->shared_rank = v; }
  else if (k == "MaxExchangeVoxels") { if (v < 1024) return set_error(c, VCT_ERR_INVALID, "MaxExchangeVoxels too small"); c->exchange_cap_user = (size_t)v; }
  else if (k == "PipelineFrames") c->pipeline_frames = v != 0;
  else if (k == "DenseResolve") c->dense_resolve = v != 0;
  else if (k == "ShardShadowMap") { c->shard_shadow = v != 0; c->depth_valid = false; c->scene_epoch++; }
  else if (k == "Profile") {
    c->profile = v != 0;
    if (c->profile) {                       // time zero of vct_pass_timeline
      if (!c->ev_ref) cudaEventCreate(&c->ev_ref);
      cudaEventRecord(c->ev_ref, c->stream);
      for (auto& gen : c->ev_recorded) for (bool& r : gen) r = false;
    }
  }
  else if (k == "ShadowMap" || k == "VoxelTexture") { /* texture unit numbers: meaningless here */ }
  else return set_error(c, VCT_ERR_INVALID, "unknown int uniform '" + k + "'");
  return VCT_OK;
}

int vct_get_i(vct_handle c, const char* name, int* v) {
  NEED(c);
  if (!name || !v) return VCT_ERR_INVALID;
  std::string k(name);
  const Params& P = c->P;
  if (k == "VoxelDimensions") *v = P.V; else if (k == "ShadowMapSize") *v = P.S;
  else if (k == "screen_width") *v = P.W; else if (k == "screen_height") *v = P.H;
  else if (k == "PcfRadius") *v = P.pcf_radius; else if (k == "CoveragePolicy") *v = P.coverage;
  else if (k == "Bounces") *v = P.bounces; else if (k == "NumDiffuseCones") *v = P.n_cones;
  else if (k == "GridFormat") *v = c->grid_format; else if (k == "MipLevels") *v = P.levels;
  else if (k == "MaxFragments") *v = (int)c->max_fragments; else if (k == "MaxTileItems") *v = (int)c->max_items;
  else if (k == "RowBegin") *v = P.row_begin; else if (k == "RowEnd") *v = P.row_end;
  else if (k == "RowInterleave") *v = P.row_il; else if (k == "RowPhase") *v = P.row_ph;
  else if (k == "DenseResolve") *v = c->dense_resolve; else if (k == "Profile") *v = c->profile;
  else if (k == "ShardShadowMap") *v = c->shard_shadow;
  else return set_error(c, VCT_ERR_INVALID, "unknown int uniform '" + k + "'");
  return VCT_OK;
}

static float* float_slot(Params& P, const std::string& k) {
  if (k == "VoxelGridWorldSize") return &P.grid_world;
  if (k == "ambientFactor") return &P.ambient;
  if (k == "DiffuseTanHalfAngle") return &P.diffuse_tan;
  if (k == "SpecularTanHalfAngle") return &P.spec_tan;
  if (k == "StepMultiplier") return &P.step_mult;
  if (k == "MaxDistance") return &P.max_dist;
  if (k == "MaxAlpha") return &P.max_alpha;
  if (k == "ShadowBias") return &P.shadow_bias;
  return nullptr;
}

int vct_set_f(vct_handle c, const char* name, float v) {
  NEED(c);
  if (!name) return VCT_ERR_INVALID;
  float* s = float_slot(c->P, name);
  if (!s) return set_error(c, VCT_ERR_INVALID, std::string("unknown float uniform '") + name + "'");
  if (!(v == v)) return set_error(c, VCT_ERR_INVALID, "NaN uniform");
  if (std::string(name) == "StepMultiplier" && !(v > 0.0f)) return set_error(c, VCT_ERR_INVALID, "StepMultiplier must be > 0");
  if (std::string(name) == "VoxelGridWorldSize" && !(v > 0.0f)) return set_error(c, VCT_ERR_INVALID, "VoxelGridWorldSize must be > 0");
  *s = v;
  return VCT_OK;
}

int vct_get_f(vct_handle c, const char* name, float* v) {
  NEED(c);
  if (!name || !v) return VCT_ERR_INVALID;
  float* s = float_slot(c->P, name);
  if (!s) return set_error(c, VCT_ERR_INVALID, std::string("unknown float uniform '") + name + "'");
  *v = *s;
  return VCT_OK;
}

int vct_set_3f(vct_handle c, const char* name, float x, float y, float z) {
  NEED(c);
  if (!name) return VCT_ERR_INVALID;
  std::string k(name);
  float* d = k == "CameraPosition" ? c->P.cam : k == "LightDirection" ? c->P.light : nullptr;
  if (!d) return set_error(c, VCT_ERR_INVALID, "unknown vec3 uniform '" + k + "'");
  d[0] = x; d[1] = y; d[2] = z;
  return VCT_OK;
}

int vct_set_mat4(vct_handle c, const char* name, const float* m) {
  NEED(c);
  if (!name || !m) return VCT_ERR_INVALID;
  std::string k(name);
  Params& P = c->P;
  float* d = k == "ModelMatrix" ? P.model : k == "ModelViewMatrix" ? P.model_view : k == "ProjectionMatrix" ? P.proj
           : k == "DepthModelViewProjectionMatrix" ? P.depth_mvp : k == "ProjX" ? P.projx : k == "ProjY" ? P.projy
           : k == "ProjZ" ? P.projz : nullptr;
  if (!d) return set_error(c, VCT_ERR_INVALID, "unknown mat4 uniform '" + k + "'");
  std::memcpy(d, m, 16 * sizeof(float));
  return VCT_OK;
}

int vct_set_cones(vct_handle c, int n, const float* dirs, const float* w) {
  NEED(c);
  if (n < 0 || n > VCT_MAX_CONES || (n && (!dirs || !w))) return set_error(c, VCT_ERR_INVALID, "vct_set_cones: bad arguments");
  c->P.n_cones = n;
  std::memcpy(c->P.cone_dir, dirs, (size_t)n * 3 * sizeof(float));
  std::memcpy(c->P.cone_w, w, (size_t)n * sizeof(float));
  return VCT_OK;
}

int vct_upload_texture(vct_handle c, int id, int w, int h, int ch, const uint8_t* px) {
  NEED(c);
  if (id < 0 || id > 65535 || w < 1 || h < 1 || w > 32768 || h > 32768 || (ch != 1 && ch != 3 && ch != 4) || !px)
    return set_error(c, VCT_ERR_INVALID, "vct_upload_texture: bad arguments");
  if ((int)c->textures.size() <= id) c->textures.resize(id + 1);
  // frames queued by vct_frame(NULL) / vct_frame_async / vct_frame_shared_begin may still sample the old texture
  if (c->textures[id].tex) { int rc = sync_all_streams(c); if (rc) return rc; }
  free_texture(c->textures[id]);
  c->materials_dirty = true;
  c->scene_epoch++;
  return make_texture(c, c->textures[id], w, h, ch, px);
}

int vct_set_material(vct_handle c, int mat, int d, int s, int h, float shininess) {
  NEED(c);
  if (mat < 0 || mat > 65535) return set_error(c, VCT_ERR_INVALID, "vct_set_material: bad material id");
  if ((int)c->materials.size() <= mat) c->materials.resize(mat + 1);
  c->materials[mat].d = d; c->materials[mat].s = s; c->materials[mat].h = h; c->materials[mat].shininess = shininess;
  c->materials_dirty = true;
  c->scene_epoch++;
  return VCT_OK;
}

int vct_upload_mesh(vct_handle c, const float* verts, size_t nv, const uint32_t* idx, size_t nt, const uint16_t* tm) {
  NEED(c);
  if (!verts || !idx || nv == 0 || nt == 0 || nt > 0x7FFFFFFFull / 3) return set_error(c, VCT_ERR_INVALID, "vct_upload_mesh: bad arguments");
  uint16_t max_mat = 0;
  for (size_t i = 0; i < nt * 3; ++i)
    if (idx[i] >= nv) return set_error(c, VCT_ERR_INVALID, "vct_upload_mesh: index out of range");
  if (tm) for (size_t i = 0; i < nt; ++i) max_mat = tm[i] > max_mat ? tm[i] : max_mat;
  if (c->d_verts) { int rc = sync_all_streams(c); if (rc) return rc; }
  cudaFree(c->d_verts); cudaFree(c->d_idx); cudaFree(c->d_trimat);
  c->d_verts = nullptr; c->d_idx = nullptr; c->d_trimat = nullptr; c->nv = c->nt = 0;
  VCT_CUDA(c, cudaMalloc(&c->d_verts, nv * 14 * sizeof(float)));
  VCT_CUDA(c, cudaMalloc(&c->d_idx, nt * 3 * sizeof(uint32_t)));
  VCT_CUDA(c, cudaMemcpyAsync(c->d_verts, verts, nv * 14 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  VCT_CUDA(c, cudaMemcpyAsync(c->d_idx, idx, nt * 3 * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  if (tm) {
    VCT_CUDA(c, cudaMalloc(&c->d_trimat, nt * sizeof(uint16_t)));
    VCT_CUDA(c, cudaMemcpyAsync(c->d_trimat, tm, nt * sizeof(uint16_t), cudaMemcpyHostToDevice, c->stream));
    if (c->materials.size() <= max_mat) { c->materials.resize((size_t)max_mat + 1); c->materials_dirty = true; }
  }
  VCT_CUDA(c, cudaStreamSynchronize(c->stream));
  c->nv = nv; c->nt = nt;
  c->depth_valid = false;
  c->vcache_valid[0] = c->vcache_valid[1] = false;
  c->scene_epoch++;
  return VCT_OK;
}

__global__ void scatter_positions(const float* __restrict__ xyz, float* __restrict__ verts, size_t nv) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nv) return;
  verts[i * 14 + 0] = xyz[i * 3 + 0];
  verts[i * 14 + 1] = xyz[i * 3 + 1];
  verts[i * 14 + 2] = xyz[i * 3 + 2];
}

int vct_update_positions(vct_handle c, const float* xyz, size_t nv, int on_device) {
  NEED(c);
  if (!xyz || nv != c->nv) return set_error(c, VCT_ERR_INVALID, "vct_update_positions: vertex count mismatch");
  auto scatter = [&](const float* src) {
    scatter_positions<<<(unsigned)((nv + 255) / 256), 256, 0, c->stream>>>(src, c->d_verts, nv);
    c->launches += 1;
    c->depth_valid = false;
    c->vcache_valid[0] = c->vcache_valid[1] = false;
    c->scene_epoch++;
    return check_cuda(c, cudaGetLastError(), "scatter_positions");
  };
  if (on_device) return scatter(xyz);
  return host_round_trip(c, "vct_update_positions", {{xyz, nullptr, nv * 12}},
                         [&](void* const* d) { return scatter((const float*)d[0]); });
}

// ---- passes
int vct_draw_depth(vct_handle c) { NEED(c); c->scene_epoch++; return launch_shadow(c); }

// clear + voxelise + resolve + mip (+ re-injection) into the current slot, on c->stream
static int draw_voxels_body(vct_context* c) {
  int rc = launch_voxel_clear(c); if (rc) return rc;
  rc = launch_voxelize(c, 0, c->nt); if (rc) return rc;
  rc = launch_resolve(c, c->dense_resolve != 0); if (rc) return rc;
  rc = launch_mip(c); if (rc) return rc;
  for (int b = 3; b <= c->P.bounces; ++b) {
    rc = launch_reinject(c); if (rc) return rc;
    rc = launch_mip(c); if (rc) return rc;
  }
  return VCT_OK;
}

int vct_draw_voxels(vct_handle c) {
  NEED(c);
  c->scene_epoch++;
  int rc = ensure_grid(c); if (rc) return rc;
  rc = begin_voxel_slot(c); if (rc) return rc;    // build into the slot no cone_trace is reading
  return draw_voxels_body(c);
}

int vct_voxelize_range(vct_handle c, size_t tb, size_t te, int clear_first) {
  NEED(c);
  int rc = ensure_grid(c); if (rc) return rc;
  c->scene_epoch++;
  if (clear_first) {
    // dense path: after an all-reduce the accumulator holds other ranks' voxels that no local list describes
    rc = begin_voxel_slot(c); if (rc) return rc;
    c->accum_list_slot = -1;
    rc = launch_voxel_clear(c); if (rc) return rc;
  }
  rc = launch_voxelize(c, tb, te);
  c->accum_list_slot = -1;
  return rc;
}

static size_t exchange_capacity(const vct_context* c) {
  const size_t n = (size_t)c->P.V * c->P.V * c->P.V;
  const size_t cap = c->exchange_cap_user ? c->exchange_cap_user : 32 * (size_t)c->P.V * c->P.V;
  return cap < n ? cap : n;
}

int vct_shared_accum_bytes(vct_handle c, size_t* bytes) {
  NEED(c);
  const size_t n = (size_t)c->P.V * c->P.V * c->P.V;
  c->exchange_cap = exchange_capacity(c);
  if (bytes) *bytes = c->shared_exchange == 1 ? n * 16 + n / 8
                                              : 4096 + 2 * (size_t)c->shared_world * c->exchange_cap * 16;
  return VCT_OK;
}

int vct_set_shared_accum(vct_handle c, void* local_ptr, void* multicast_ptr) {
  NEED(c);
  if (c->shared_frame_open) return set_error(c, VCT_ERR_STATE, "vct_set_shared_accum: a shared frame is open (call vct_frame_shared_end first)");
  if (c->comm) return set_error(c, VCT_ERR_STATE, "vct_set_shared_accum: the exchange buffer belongs to vct_comm_init (call vct_comm_destroy first)");
  if (c->shared_local) { int rc = sync_all_streams(c); if (rc) return rc; }   // queued exchange kernels use the old buffer
  c->shared_peers = nullptr; c->shared_seg = 0;
  c->shared_local = (unsigned long long*)local_ptr;
  c->shared_mc = (unsigned long long*)multicast_ptr;
  c->exchange_parity = 0;
  c->exchange_cap = exchange_capacity(c);   // the size vct_shared_accum_bytes reported for the current settings
  c->scene_epoch++;
  return VCT_OK;
}

int vct_voxelize_shared(vct_handle c, size_t tb, size_t te) {
  NEED(c);
  c->scene_epoch++;
  int rc = ensure_grid(c); if (rc) return rc;
  return launch_voxelize_shared(c, tb, te);
}

int vct_resolve_shared(vct_handle c) {
  NEED(c);
  c->scene_epoch++;
  int rc = launch_resolve_shared(c); if (rc) return rc;
  rc = launch_mip(c); if (rc) return rc;
  for (int b = 3; b <= c->P.bounces; ++b) {
    rc = launch_reinject(c); if (rc) return rc;
    rc = launch_mip(c); if (rc) return rc;
  }
  return VCT_OK;
}

static int ensure_overlap(vct_context* c);

// Pipelined form of one sharded frame (inbox flavour).  begin: the rank's triangle share is voxelised and multicast on
// the library's voxel stream, primary visibility runs on the visibility stream; the HOST then enqueues its cross-rank
// barrier on vct_exchange_stream; end: merge + resolve + mip on the voxel stream, cone_trace on the main stream after
// both.  As in vct_frame, with PipelineFrames the voxel/visibility stages of frame i+1 run beside cone_trace of frame i.
int vct_frame_shared_begin(vct_handle c, size_t tb, size_t te) {
  NEED(c);
  if (!c->shared_local) return set_error(c, VCT_ERR_STATE, "vct_frame_shared_begin: call vct_set_shared_accum first");
  if (c->shared_exchange != 0) return set_error(c, VCT_ERR_STATE, "vct_frame_shared_begin: needs SharedExchange = 0 (inbox)");
  if (c->shared_frame_open) return set_error(c, VCT_ERR_STATE, "vct_frame_shared_begin: previous frame not ended");
  int rc = ensure_grid(c); if (rc) return rc;
  rc = ensure_frame(c); if (rc) return rc;
  rc = ensure_queues(c); if (rc) return rc;
  rc = sync_materials(c); if (rc) return rc;
  rc = ensure_overlap(c); if (rc) return rc;
  const bool ordered = !c->pipeline_frames || c->scene_epoch != c->frame_epoch;
  next_event_generation(c);
  cudaStream_t main_stream = c->stream; TileItem* main_items = c->d_items; Counters* main_ctr = c->d_counters;
  if (ordered) VCT_CUDA(c, cudaEventRecord(c->ev_fork, main_stream));
  c->stream = c->stream_vox;
  rc = VCT_OK;
  if (ordered) rc = check_cuda(c, cudaStreamWaitEvent(c->stream_vox, c->ev_fork, 0), "wait fork");
  if (!rc) rc = begin_voxel_slot(c);
  if (!rc) rc = ensure_vertex_cache(c);
  if (!rc) rc = check_cuda(c, cudaEventRecord(c->ev_vtx_done, c->stream_vox), "record vtx");
  if (!rc) rc = launch_voxelize_inbox_into_slot(c, tb, te);
  if (!rc) {
    c->stream = c->stream2; c->d_items = c->d_items_vis; c->d_counters = c->d_counters_vis;
    rc = check_cuda(c, cudaStreamWaitEvent(c->stream2, c->ev_vtx_done, 0), "wait vtx");
    if (!rc) rc = launch_visibility(c);
    if (!rc) rc = check_cuda(c, cudaEventRecord(c->ev_join, c->stream2), "record join");
  }
  c->stream = main_stream; c->d_items = main_items; c->d_counters = main_ctr;
  if (rc) return rc;
  c->shared_frame_open = true;
  return VCT_OK;
}

int vct_exchange_stream(vct_handle c, void** cuda_stream) {
  NEED(c);
  int rc = ensure_overlap(c); if (rc) return rc;
  if (cuda_stream) *cuda_stream = (void*)c->stream_vox;
  return VCT_OK;
}

int vct_frame_shared_end(vct_handle c, uint8_t* host_rgba) {
  NEED(c);
  if (!c->shared_frame_open) return set_error(c, VCT_ERR_STATE, "vct_frame_shared_end: no frame begun");
  c->shared_frame_open = false;
  cudaStream_t main_stream = c->stream;
  c->stream = c->stream_vox;
  int rc = launch_resolve_shared(c);
  if (!rc) rc = launch_mip(c);
  for (int b = 3; !rc && b <= c->P.bounces; ++b) {
    rc = launch_reinject(c);
    if (!rc) rc = launch_mip(c);
  }
  if (!rc) rc = check_cuda(c, cudaEventRecord(c->ev_vox_done, c->stream_vox), "record vox");
  c->stream = main_stream;
  if (rc) return rc;
  VCT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_vox_done, 0));
  VCT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
  c->frame_epoch = c->scene_epoch;
  rc = launch_cone(c); if (rc) return rc;
  if (host_rgba) {
    VCT_CUDA(c, cudaMemcpyAsync(host_rgba, c->d_frame, (size_t)c->P.W * c->P.H * 4, cudaMemcpyDeviceToHost, c->stream));
    VCT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_overflow(c);       // a truncated queue must not pass for a frame (device-only paths: vct_sync)
  }
  return VCT_OK;
}

int vct_accum_buffer(vct_handle c, void** p, size_t* n) {
  NEED(c);
  int rc = ensure_grid(c); if (rc) return rc;
  if (p) *p = c->d_accum;
  if (n) *n = (size_t)c->P.V * c->P.V * c->P.V * 4;
  return VCT_OK;
}

int vct_resolve_and_mip(vct_handle c) {
  NEED(c);
  c->scene_epoch++;
  int rc = launch_resolve(c, true); if (rc) return rc;
  rc = launch_mip(c); if (rc) return rc;
  for (int b = 3; b <= c->P.bounces; ++b) {
    rc = launch_reinject(c); if (rc) return rc;
    rc = launch_mip(c); if (rc) return rc;
  }
  return VCT_OK;
}

int vct_render(vct_handle c, uint8_t* host_rgba) {
  NEED(c);
  c->scene_epoch++;
  int rc = launch_visibility(c); if (rc) return rc;
  rc = launch_cone(c); if (rc) return rc;
  if (host_rgba) {
    VCT_CUDA(c, cudaMemcpyAsync(host_rgba, c->d_frame, (size_t)c->P.W * c->P.H * 4, cudaMemcpyDeviceToHost, c->stream));
    VCT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_overflow(c);       // a truncated queue must not pass for a frame (device-only paths: vct_sync)
  }
  return VCT_OK;
}

// ---- voxel view
// C = A * B for column-major 4x4 matrices, double, glm's operator* order: column j = ((A0 b0j + A1 b1j) + A2 b2j) + A3 b3j
static void mat4_mul(const double* A, const double* B, double* C) {
  for (int j = 0; j < 4; ++j)
    for (int i = 0; i < 4; ++i)
      C[j * 4 + i] = ((A[0 * 4 + i] * B[j * 4 + 0] + A[1 * 4 + i] * B[j * 4 + 1]) + A[2 * 4 + i] * B[j * 4 + 2]) +
                     A[3 * 4 + i] * B[j * 4 + 3];
}

// glm::inverse(mat4) (glm/detail/func_matrix.inl, compute_inverse<4, 4>): cofactors, then times 1 / determinant.
// m[c][r] = column c, row r.  The CPU reference of the tests writes out the same operations in the same order (DESIGN.md section 3).
static void mat4_inverse_glm(const double* a, double* out) {
  auto m = [&](int c, int r) { return a[c * 4 + r]; };
  const double c00 = m(2, 2) * m(3, 3) - m(3, 2) * m(2, 3), c02 = m(1, 2) * m(3, 3) - m(3, 2) * m(1, 3), c03 = m(1, 2) * m(2, 3) - m(2, 2) * m(1, 3);
  const double c04 = m(2, 1) * m(3, 3) - m(3, 1) * m(2, 3), c06 = m(1, 1) * m(3, 3) - m(3, 1) * m(1, 3), c07 = m(1, 1) * m(2, 3) - m(2, 1) * m(1, 3);
  const double c08 = m(2, 1) * m(3, 2) - m(3, 1) * m(2, 2), c10 = m(1, 1) * m(3, 2) - m(3, 1) * m(1, 2), c11 = m(1, 1) * m(2, 2) - m(2, 1) * m(1, 2);
  const double c12 = m(2, 0) * m(3, 3) - m(3, 0) * m(2, 3), c14 = m(1, 0) * m(3, 3) - m(3, 0) * m(1, 3), c15 = m(1, 0) * m(2, 3) - m(2, 0) * m(1, 3);
  const double c16 = m(2, 0) * m(3, 2) - m(3, 0) * m(2, 2), c18 = m(1, 0) * m(3, 2) - m(3, 0) * m(1, 2), c19 = m(1, 0) * m(2, 2) - m(2, 0) * m(1, 2);
  const double c20 = m(2, 0) * m(3, 1) - m(3, 0) * m(2, 1), c22 = m(1, 0) * m(3, 1) - m(3, 0) * m(1, 1), c23 = m(1, 0) * m(2, 1) - m(2, 0) * m(1, 1);
  const double fac[6][4] = {{c00, c00, c02, c03}, {c04, c04, c06, c07}, {c08, c08, c10, c11},
                            {c12, c12, c14, c15}, {c16, c16, c18, c19}, {c20, c20, c22, c23}};
  double vec[4][4];   // Vec0..Vec3 = (m[1][r], m[0][r], m[0][r], m[0][r]) for r = 0..3
  for (int r = 0; r < 4; ++r) { vec[r][0] = m(1, r); vec[r][1] = vec[r][2] = vec[r][3] = m(0, r); }
  // Inv0 = V1 F0 - V2 F1 + V3 F2;  Inv1 = V0 F0 - V2 F3 + V3 F4;  Inv2 = V0 F1 - V1 F3 + V3 F5;  Inv3 = V0 F2 - V1 F4 + V2 F5
  static const int terms[4][6] = {{1, 0, 2, 1, 3, 2}, {0, 0, 2, 3, 3, 4}, {0, 1, 1, 3, 3, 5}, {0, 2, 1, 4, 2, 5}};
  double inv[16];
  for (int c = 0; c < 4; ++c) {
    const int* t = terms[c];
    const double sign0 = (c & 1) ? -1.0 : 1.0;   // SignA = (+,-,+,-) for columns 0 and 2, SignB = (-,+,-,+) for 1 and 3
    for (int k = 0; k < 4; ++k) {
      const double v = (vec[t[0]][k] * fac[t[1]][k] - vec[t[2]][k] * fac[t[3]][k]) + vec[t[4]][k] * fac[t[5]][k];
      inv[c * 4 + k] = v * ((k & 1) ? -sign0 : sign0);
    }
  }
  const double d0 = m(0, 0) * inv[0], d1 = m(0, 1) * inv[4], d2 = m(0, 2) * inv[8], d3 = m(0, 3) * inv[12];
  const double one_over_det = 1.0 / ((d0 + d1) + (d2 + d3));
  for (int k = 0; k < 16; ++k) out[k] = inv[k] * one_over_det;
}

// InvVP = ModelMatrix * inverse(ProjectionMatrix * ModelViewMatrix): clip space -> world space, in double from the float
// uniforms, rounded to float once per element
static void voxel_view_matrix(const Params& P, float* inv_vp) {
  double model[16], mv[16], proj[16], pmv[16], ipmv[16], r[16];
  for (int k = 0; k < 16; ++k) { model[k] = P.model[k]; mv[k] = P.model_view[k]; proj[k] = P.proj[k]; }
  mat4_mul(proj, mv, pmv);
  mat4_inverse_glm(pmv, ipmv);
  mat4_mul(model, ipmv, r);
  for (int k = 0; k < 16; ++k) inv_vp[k] = (float)r[k];
}

int vct_render_voxels(vct_handle c, int level, uint8_t* host_rgba, uint32_t* host_voxel) {
  NEED(c);
  if (level < 0 || level >= c->P.levels) return set_error(c, VCT_ERR_INVALID, "vct_render_voxels: level outside [0, levels)");
  int rc = need_pyramid(c, "vct_render_voxels", level); if (rc) return rc;
  rc = ensure_frame(c); if (rc) return rc;
  float inv_vp[16];
  voxel_view_matrix(c->P, inv_vp);
  if (!host_rgba && !host_voxel) return launch_voxel_view(c, level, inv_vp, nullptr);
  const size_t n = (size_t)c->P.W * c->P.H;
  return host_round_trip(c, "vct_render_voxels", {{nullptr, host_voxel, n * 4}}, [&](void* const* d) {
    const int r = launch_voxel_view(c, level, inv_vp, (uint32_t*)d[0]);
    if (r || !host_rgba) return r;
    // the view itself is in the frame buffer
    return check_cuda(c, cudaMemcpyAsync(host_rgba, c->d_frame, n * 4, cudaMemcpyDeviceToHost, c->stream), "vct_render_voxels");
  });
}

static int ensure_overlap(vct_context* c) {
  if (!c->stream2) {
    // higher priority than the main stream: cone_trace fills the machine with ~32 K small blocks, and the block
    // scheduler only hands SM slots to another grid ahead of them if that grid's stream has priority
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    VCT_CUDA(c, cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, prio_hi));
    VCT_CUDA(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    VCT_CUDA(c, cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming));
    VCT_CUDA(c, cudaMalloc(&c->d_counters_vis, sizeof(Counters)));
    VCT_CUDA(c, cudaMemset(c->d_counters_vis, 0, sizeof(Counters)));
    VCT_CUDA(c, cudaStreamCreateWithPriority(&c->stream_vox, cudaStreamNonBlocking, prio_hi));
    VCT_CUDA(c, cudaEventCreateWithFlags(&c->ev_vox_done, cudaEventDisableTiming));
    VCT_CUDA(c, cudaEventCreateWithFlags(&c->ev_vtx_done, cudaEventDisableTiming));
  }
  if (c->items_vis_cap != c->max_items || !c->d_items_vis) {
    cudaFree(c->d_items_vis); c->d_items_vis = nullptr;
    VCT_CUDA(c, cudaMalloc(&c->d_items_vis, c->max_items * sizeof(TileItem)));
    c->items_vis_cap = c->max_items;
  }
  return VCT_OK;
}

int vct_frame(vct_handle c, uint8_t* host_rgba) {
  NEED(c);
  next_event_generation(c);
  const int frame_gen = c->ev_gen;
  if (c->profile) cudaEventRecord(c->ev_begin[frame_gen][VCT_PASS_FRAME], c->stream);
  int rc = ensure_grid(c); if (rc) return rc;
  if (c->overlap_visibility) {
    // Three streams.  voxel stream: vertex pass -> clear -> voxelise -> resolve -> mip into the slot that the
    // previous frame's cone_trace is not reading; visibility stream: primary visibility (needs only the vertex
    // cache); main stream: cone_trace after both.  With PipelineFrames the voxel and visibility stages of frame
    // i+1 do not wait for cone_trace of frame i (they are latency-bound, cone_trace is texture-bound), unless
    // device-side inputs changed in between (scene_epoch), in which case they are ordered after the main stream.
    rc = ensure_frame(c); if (rc) return rc;
    rc = ensure_queues(c); if (rc) return rc;
    rc = sync_materials(c); if (rc) return rc;
    rc = ensure_overlap(c); if (rc) return rc;
    const bool ordered = !c->pipeline_frames || c->scene_epoch != c->frame_epoch;
    cudaStream_t main_stream = c->stream; TileItem* main_items = c->d_items; Counters* main_ctr = c->d_counters;
    if (ordered) VCT_CUDA(c, cudaEventRecord(c->ev_fork, main_stream));
    // --- voxel stream
    c->stream = c->stream_vox;
    rc = VCT_OK;
    if (ordered) rc = check_cuda(c, cudaStreamWaitEvent(c->stream_vox, c->ev_fork, 0), "wait fork");
    if (!rc) rc = begin_voxel_slot(c);
    if (!rc) rc = ensure_vertex_cache(c);
    if (!rc) rc = check_cuda(c, cudaEventRecord(c->ev_vtx_done, c->stream_vox), "record vtx");
    if (!rc) rc = draw_voxels_body(c);
    if (!rc) rc = check_cuda(c, cudaEventRecord(c->ev_vox_done, c->stream_vox), "record vox");
    // --- visibility stream (ordered after the vertex pass, hence after the slot became free)
    if (!rc) {
      c->stream = c->stream2; c->d_items = c->d_items_vis; c->d_counters = c->d_counters_vis;
      rc = check_cuda(c, cudaStreamWaitEvent(c->stream2, c->ev_vtx_done, 0), "wait vtx");
      if (!rc) rc = launch_visibility(c);
      if (!rc) rc = check_cuda(c, cudaEventRecord(c->ev_join, c->stream2), "record join");
    }
    c->stream = main_stream; c->d_items = main_items; c->d_counters = main_ctr;
    if (rc) return rc;
    // --- main stream
    VCT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_vox_done, 0));
    VCT_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));
    c->frame_epoch = c->scene_epoch;
  } else {
    rc = begin_voxel_slot(c); if (rc) return rc;
    rc = draw_voxels_body(c); if (rc) return rc;
    rc = launch_visibility(c); if (rc) return rc;
  }
  rc = launch_cone(c); if (rc) return rc;
  if (c->profile) { cudaEventRecord(c->ev_end[frame_gen][VCT_PASS_FRAME], c->stream); c->ev_recorded[frame_gen][VCT_PASS_FRAME] = true; }
  if (host_rgba) {
    VCT_CUDA(c, cudaMemcpyAsync(host_rgba, c->d_frame, (size_t)c->P.W * c->P.H * 4, cudaMemcpyDeviceToHost, c->stream));
    VCT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_overflow(c);       // a truncated queue must not pass for a frame (device-only paths: vct_sync)
  }
  return VCT_OK;
}

constexpr int VCT_ASYNC_FRAMES = 3;

static int ensure_async(vct_context* c) {
  if (!c->copy_stream) {
    VCT_CUDA(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int k = 0; k < VCT_ASYNC_FRAMES; ++k) {
      VCT_CUDA(c, cudaEventCreateWithFlags(&c->ev_rendered[k], cudaEventDisableTiming));
      VCT_CUDA(c, cudaEventCreateWithFlags(&c->ev_copied[k], cudaEventDisableTiming));
    }
    VCT_CUDA(c, cudaMallocHost(&c->h_overflow, VCT_ASYNC_FRAMES * 2 * sizeof(unsigned int)));
    std::memset(c->h_overflow, 0, VCT_ASYNC_FRAMES * 2 * sizeof(unsigned int));
  }
  if (c->frame2_W != c->P.W || c->frame2_H != c->P.H || !c->d_frame2[0]) {
    for (int k = 0; k < VCT_ASYNC_FRAMES; ++k) {
      if (c->in_flight[k]) { cudaEventSynchronize(c->ev_copied[k]); c->in_flight[k] = false; }
      cudaFree(c->d_frame2[k]); c->d_frame2[k] = nullptr;
      VCT_CUDA(c, cudaMalloc(&c->d_frame2[k], (size_t)c->P.W * c->P.H * 4));
    }
    c->frame2_W = c->P.W; c->frame2_H = c->P.H;
    c->frame_oldest = c->frame_seq;
  }
  return VCT_OK;
}

// the overflow words that travelled to the host behind frame `slot` (a truncated queue must not pass for a frame)
static int async_overflow(vct_context* c, int slot) {
  unsigned int* f = c->h_overflow + 2 * slot;
  if (!(f[0] | f[1])) return VCT_OK;
  f[0] = f[1] = 0;
  cudaMemsetAsync(&c->d_counters->overflow, 0, 4, c->stream);
  if (c->d_counters_vis) cudaMemsetAsync(&c->d_counters_vis->overflow, 0, 4, c->stream);
  return set_error(c, VCT_ERR_OVERFLOW, "device work queue overflow in an asynchronous frame: raise MaxFragments / MaxTileItems / MaxExchangeVoxels");
}

// blocks until the OLDEST frame still in flight has fully arrived in its host buffer
int vct_frame_wait(vct_handle c) {
  NEED(c);
  while (c->frame_oldest != c->frame_seq) {
    const int slot = c->frame_oldest % VCT_ASYNC_FRAMES;
    c->frame_oldest++;
    if (c->in_flight[slot]) {
      VCT_CUDA(c, cudaEventSynchronize(c->ev_copied[slot]));
      c->in_flight[slot] = false;
      return async_overflow(c, slot);
    }
  }
  return VCT_OK;
}

int vct_frame_async(vct_handle c, uint8_t* host_rgba) {
  NEED(c);
  if (!host_rgba) return set_error(c, VCT_ERR_INVALID, "vct_frame_async: host buffer required");
  int rc = ensure_frame(c); if (rc) return rc;
  rc = ensure_async(c); if (rc) return rc;
  const int slot = c->frame_seq % VCT_ASYNC_FRAMES;
  if (c->in_flight[slot]) {                       // ring full: this device buffer is still being copied out
    VCT_CUDA(c, cudaEventSynchronize(c->ev_copied[slot]));
    c->in_flight[slot] = false;
    if (c->frame_oldest + VCT_ASYNC_FRAMES == c->frame_seq) c->frame_oldest++;
    rc = async_overflow(c, slot); if (rc) return rc;
  }
  uchar4* saved = c->d_frame;
  c->d_frame = c->d_frame2[slot];                 // render straight into the slot
  rc = vct_frame(c, nullptr);
  c->d_frame = saved;
  if (rc) return rc;
  VCT_CUDA(c, cudaEventRecord(c->ev_rendered[slot], c->stream));
  VCT_CUDA(c, cudaStreamWaitEvent(c->copy_stream, c->ev_rendered[slot], 0));
  VCT_CUDA(c, cudaMemcpyAsync(host_rgba, c->d_frame2[slot], (size_t)c->P.W * c->P.H * 4, cudaMemcpyDeviceToHost, c->copy_stream));
  VCT_CUDA(c, cudaMemcpyAsync(c->h_overflow + 2 * slot, &c->d_counters->overflow, 4, cudaMemcpyDeviceToHost, c->copy_stream));
  if (c->d_counters_vis)
    VCT_CUDA(c, cudaMemcpyAsync(c->h_overflow + 2 * slot + 1, &c->d_counters_vis->overflow, 4, cudaMemcpyDeviceToHost, c->copy_stream));
  VCT_CUDA(c, cudaEventRecord(c->ev_copied[slot], c->copy_stream));
  c->in_flight[slot] = true;
  c->frame_seq++;
  return VCT_OK;
}

// ---- read-back
int vct_readback_depth(vct_handle c, uint32_t* d) {
  NEED(c);
  if (!d || !c->d_depth || !c->depth_valid) return set_error(c, VCT_ERR_STATE, "no shadow map");
  VCT_CUDA(c, cudaMemcpyAsync(d, c->d_depth, (size_t)c->P.S * c->P.S * 4, cudaMemcpyDeviceToHost, c->stream));
  return check_cuda(c, cudaStreamSynchronize(c->stream), "sync");
}
int vct_readback_counts(vct_handle c, uint32_t* counts) { NEED(c); return readback_accum(c, counts, nullptr); }
int vct_readback_sums(vct_handle c, uint32_t* sums) { NEED(c); return readback_accum(c, nullptr, sums); }

int vct_readback_grid(vct_handle c, int level, uint8_t* rgba) {
  NEED(c);
  int rc = ensure_grid(c); if (rc) return rc;
  if (level < 0 || level >= c->P.levels || !rgba) return set_error(c, VCT_ERR_INVALID, "bad mip level");
  const int n = c->P.V >> level;
  cudaArray_t lvl;
  VCT_CUDA(c, cudaGetMipmappedArrayLevel(&lvl, c->grid[c->cur].array, level));
  cudaMemcpy3DParms p{};
  const size_t bpt = c->grid_format == 1 ? 8 : 4;
  p.srcArray = lvl;
  p.dstPtr = make_cudaPitchedPtr(rgba, (size_t)n * bpt, n, n);
  p.extent = make_cudaExtent(n, n, n);
  p.kind = cudaMemcpyDeviceToHost;
  VCT_CUDA(c, cudaMemcpy3DAsync(&p, c->stream));
  return check_cuda(c, cudaStreamSynchronize(c->stream), "sync");
}

int vct_upload_grid_level0(vct_handle c, const uint8_t* rgba) {
  NEED(c);
  int rc = ensure_grid(c); if (rc) return rc;
  const int n = c->P.V;
  cudaArray_t lvl;
  VCT_CUDA(c, cudaGetMipmappedArrayLevel(&lvl, c->grid[c->cur].array, 0));
  cudaMemcpy3DParms p{};
  const size_t bpt = c->grid_format == 1 ? 8 : 4;
  p.srcPtr = make_cudaPitchedPtr(const_cast<uint8_t*>(rgba), (size_t)n * bpt, n, n);
  p.dstArray = lvl;
  p.extent = make_cudaExtent(n, n, n);
  p.kind = cudaMemcpyHostToDevice;
  VCT_CUDA(c, cudaMemcpy3DAsync(&p, c->stream));
  c->grid[c->cur].list_valid = false;   // level 0 no longer matches the touched list
  c->grid[c->cur].dirty_valid = false; c->grid[c->cur].occ_valid = false; c->grid[c->cur].mips_current = false;
  c->mask_valid[c->cur] = false;
  c->scene_epoch++;
  return check_cuda(c, cudaStreamSynchronize(c->stream), "sync");
}

int vct_build_mips(vct_handle c) { NEED(c); return launch_mip(c); }

__global__ void vis_to_tri(const unsigned long long* __restrict__ vis, uint32_t* __restrict__ tri, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) tri[i] = vis[i] == ~0ull ? 0xFFFFFFFFu : (uint32_t)vis[i];
}

int vct_readback_visibility(vct_handle c, uint32_t* tri) {
  NEED(c);
  if (!c->d_vis2[c->cur] || !tri) return set_error(c, VCT_ERR_STATE, "no frame rendered");
  const size_t n = (size_t)c->P.W * c->P.H;
  return host_round_trip(c, "vct_readback_visibility", {{nullptr, tri, n * 4}}, [&](void* const* d) {
    vis_to_tri<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_vis2[c->cur], (uint32_t*)d[0], n);
    c->launches += 1;
    return check_cuda(c, cudaGetLastError(), "vis_to_tri");
  });
}

int vct_readback_frame(vct_handle c, uint8_t* rgba) {
  NEED(c);
  if (!c->d_frame || !rgba) return set_error(c, VCT_ERR_STATE, "no frame rendered");
  // the most recent frame, wherever it was rendered (vct_render / vct_frame: d_frame; vct_frame_async and
  // vct_frame_sharded: a ring slot -- on ranks other than 0 of a sharded frame only the own rows are meaningful)
  const uchar4* src = c->last_frame ? c->last_frame : c->d_frame;
  VCT_CUDA(c, cudaMemcpyAsync(rgba, src, (size_t)c->P.W * c->P.H * 4, cudaMemcpyDeviceToHost, c->stream));
  return check_cuda(c, cudaStreamSynchronize(c->stream), "sync");
}

int vct_frame_buffer(vct_handle c, void** p, size_t* n) {
  NEED(c);
  int rc = ensure_frame(c); if (rc) return rc;
  if (p) *p = c->d_frame;
  if (n) *n = (size_t)c->P.W * c->P.H * 4;
  return VCT_OK;
}

static int read_counter(vct_context* c, const void* dptr, void* out, size_t bytes) {
  VCT_CUDA(c, cudaMemcpyAsync(out, dptr, bytes, cudaMemcpyDeviceToHost, c->stream));
  return check_cuda(c, cudaStreamSynchronize(c->stream), "sync");
}
static int read_steps(vct_context* c, StepCounter k, uint64_t* n) {
  unsigned long long parts[64 * 4];
  int rc = read_counter(c, c->d_counters->steps[k], parts, sizeof(parts));
  unsigned long long v = 0;
  for (int s = 0; s < 64; ++s) v += parts[s * 4];
  if (n) *n = v;
  return rc;
}
int vct_cone_samples(vct_handle c, uint64_t* n) { NEED(c); return read_steps(c, STEPS_CONE, n); }
int vct_fragment_count(vct_handle c, uint64_t* n) {
  NEED(c);
  unsigned int v = 0;
  int rc = read_counter(c, &c->d_counters->n_fragments, &v, 4);
  if (n) *n = v;
  return rc;
}
int vct_debug_counter(vct_handle c, int which, uint64_t* n) {   /* 0 = work items of the last raster pass */
  NEED(c);
  if (which >= STEPS_VIEW && which <= STEPS_RAYS) return read_steps(c, (StepCounter)which, n);
  unsigned int v = 0;
  int rc = read_counter(c, which == 0 ? (const void*)&c->d_counters->n_items : (const void*)&c->d_counters->overflow, &v, 4);
  if (n) *n = v;
  return rc;
}
int vct_occupied_voxels(vct_handle c, uint64_t* n) {
  NEED(c);
  unsigned int v = 0;
  int rc = ensure_grid(c); if (rc) return rc;
  rc = read_counter(c, c->grid[c->cur].n_touched, &v, 4);
  if (n) *n = v;
  return rc;
}

int vct_trace_cones(vct_handle c, size_t n, const float* starts, const float* dirs, const float* tans, float* out,
                    uint32_t* steps) {
  NEED(c);
  if (n && (!starts || !dirs || !tans || !out)) return set_error(c, VCT_ERR_INVALID, "vct_trace_cones: null argument");
  int rc = ensure_grid(c); if (rc) return rc;
  if (!n) return VCT_OK;
  return host_round_trip(c, "vct_trace_cones",
                         {{starts, nullptr, n * 12}, {dirs, nullptr, n * 12}, {tans, nullptr, n * 4}, {nullptr, out, n * 16},
                          {nullptr, steps, n * 4}},
                         [&](void* const* d) {
                           return launch_trace_cones(c, n, (const float*)d[0], (const float*)d[1], (const float*)d[2],
                                                     (float*)d[3], (uint32_t*)d[4]);
                         });
}

int vct_bake_probes(vct_handle c, size_t n, const float* xyz, float* out, uint32_t* steps, int on_device) {
  NEED(c);
  if (!n) return VCT_OK;
  if (!xyz || !out) return set_error(c, VCT_ERR_INVALID, "vct_bake_probes: null argument");
  if (n > SIZE_MAX / 256) return set_error(c, VCT_ERR_INVALID, "vct_bake_probes: n too large");
  int rc = need_pyramid(c, "vct_bake_probes", c->P.levels - 1); if (rc) return rc;   // every cone reads every level
  if (on_device) return launch_probes(c, n, xyz, out, steps);
  return host_round_trip(c, "vct_bake_probes", {{xyz, nullptr, n * 12}, {nullptr, out, n * 96}, {nullptr, steps, n * 24}},
                         [&](void* const* d) { return launch_probes(c, n, (const float*)d[0], (float*)d[1], (uint32_t*)d[2]); });
}

int vct_cast_rays(vct_handle c, int level, size_t n, const float* segments, uint32_t* voxel, float* t, uint8_t* face,
                  uint8_t* rgba, uint32_t* steps, int on_device) {
  NEED(c);
  if (!n) return VCT_OK;
  if (level < 0 || level >= c->P.levels) return set_error(c, VCT_ERR_INVALID, "vct_cast_rays: level outside [0, levels)");
  if (!segments || !voxel) return set_error(c, VCT_ERR_INVALID, "vct_cast_rays: null argument");
  if (n > SIZE_MAX / 64) return set_error(c, VCT_ERR_INVALID, "vct_cast_rays: n too large");
  if (on_device && ((uintptr_t)rgba & 3u)) return set_error(c, VCT_ERR_INVALID, "vct_cast_rays: rgba is not 4-byte aligned");
  int rc = need_pyramid(c, "vct_cast_rays", level); if (rc) return rc;
  if (on_device) return launch_cast_rays(c, level, n, segments, voxel, t, face, rgba, steps);
  return host_round_trip(c, "vct_cast_rays",
                         {{segments, nullptr, n * 24}, {nullptr, voxel, n * 4}, {nullptr, t, n * 4}, {nullptr, face, n},
                          {nullptr, rgba, n * 4}, {nullptr, steps, n * 4}},
                         [&](void* const* d) {
                           return launch_cast_rays(c, level, n, (const float*)d[0], (uint32_t*)d[1], (float*)d[2],
                                                   (uint8_t*)d[3], (uint8_t*)d[4], (uint32_t*)d[5]);
                         });
}

// ---- execution control
int vct_sample_voxels(vct_handle c, size_t n, const float* pos, const float* lod, float* out) {
  NEED(c);
  if (n && (!pos || !lod || !out)) return set_error(c, VCT_ERR_INVALID, "vct_sample_voxels: null argument");
  int rc = ensure_grid(c); if (rc) return rc;
  if (!n) return VCT_OK;
  return host_round_trip(c, "vct_sample_voxels", {{pos, nullptr, n * 12}, {lod, nullptr, n * 4}, {nullptr, out, n * 16}},
                         [&](void* const* d) {
                           return launch_sample_voxels(c, n, (const float*)d[0], (const float*)d[1], (float*)d[2]);
                         });
}

int vct_set_stream(vct_handle c, void* s) {
  NEED(c);
  cudaStreamSynchronize(c->stream);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)s;     // NULL = the CUDA default stream
  c->own_stream = false;
  return VCT_OK;
}

int vct_use_own_stream(vct_handle c) {
  NEED(c);
  cudaStreamSynchronize(c->stream);
  if (c->own_stream) return VCT_OK;
  VCT_CUDA(c, cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  return VCT_OK;
}

int vct_sync(vct_handle c) {
  NEED(c);
  int rc = check_cuda(c, cudaStreamSynchronize(c->stream), "cudaStreamSynchronize");
  if (rc) return rc;
  rc = comm_check(c); if (rc) return rc;
  return check_overflow(c);
}

int vct_pass_time_us(vct_handle c, int pass, float* us) {
  NEED(c);
  if (pass < 0 || pass >= VCT_PASS_COUNT || !us) return VCT_ERR_INVALID;
  int g = -1;
  if (pass == VCT_PASS_DEPTH && c->ev_recorded[0][pass]) g = 0;
  for (int k = 0; k < VCT_EVENT_GENS && g < 0; ++k) {            // the most recent generation in which the pass ran
    const int q = (c->ev_gen - k + VCT_EVENT_GENS) % VCT_EVENT_GENS;
    if (c->ev_recorded[q][pass]) g = q;
  }
  if (g < 0) return set_error(c, VCT_ERR_STATE, "pass has not run (or Profile = 0)");
  VCT_CUDA(c, cudaEventSynchronize(c->ev_end[g][pass]));
  float ms = 0.0f;
  VCT_CUDA(c, cudaEventElapsedTime(&ms, c->ev_begin[g][pass], c->ev_end[g][pass]));
  *us = ms * 1000.0f;
  return VCT_OK;
}

// begin / end of a pass of the frame `frames_back` frames ago (0 = the latest; < VCT_EVENT_GENS), in microseconds
// since Profile was switched on: all streams of all recent frames on one time axis
int vct_pass_timeline(vct_handle c, int frames_back, int pass, float* begin_us, float* end_us) {
  NEED(c);
  if (pass < 0 || pass >= VCT_PASS_COUNT || frames_back < 0 || frames_back >= VCT_EVENT_GENS || !begin_us || !end_us) return VCT_ERR_INVALID;
  const int g = (c->ev_gen - frames_back + VCT_EVENT_GENS) % VCT_EVENT_GENS;
  if (!c->ev_ref || !c->ev_recorded[g][pass]) return set_error(c, VCT_ERR_STATE, "vct_pass_timeline: pass not recorded in that frame");
  VCT_CUDA(c, cudaEventSynchronize(c->ev_end[g][pass]));
  float a = 0.0f, b = 0.0f;
  VCT_CUDA(c, cudaEventElapsedTime(&a, c->ev_ref, c->ev_begin[g][pass]));
  VCT_CUDA(c, cudaEventElapsedTime(&b, c->ev_ref, c->ev_end[g][pass]));
  *begin_us = a * 1000.0f; *end_us = b * 1000.0f;
  return VCT_OK;
}

int vct_kernel_launches(vct_handle c, uint64_t* n) { NEED(c); if (n) *n = c->launches; return VCT_OK; }

static int bench_tex3d(vct_context* c, int V, int f16, uint64_t n_samples, int pattern, float lod, int iters, float* gsps) {
  if (V < 8 || V > 1024 || (V & (V - 1)) || iters < 1 || !gsps) return set_error(c, VCT_ERR_INVALID, "vct_bench_tex3d: bad arguments");
  const int levels = ilog2(V) + 1;
  cudaMipmappedArray_t arr = nullptr;
  cudaChannelFormatDesc desc = f16 ? cudaCreateChannelDescHalf4() : cudaCreateChannelDesc<uchar4>();
  VCT_CUDA(c, cudaMallocMipmappedArray(&arr, &desc, make_cudaExtent(V, V, V), levels, cudaArraySurfaceLoadStore));
  for (int l = 0; l < levels; ++l) {
    cudaArray_t lvl;
    cudaGetMipmappedArrayLevel(&lvl, arr, l);
    cudaResourceDesc rd{}; rd.resType = cudaResourceTypeArray; rd.res.array.array = lvl;
    cudaSurfaceObject_t s;
    cudaCreateSurfaceObject(&s, &rd);
    int n = V >> l;
    dim3 b(32, 8), g((n + 31) / 32, (n + 7) / 8, n);
    fill_level_random<<<g, b, 0, c->stream>>>(s, n, 1234u + l, f16);
    cudaStreamSynchronize(c->stream);
    cudaDestroySurfaceObject(s);
  }
  cudaResourceDesc rd{}; rd.resType = cudaResourceTypeMipmappedArray; rd.res.mipmap.mipmap = arr;
  cudaTextureDesc td{};
  td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeWrap;
  td.filterMode = cudaFilterModeLinear; td.mipmapFilterMode = cudaFilterModeLinear;
  td.readMode = f16 ? cudaReadModeElementType : cudaReadModeNormalizedFloat; td.normalizedCoords = 1; td.maxMipmapLevelClamp = (float)(levels - 1);
  cudaTextureObject_t tex;
  VCT_CUDA(c, cudaCreateTextureObject(&tex, &rd, &td, nullptr));
  const int Wp = 1920, Hp = 1080, steps = (int)((n_samples + (uint64_t)Wp * Hp - 1) / ((uint64_t)Wp * Hp));
  float4* sink; VCT_CUDA(c, cudaMalloc(&sink, 16));
  dim3 b(256), g((Wp + 31) / 32, (Hp + 7) / 8);
  const float step_len = 1.0f / (float)(V >> (int)lod);   // one texel of the sampled level per step
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  tex3d_bench<<<g, b, 0, c->stream>>>(tex, steps, lod, pattern, step_len, sink, Wp);   // warm-up
  float best = 1e30f;
  for (int it = 0; it < iters; ++it) {
    cudaEventRecord(e0, c->stream);
    tex3d_bench<<<g, b, 0, c->stream>>>(tex, steps, lod, pattern, step_len, sink, Wp);
    cudaEventRecord(e1, c->stream);
    cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    best = ms < best ? ms : best;
  }
  c->launches += iters + 1 + levels;
  const double total = (double)g.x * 32 * g.y * 8 * steps;
  *gsps = (float)(total / (best * 1e-3) * 1e-9);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaDestroyTextureObject(tex); cudaFreeMipmappedArray(arr); cudaFree(sink);
  return check_cuda(c, cudaGetLastError(), "vct_bench_tex3d");
}

int vct_bench_tex3d(vct_handle c, int V, uint64_t n_samples, int pattern, float lod, int iters, float* gsps) {
  NEED(c);
  return bench_tex3d(c, V, 0, n_samples, pattern, lod, iters, gsps);
}

int vct_bench_tex3d_format(vct_handle c, int V, int grid_format, uint64_t n_samples, int pattern, float lod, int iters,
                           float* gsps) {
  NEED(c);
  if (grid_format != 0 && grid_format != 1) return set_error(c, VCT_ERR_INVALID, "vct_bench_tex3d_format: 0 = RGBA8, 1 = RGBA16F");
  return bench_tex3d(c, V, grid_format, n_samples, pattern, lod, iters, gsps);
}

int vct_bench_atomics(vct_handle c, uint64_t n_fragments, int iters, float* gatomics_per_s) {
  NEED(c);
  if (!gatomics_per_s || iters < 1 || n_fragments < 1 || n_fragments > 0xFFFFFFFFull) return set_error(c, VCT_ERR_INVALID, "vct_bench_atomics: bad arguments");
  int rc = ensure_grid(c); if (rc) return rc;
  rc = sync_all_streams(c); if (rc) return rc;
  unsigned int n_touched = 0;
  VCT_CUDA(c, cudaMemcpy(&n_touched, c->grid[c->cur].n_touched, 4, cudaMemcpyDeviceToHost));
  if (!n_touched || !c->grid[c->cur].list_valid) return set_error(c, VCT_ERR_STATE, "vct_bench_atomics: voxelise first (needs the touched-voxel list)");
  // a scratch accumulator: the context's own one must stay consistent with its lists
  unsigned long long* scratch = nullptr;
  const size_t n = (size_t)c->P.V * c->P.V * c->P.V;
  VCT_CUDA(c, cudaMalloc(&scratch, n * 16));
  VCT_CUDA(c, cudaMemsetAsync(scratch, 0, n * 16, c->stream));
  uint32_t mult = (uint32_t)((n_fragments + n_touched - 1) / n_touched);
  if (mult < 1) mult = 1;
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  atomics_bench<<<148 * 8, 256, 0, c->stream>>>(scratch, c->grid[c->cur].touched, n_touched, (uint32_t)n_fragments, mult);
  float best = 1e30f;
  for (int it = 0; it < iters; ++it) {
    cudaEventRecord(e0, c->stream);
    atomics_bench<<<148 * 8, 256, 0, c->stream>>>(scratch, c->grid[c->cur].touched, n_touched, (uint32_t)n_fragments, mult);
    cudaEventRecord(e1, c->stream);
    cudaEventSynchronize(e1);
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    best = ms < best ? ms : best;
  }
  c->launches += iters + 1;
  *gatomics_per_s = (float)(2.0 * (double)n_fragments / (best * 1e-3) * 1e-9);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(scratch);
  return check_cuda(c, cudaGetLastError(), "vct_bench_atomics");
}

}  // extern "C"
