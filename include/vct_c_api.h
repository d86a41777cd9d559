/*
 * vct_c_api.h -- C ABI of libvct_b200.so, the B200 (sm_100a) implementation of the hot path of
 * AlerianEmperor/Voxel-Cone-Tracing: shadow map -> voxelisation with PCF light injection -> 3D mip
 * pyramid -> per-pixel cone tracing.
 *
 * Every entry point replaces a piece of the reference's OpenGL pipeline; the reference location is
 * cited as file:line relative to /root/reference/Voxel_Cone_Tracing_Final/.  Plain pointers and sizes
 * only: no C++ or torch types cross this boundary.  All functions return 0 on success and a negative
 * vct_status otherwise; vct_last_error() gives the message.  A handle is not thread-safe (the
 * reference is single threaded: one GL context, main.cpp:44).  There is NO CPU fallback: creating a
 * context without a CUDA device fails with VCT_ERR_CUDA.
 */
#ifndef VCT_C_API_H_
#define VCT_C_API_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vct_context* vct_handle;

typedef enum vct_status {
  VCT_OK = 0,
  VCT_ERR_INVALID = -1,     /* bad argument / unknown uniform name (GL silently ignores location -1) */
  VCT_ERR_CUDA = -2,        /* a CUDA runtime call failed, or no device */
  VCT_ERR_STATE = -3,       /* pass called before its inputs exist (no mesh, no shadow map, ...) */
  VCT_ERR_OVERFLOW = -4     /* a device work queue overflowed; raise MaxFragments / MaxTileItems */
} vct_status;

/* pass identifiers for vct_pass_time_us */
typedef enum vct_pass {
  VCT_PASS_DEPTH = 0,       /* DrawDepthTexture                         Voxel_Cone_Tracing.h:192-211 */
  VCT_PASS_VOX_CLEAR = 1,   /* (reference never clears: texture zeroed once, :115-121)              */
  VCT_PASS_VOX_COVER = 2,   /* Voxelization.vs/.gs + rasteriser         Shader/Voxelization.gs:22-51 */
  VCT_PASS_VOX_SHADE = 3,   /* Voxelization.fs (albedo, PCF, store)     Shader/Voxelization.fs:54-89 */
  VCT_PASS_RESOLVE = 4,     /* accumulator -> RGBA8 level 0 (imageStore's unorm8 conversion)        */
  VCT_PASS_MIP = 5,         /* glGenerateMipmap(GL_TEXTURE_3D)          Voxel_Cone_Tracing.h:246-248 */
  VCT_PASS_VISIBILITY = 6,  /* VoxelConeTracing.vs + raster + depth test + discard                  */
  VCT_PASS_CONE = 7,        /* VoxelConeTracing.fs                      Shader/VoxelConeTracing.fs:165-229 */
  VCT_PASS_FRAME = 8,       /* whole vct_frame() call                                               */
  VCT_PASS_REINJECT = 9,    /* Bounces >= 3 extension                                               */
  VCT_PASS_EXCHANGE_PUSH = 10,  /* vct_voxelize_shared: multicast of the touched voxels (multimem.st / multimem.red) */
  VCT_PASS_EXCHANGE_MERGE = 11, /* vct_resolve_shared (inbox): the other ranks' records added to the accumulator     */
  VCT_PASS_VOXEL_VIEW = 12, /* vct_render_voxels (no reference counterpart)                          */
  VCT_PASS_PROBES = 13,     /* vct_bake_probes (no reference counterpart)                            */
  VCT_PASS_RAYS = 14,       /* vct_cast_rays (no reference counterpart)                              */
  VCT_PASS_COUNT = 15
} vct_pass;

/* ---- lifetime.  Replaces Voxel_Cone_Tracing::Voxel_Cone_Tracing + init_voxel_cone_tracing resource
 * creation (Voxel_Cone_Tracing.h:57-136: FBO, depth texture, 3D texture).  Defaults are the
 * reference's constants (VoxelDimensions 128, VoxelGridWorldSize 150, ShadowMapSize 4096, 1280x720). */
int vct_create(int cuda_device, vct_handle* out);
int vct_destroy(vct_handle h);
const char* vct_last_error(vct_handle h);     /* h may be NULL: error of the last failed vct_create */
const char* vct_version(void);

/* ---- uniforms.  Replace Shader::setInt/setFloat/setVec3/setMat4 (Shader.h:362-417) with the same
 * string keys the reference passes (Voxel_Cone_Tracing.h:167-187,224-243):
 *   int   : VoxelDimensions ShadowMapSize screen_width screen_height PcfRadius CoveragePolicy
 *           Bounces NumDiffuseCones GridFormat MaxFragments MaxTileItems DenseResolve Profile
 *           RowBegin RowEnd (rows [RowBegin, RowEnd) of the frame are rendered; RowEnd 0 = all: row-band sharding)
 *           RowInterleave RowPhase (instead: the frame is cut into strips of 8 rows and this context renders every
 *             RowInterleave-th strip, starting at strip RowPhase -- balanced row sharding, one phase per rank)
 *           TriangleInterleave TrianglePhase (voxelisation takes every TriangleInterleave-th block of 128 triangles of
 *             the requested range, starting at block TrianglePhase: balanced triangle sharding, one phase per rank)
 *           SharedExchange SharedWorld SharedRank MaxExchangeVoxels (fused sharded voxelisation, see below)
 *           ShardShadowMap (1, set before vct_comm_init: vct_draw_depth rasterises only this rank's triangle share and
 *             min-reduces every depth fragment into all ranks' D24 images -- multimem.red.min.u32 in the NVSwitch; the
 *             resulting map is bit-identical to the single-GPU one.  SURVEY 8e "shadow map")
 *           ShadowMap VoxelTexture (texture-unit numbers: accepted and ignored)
 *           PipelineFrames OverlapVisibility (frame pipeline; defaults are the measured best)
 *   float : VoxelGridWorldSize ambientFactor DiffuseTanHalfAngle SpecularTanHalfAngle StepMultiplier
 *           MaxDistance MaxAlpha ShadowBias
 *   vec3  : CameraPosition LightDirection
 *   mat4  : ModelMatrix ModelViewMatrix ProjectionMatrix DepthModelViewProjectionMatrix ProjX ProjY ProjZ
 *           (16 floats, column-major, i.e. glm memory order with transpose = GL_FALSE)             */
int vct_set_i(vct_handle h, const char* name, int v);
int vct_set_f(vct_handle h, const char* name, float v);
int vct_set_3f(vct_handle h, const char* name, float x, float y, float z);
int vct_set_mat4(vct_handle h, const char* name, const float* colmajor16);
int vct_get_i(vct_handle h, const char* name, int* v);
int vct_get_f(vct_handle h, const char* name, float* v);
/* Cone_Directions / Cone_Weights tables (VoxelConeTracing.fs:48-57); n <= 16 */
int vct_set_cones(vct_handle h, int n, const float* directions_xyz, const float* weights);

/* ---- scene.  Replace Model/Mesh upload (Mesh.h:49-82 glBufferData; Model.h:141-186 glTexImage2D +
 * glGenerateMipmap) and the per-mesh sampler binding (Mesh.h:84-111).  Host arrays stay owned by the
 * caller; the library copies them to the device. */
int vct_upload_texture(vct_handle h, int tex_id, int width, int height, int channels /*1,3,4*/,
                       const uint8_t* pixels);
int vct_set_material(vct_handle h, int material_id, int diffuse_tex, int specular_tex, int height_tex,
                     float shininess /* Mesh.h:86: 20 */);
/* verts14 = struct Vertex (Mesh.h:12-19): Position3 Normal3 TexCoords2 Tangents3 Bi_Tangents3 */
int vct_upload_mesh(vct_handle h, const float* verts14, size_t n_verts, const uint32_t* indices,
                    size_t n_tris, const uint16_t* tri_material /* may be NULL */);
/* dynamic meshes: overwrite Position of every vertex; src is n_verts*3 floats on the host or, with
 * on_device != 0, a device pointer on the context's device (copied on the context's stream) */
int vct_update_positions(vct_handle h, const float* xyz, size_t n_verts, int on_device);

/* ---- passes.  One per reference method. */
int vct_draw_depth(vct_handle h);        /* DrawDepthTexture   Voxel_Cone_Tracing.h:192-211 */
int vct_draw_voxels(vct_handle h);       /* DrawVoxelTexture   Voxel_Cone_Tracing.h:213-250 (clear+voxelise+resolve+mip) */
/* Render, Voxel_Cone_Tracing.h:146-190.  host_rgba (H*W*4 bytes, row 0 = bottom row as in GL window
 * coordinates) may be NULL: then the frame stays on the device and the call is asynchronous. */
int vct_render(vct_handle h, uint8_t* host_rgba);
/* vct_draw_voxels + vct_render as one call (what the metric "full frames/s" times) */
int vct_frame(vct_handle h, uint8_t* host_rgba);
/* Voxel view (no reference counterpart): the W*H view of mip level `level` of the current pyramid from the camera of
 * vct_render (ModelMatrix, ModelViewMatrix, ProjectionMatrix, screen size).  Each pixel shows the first occupied texel
 * its ray meets between the near and far planes, un-premultiplied and shaded by the axis of the face it entered through;
 * a miss shows the frame background.  host_rgba (H*W*4, row 0 = bottom row) and host_voxel (H*W texel indices
 * (z*N+y)*N+x at that level, 0xFFFFFFFF = miss) may each be NULL; with both NULL the call is asynchronous.  Writes the
 * frame buffer (vct_readback_frame / vct_frame_buffer return the view), renders every row whatever the row-sharding
 * uniforms say, and is stream-ordered after earlier frames.  VCT_ERR_INVALID: level outside [0, levels);
 * VCT_ERR_STATE: level > 0 after vct_upload_grid_level0 without vct_build_mips.  DESIGN.md section 3 "Voxel view". */
int vct_render_voxels(vct_handle h, int level, uint8_t* host_rgba, uint32_t* host_voxel);

/* Pipelined form of vct_frame for render loops (the reference's loop is glClear -> Render -> glfwSwapBuffers,
 * main.cpp:77-94; swapping is what lets a GL driver overlap frames).  vct_frame_async renders into one of a ring
 * of three device frame buffers and queues the device->host copy of that frame to host_rgba on a separate copy
 * stream; it returns without waiting.  vct_frame_wait blocks until the OLDEST frame still in flight has fully
 * arrived in its host buffer (at most three frames are in flight; a fourth vct_frame_async waits for the oldest
 * itself).  Keeping two frames queued lets the next frame's voxel stages start beside the current cone_trace.
 * host_rgba should be pinned memory for the copy to overlap. */
int vct_frame_async(vct_handle h, uint8_t* host_rgba);
int vct_frame_wait(vct_handle h);

/* split form of vct_draw_voxels for triangle-sharded voxelisation across GPUs: accumulate a triangle
 * range into the integer accumulator, exchange (all-reduce the buffer returned by vct_accum_buffer as
 * uint32 sum), then resolve + mip.  clear_first zeroes the accumulator. */
int vct_voxelize_range(vct_handle h, size_t tri_begin, size_t tri_end, int clear_first);
int vct_accum_buffer(vct_handle h, void** device_ptr, size_t* n_uint32);
int vct_resolve_and_mip(vct_handle h);   /* dense resolve of the whole accumulator, then mip */

/* Fused form of the same exchange over NVLink / NVSwitch (one process per GPU).  The caller provides ONE symmetric
 * allocation per rank (same size everywhere, e.g. torch symmetric memory) that is also mapped through a MULTICAST
 * address.  Set SharedWorld / SharedRank (vct_set_i) first; vct_shared_accum_bytes gives the size.  Two flavours
 * (vct_set_i "SharedExchange"):
 *   0 (default) inbox: every rank voxelises its triangle range privately, then multicasts one record per
 *     voxel it touched (one 16-byte record: index, 24-bit integer sums, 24-bit count) with multimem.st into its row of every rank's inbox; after the
 *     barrier each rank adds the other rows into its private accumulator -- which then equals a single-GPU
 *     voxelisation bit for bit -- and the ordinary sparse resolve + mip follow.  Exchange volume = touched voxels.
 *   1 in-switch reduction: the accumulator itself is the symmetric buffer ([16 B * V^3][V^3/8 B occupancy mask]) and
 *     every touched voxel is added into all copies at once with multimem.red.add.v4.f32 (reduced in the switch),
 *     followed by a mask-driven resolve.
 * With multicast_ptr == NULL (single GPU) plain local stores / atomics are used.
 *   per frame:  vct_voxelize_shared(range of this rank) -> cross-rank barrier -> vct_resolve_shared()
 *   (flavour 1 needs a second barrier after vct_resolve_shared) */
int vct_shared_accum_bytes(vct_handle h, size_t* bytes);
int vct_set_shared_accum(vct_handle h, void* local_ptr, void* multicast_ptr);
int vct_voxelize_shared(vct_handle h, size_t tri_begin, size_t tri_end);
int vct_resolve_shared(vct_handle h);
/* The same frame, pipelined like vct_frame (inbox flavour only).  begin: this rank's share is voxelised and multicast on
 * the library's voxel stream while primary visibility runs on a second stream; the caller then enqueues its cross-rank
 * barrier ON vct_exchange_stream (stream order is the only synchronisation needed); end: merge + resolve + mip on the
 * voxel stream and cone_trace (rows RowBegin..RowEnd) on the main stream after both.  With PipelineFrames = 1 the
 * voxel / exchange / visibility stages of frame i+1 overlap cone_trace of frame i -- the replicated part of a sharded
 * frame (clear, merge, resolve, mip) hides behind the sharded one.  Replaces main.cpp:81-92 for a multi-GPU loop. */
int vct_frame_shared_begin(vct_handle h, size_t tri_begin, size_t tri_end);
int vct_exchange_stream(vct_handle h, void** cuda_stream);
int vct_frame_shared_end(vct_handle h, uint8_t* host_rgba_or_null);

/* ---- multi-GPU, owned by the library (SURVEY.md 8b "pass entry points": vct_create_multi; 8e).  The reference is one
 * GL context on one GPU (main.cpp:44); a sharded frame replaces its loop body glClear -> Render -> glfwSwapBuffers
 * (main.cpp:81-92).  No torch, NCCL or MPI is involved: the library allocates one symmetric segment per rank
 * (cuMemCreate), maps every rank's segment on every rank (NVLink peer access) and binds them to one NVSwitch multicast
 * object (cuMulticastCreate / cuMulticastBindMem), passes the handles between processes itself (POSIX file descriptors
 * over an abstract unix socket named after `session`; rank 0 is the hub) and synchronises ranks with a device-side
 * barrier kernel enqueued in stream order.  One node only.
 *
 *   one process per GPU:   vct_create(device) ; set uniforms + scene (identical on every rank) ; vct_draw_depth ;
 *                          vct_comm_init(h, rank, world, session, flags) ; loop { vct_frame_sharded(h, host) } ;
 *                          vct_frame_sharded_wait(h)
 *   one process, n GPUs:   vct_create_multi(devices, n, hs) ; same set-up on every handle ; vct_comm_init_multi(hs, n, flags) ;
 *                          loop { vct_frame_sharded_multi(hs, n, host) } ; vct_frame_sharded_wait(hs[r]) for every r
 *
 * vct_comm_init sizes the segment from the CURRENT VoxelDimensions / screen size / MaxExchangeVoxels (call it again after
 * changing them) and, unless VCT_COMM_KEEP_SHARES is given, deals the work: triangles in blocks of 128 round-robin
 * (TriangleInterleave / TrianglePhase) and rows in strips of 8 round-robin (RowInterleave / RowPhase; contiguous bands
 * RowBegin / RowEnd with VCT_COMM_ROW_BANDS).  All ranks must call it with the same
 * world, session and settings; it blocks until every rank has joined (120 s limit). */
#define VCT_COMM_NO_MULTICAST 1   /* do not create a multicast object: exchange by one peer store per rank */
#define VCT_COMM_KEEP_SHARES  2   /* leave TriangleInterleave / TrianglePhase / RowInterleave / RowPhase / RowBegin / RowEnd as the caller set them */
#define VCT_COMM_ROW_BANDS    4   /* contiguous row bands (RowBegin / RowEnd) instead of interleaved strips of 8 rows */
int vct_comm_init(vct_handle h, int rank, int world, const char* session, int flags);
int vct_comm_destroy(vct_handle h);
int vct_comm_info(vct_handle h, int* rank, int* world, int* multicast, size_t* segment_bytes);
int vct_comm_barrier(vct_handle h);     /* enqueue the device-side cross-rank barrier on the context's stream */
/* One sharded frame: this rank voxelises its triangle share and multicasts the voxels it touched (multimem.st), merges
 * the other ranks' records after a device barrier, builds the pyramid, traces its row band and writes the pixels
 * straight into RANK 0's frame ring over NVLink (cone_trace's own epilogue -- no staging copy, no collective call).
 * Rank 0 then queues the device->host copy of the assembled frame into host_rgba (pinned memory recommended; NULL
 * keeps the frame on the device; ignored on other ranks).  Returns without waiting: up to three frames are in flight
 * and the voxel stages of frame i+1 run beside cone_trace of frame i.  vct_frame_sharded_wait blocks until every frame
 * issued so far is complete on this rank (rank 0: has arrived in host memory) and reports queue overflows and barrier
 * time-outs. */
int vct_frame_sharded(vct_handle h, uint8_t* host_rgba);
int vct_frame_sharded_wait(vct_handle h);
int vct_comm_frame_buffer(vct_handle h, void** device_ptr, size_t* n_bytes);   /* rank 0: the last assembled frame */
/* the same for one process that drives n devices (out / hs: arrays of n handles; rank = array index) */
int vct_create_multi(const int* devices, int n, vct_handle* out);
int vct_comm_init_multi(vct_handle* hs, int n, int flags);
int vct_frame_sharded_multi(vct_handle* hs, int n, uint8_t* host_rgba);

/* ---- read-back (the reference reads nothing back; these exist for parity checks and hosts) */
int vct_readback_depth(vct_handle h, uint32_t* d24 /* S*S */);
int vct_readback_counts(vct_handle h, uint32_t* counts /* V^3, (z*V+y)*V+x */);
int vct_readback_sums(vct_handle h, uint32_t* rgb /* V^3*3 */);
int vct_readback_grid(vct_handle h, int level, uint8_t* rgba /* (V>>level)^3 texels: 4 B (RGBA8) or 8 B (RGBA16F half bits) each */);
int vct_upload_grid_level0(vct_handle h, const uint8_t* rgba);   /* then vct_build_mips */
int vct_build_mips(vct_handle h);
int vct_readback_visibility(vct_handle h, uint32_t* tri_id /* H*W, 0xFFFFFFFF = background */);
int vct_readback_frame(vct_handle h, uint8_t* rgba /* H*W*4 */);
int vct_frame_buffer(vct_handle h, void** device_ptr, size_t* n_bytes);
int vct_cone_samples(vct_handle h, uint64_t* n);       /* textureLod calls of the last vct_render */
int vct_fragment_count(vct_handle h, uint64_t* n);     /* fragments of the last voxelisation */
int vct_occupied_voxels(vct_handle h, uint64_t* n);
/* diagnostics: 0 = tile work items of the last raster pass, 1 = texels the last voxel view visited (all pixels),
 * 2 = textureLod calls of the last vct_bake_probes (all probes and faces), 3 = texels the last vct_cast_rays visited
 * (all segments) */
int vct_debug_counter(vct_handle h, int which, uint64_t* n);

/* ---- cone queries: Voxel_Cone_Tracing(direction, tanHalfAngle) (VoxelConeTracing.fs:82-107) for arbitrary
 * start points (already offset along the normal, :92).  Host arrays: starts/dirs n*3, tan_half n,
 * out_rgb_occ n*4 (rgb, occlusion), out_steps n (may be NULL).  Used by probes and by the parity tests to
 * exercise the hardware-filtered tex3DLod path sample by sample. */
int vct_trace_cones(vct_handle h, size_t n, const float* starts, const float* dirs, const float* tan_half,
                    float* out_rgb_occ, uint32_t* out_steps);

/* Irradiance probes (no reference counterpart): the frame's diffuse term -- indirect light ind.rgb and occlusion,
 * VoxelConeTracing.fs:196-201 -- at n points p (xyz n*3, world space as Position_world) for a surface facing each of
 * +X, -X, +Y, -Y, +Z, -Z in that order.  Face f turns the current cone table (vct_set_cones) by a fixed orthonormal basis
 * (T, B, N) with N the face's axis, starts at p + N * VoxelGridWorldSize / VoxelDimensions and marches every cone as
 * vct_trace_cones does with DiffuseTanHalfAngle, weighted sum in cone order.  out[((p*6)+f)*4 + k] = (ind.r, ind.g,
 * ind.b, 1 - ind.a); steps[p*6+f] (may be NULL) = textureLod calls of that face.  A probe with a non-finite coordinate
 * gives NaN and 0 steps.  Camera, screen size and row-sharding uniforms have no effect.  With on_device != 0 all
 * pointers are device pointers on the context's device and the call is asynchronous on the context's stream (no
 * allocation, no synchronisation); otherwise they are host arrays and the call returns when they are filled.  Reads the
 * current pyramid after the frames issued before it and keeps a later frame from overwriting it while it runs; the frame
 * buffer and vct_cone_samples are untouched.  n = 0: no-op.  VCT_ERR_INVALID: NULL xyz or out with n > 0, n too large;
 * VCT_ERR_STATE: mip levels stale (vct_upload_grid_level0 without vct_build_mips).  DESIGN.md section 3 "Irradiance
 * probes". */
int vct_bake_probes(vct_handle h, size_t n, const float* xyz, float* out, uint32_t* steps, int on_device);

/* Ray casts (no reference counterpart): for each of n world-space segments a -> b (segments: n*6 floats a.xyz, b.xyz, in
 * the space of Position_world / vct_bake_probes), the first occupied texel of mip `level` of the current pyramid.  The
 * walk is the voxel view's (DESIGN.md section 3 "Voxel view" steps 3-5, "Ray casts") from o = (a/G + 0.5)*N to
 * e = (b/G + 0.5)*N in texel space, N = VoxelDimensions >> level, G = VoxelGridWorldSize; the segment is t in [0, 1], the
 * grid does not repeat.  Per segment on a hit: voxel = (z*N + y)*N + x; t = the segment parameter at which the walk
 * entered that texel; face = the outward normal of the face it entered through, 1..6 = +X, -X, +Y, -Y, +Z, -Z, 0 when
 * the segment starts inside it; rgba = its colour un-premultiplied as the view shows it before face shading, alpha = its
 * alpha as unorm8; steps = texels visited.  On a miss: voxel 0xFFFFFFFF, t +inf, face 0, rgba 0.  a == b is a point
 * query; a non-finite coordinate is a miss with 0 steps.  t, face, rgba (4 bytes per segment) and steps may be NULL.
 * With on_device != 0 all pointers are device pointers on the context's device (rgba 4-byte aligned) and the call is
 * asynchronous on the context's stream (no allocation, no synchronisation); otherwise they are host arrays and the call
 * returns when they are filled.  Reads the current pyramid after the frames issued before it and keeps a later frame
 * from overwriting it while it runs; the frame buffer and vct_cone_samples are untouched; the camera, screen size and
 * row-sharding uniforms have no effect.  n = 0: no-op.  VCT_ERR_INVALID: level outside [0, levels), NULL segments or
 * voxel with n > 0, n too large, a misaligned device rgba; VCT_ERR_STATE: level > 0 with the mip levels stale
 * (vct_upload_grid_level0 without vct_build_mips). */
int vct_cast_rays(vct_handle h, int level, size_t n, const float* segments, uint32_t* voxel, float* t, uint8_t* face,
                  uint8_t* rgba, uint32_t* steps, int on_device);

/* SampleVoxels(World_Position, lod) (VoxelConeTracing.fs:59-66) for n points: pos n*3, lod n, out n*4 */
int vct_sample_voxels(vct_handle h, size_t n, const float* world_pos, const float* lod, float* out_rgba);

/* ---- execution control */
/* run on the caller's stream (e.g. torch's current stream); NULL selects the CUDA default stream, exactly as
 * in the CUDA API.  vct_use_own_stream returns to the context's private non-blocking stream. */
int vct_set_stream(vct_handle h, void* cuda_stream);
int vct_use_own_stream(vct_handle h);
int vct_sync(vct_handle h);
int vct_pass_time_us(vct_handle h, int pass, float* us);   /* CUDA-event time of the last run of a pass */
int vct_kernel_launches(vct_handle h, uint64_t* n);        /* kernels launched by this context so far */
/* begin / end of `pass` in the frame `frames_back` frames ago (0 = latest, at most 3), in microseconds since Profile was
 * last switched on: the passes of consecutive frames on one time axis, i.e. how the three streams overlap */
int vct_pass_timeline(vct_handle h, int frames_back, int pass, float* begin_us, float* end_us);

/* ---- micro-benchmarks used for the roofline denominators (DESIGN.md "Rooflines") */
/* trilinear+mip-linear tex3DLod throughput on a V^3 RGBA8 pyramid: n_samples per launch, pattern 0 =
 * coherent cone-like walks, 1 = random.  Returns giga-samples/s. */
int vct_bench_tex3d(vct_handle h, int V, uint64_t n_samples, int pattern, float lod, int iters,
                    float* gsamples_per_s);
/* the same on a pyramid of the given GridFormat (0 = RGBA8, 1 = RGBA16F: 8 B texels, BASELINE config 3); V also sets
 * the residency: 64^3 RGBA8 = 1 MiB (L1/L2), 256^3 = 73 MiB (L2), 512^3 RGBA16F = 1.17 GiB (HBM) */
int vct_bench_tex3d_format(vct_handle h, int V, int grid_format, uint64_t n_samples, int pattern, float lod, int iters,
                           float* gsamples_per_s);
/* 64-bit atomicAdd rate of the voxel accumulation (two atomics per fragment, vox_shade) on the voxel population of
 * the last voxelisation with its mean fragments-per-voxel multiplicity.  Returns giga-atomics/s. */
int vct_bench_atomics(vct_handle h, uint64_t n_fragments, int iters, float* gatomics_per_s);

#ifdef __cplusplus
}
#endif
#endif /* VCT_C_API_H_ */
