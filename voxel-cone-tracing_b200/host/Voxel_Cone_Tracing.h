// Voxel_Cone_Tracing.h -- C++ host facade with the reference's own class surface.
//
// Mirrors `struct Voxel_Cone_Tracing` of /root/reference/Voxel_Cone_Tracing_Final/Voxel_Cone_Tracing.h:11-252: same
// struct name, field names and method names (init_voxel_cone_tracing / Render / DrawDepthTexture / DrawVoxelTexture);
// every GL call in the method bodies is replaced by calls through the C ABI of include/vct_c_api.h, with the same
// uniform names the reference passes to Shader::set*.  GL object ids become one opaque device handle; `window` is an
// ignored void*; VoxelDimensions / VoxelGridWorldSize are runtime values (reference defaults 128 / 150).  The scene is
// handed over as the flattened output of the reference's loader (struct Vertex of Mesh.h:12-19) instead of a file path.
#ifndef _VOXEL_CONE_TRACING_H_
#define _VOXEL_CONE_TRACING_H_

#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "vct_c_api.h"
#include "vct_glm.h"

using vctm::mat4;
using vctm::vec3;

// Camera.h: the fly camera -- position, Yaw = -90, Pitch = 0, Zoom = 45, MovementSpeed = 2.6, MouseSensitivity = 0.1
// (Camera.h:21-25, 50-60); GetViewMatrix (:75-78), ProcessKeyBoard (:80-101), ProcessMouseMovement (:103-119),
// ProcessMouseScroll (:121-129), UpdateCamera (:131-144)
enum Camera_Direction { FORWARD, BACKWARD, LEFT, RIGHT, UP, DOWN };
struct Camera {
  vec3 position;
  vec3 Front = vec3(0.0f, 0.0f, -1.0f), Up = vec3(0.0f, 1.0f, 0.0f), Right = vec3(1.0f, 0.0f, 0.0f), WorldUp = vec3(0.0f, 1.0f, 0.0f);
  float Yaw = -90.0f, Pitch = 0.0f, Zoom = 45.0f;
  float MovementSpeed = 2.6f, MouseSensitivity = 0.1f;
  explicit Camera(vec3 p = vec3(0.0f, 4.0f, 0.0f)) : position(p) { UpdateCamera(); }
  void UpdateCamera() {
    float y = vctm::radians(Yaw), p = vctm::radians(Pitch);
    Front = vctm::normalize(vec3(std::cos(y) * std::cos(p), std::sin(p), std::sin(y) * std::cos(p)));
    Right = vctm::normalize(vctm::cross(Front, WorldUp));
    Up = vctm::normalize(vctm::cross(Right, Front));
  }
  mat4 GetViewMatrix() const {
    float y = vctm::radians(Yaw), p = vctm::radians(Pitch);
    vec3 front = vctm::normalize(vec3(std::cos(y) * std::cos(p), std::sin(p), std::sin(y) * std::cos(p)));
    vec3 right = vctm::normalize(vctm::cross(front, vec3(0.0f, 1.0f, 0.0f)));
    vec3 up = vctm::normalize(vctm::cross(right, front));
    return vctm::lookAt(position, position + front, up);
  }
  void ProcessKeyBoard(Camera_Direction direction, float deltaTime) {
    float velocity = MovementSpeed * deltaTime;
    if (direction == FORWARD) position = position + Front * velocity;
    if (direction == BACKWARD) position = position - Front * velocity;
    if (direction == LEFT) position = position - Right * velocity;
    if (direction == RIGHT) position = position + Right * velocity;
    if (direction == UP) position = position + WorldUp * velocity;
    if (direction == DOWN) position = position - WorldUp * velocity;
  }
  void ProcessMouseMovement(float xOffset, float yOffset, bool constrainPitch = true) {
    Yaw += xOffset * MouseSensitivity;
    Pitch += yOffset * MouseSensitivity;
    if (constrainPitch) { if (Pitch > 89.0f) Pitch = 89.0f; if (Pitch < -89.0f) Pitch = -89.0f; }
    UpdateCamera();
  }
  void ProcessMouseScroll(float yOffset) {
    Zoom -= yOffset;
    if (Zoom < 1.0f) Zoom = 1.0f;
    if (Zoom > 45.0f) Zoom = 45.0f;
  }
};

static Camera camera(vec3(0.0f, 4.0f, 0.0f));   // the reference's global, Voxel_Cone_Tracing.h:8

// Flattened Model (Model.h / Mesh.h): what Model("...obj") produces after assimp, as plain arrays.
struct Vertex { float Position[3], Normal[3], TexCoords[2], Tangents[3], Bi_Tangents[3]; };   // Mesh.h:12-19, 56 bytes
struct TextureImage { int width, height, channels; std::vector<uint8_t> pixels; };
struct MaterialRef { int diffuse, specular, height; float shininess; };
struct Model {
  std::vector<Vertex> vertices;
  std::vector<unsigned int> indices;        // 3 per triangle
  std::vector<uint16_t> triangle_material;  // optional, one per triangle
  std::vector<TextureImage> textures;
  std::vector<MaterialRef> materials;
};

struct Voxel_Cone_Tracing {
  // Global Properties
  vec3 lightDirection = vec3(0.0f, 1.0f, 0.25f);
  int VoxelDimensions = 128;
  float VoxelGridWorldSize = 150.0f;

  void* window = nullptr;
  int screen_width = 1280;
  int screen_height = 720;

  // the three Shader objects + FBO / texture ids of the reference collapse into one device context
  vct_handle device = nullptr;
  unsigned int ShadowMapSize = 4096;

  // Matrix
  mat4 DepthViewProjectionMatrix, ProjX, ProjY, ProjZ;

  Model model;

  bool ShowDiffuse = true, ShowIndirectDiffuse = true, ShowSpecular = true, ShowIndirectSpecular = true, ShowAmbientOcclusion = true;
  float AmbientFactor = 0.1f;
  int CoveragePolicy = 1;   // 0 CENTER, 1 MSAA4_ANY (the reference's 4x MSAA window, main.cpp:30), 2 CONSERVATIVE

  Voxel_Cone_Tracing() {}
  Voxel_Cone_Tracing(int screen_width_, int screen_height_, void* window_, int cuda_device = 0) {
    screen_width = screen_width_;
    screen_height = screen_height_;
    window = window_;
    check(vct_create(cuda_device, &device));
  }
  ~Voxel_Cone_Tracing() { if (device) vct_destroy(device); }
  Voxel_Cone_Tracing(const Voxel_Cone_Tracing&) = delete;
  Voxel_Cone_Tracing& operator=(const Voxel_Cone_Tracing&) = delete;

  void check(int rc) const {
    if (rc != VCT_OK) throw std::runtime_error(std::string("vct: ") + vct_last_error(device));
  }

  void init_voxel_cone_tracing(const Model& m) {
    ShadowMapSize = 4096;
    model = m;
    if (!device) check(vct_create(0, &device));
    // upload replaces Mesh::setup_Mesh (Mesh.h:49-82) and TextureFromFile (Model.h:141-186)
    for (size_t i = 0; i < model.textures.size(); ++i) {
      const TextureImage& t = model.textures[i];
      check(vct_upload_texture(device, (int)i, t.width, t.height, t.channels, t.pixels.data()));
    }
    for (size_t i = 0; i < model.materials.size(); ++i) {
      const MaterialRef& r = model.materials[i];
      check(vct_set_material(device, (int)i, r.diffuse, r.specular, r.height, r.shininess));
    }
    check(vct_upload_mesh(device, &model.vertices[0].Position[0], model.vertices.size(), model.indices.data(),
                          model.indices.size() / 3, model.triangle_material.empty() ? nullptr : model.triangle_material.data()));

    mat4 vMat = vctm::lookAt(lightDirection, vec3(0.0f, 0.0f, 0.0f), vec3(0.0f, 1.0f, 0.0f));
    mat4 pMat = vctm::ortho(-120, 120, -120, 120, -100, 100);
    DepthViewProjectionMatrix = pMat * vMat;
    check(vct_set_i(device, "ShadowMapSize", (int)ShadowMapSize));
    check(vct_set_i(device, "VoxelDimensions", VoxelDimensions));

    float size = VoxelGridWorldSize;
    mat4 voxelize_pMat = vctm::ortho(-size * 0.5f, size * 0.5f, -size * 0.5f, size * 0.5f, size * 0.5f, size * 1.5f);
    ProjX = voxelize_pMat * vctm::lookAt(vec3(size, 0.0f, 0.0f), vec3(0.0f, 0.0f, 0.0f), vec3(0.0f, 1.0f, 0.0f));
    ProjY = voxelize_pMat * vctm::lookAt(vec3(0.0f, size, 0.0f), vec3(0.0f, 0.0f, 0.0f), vec3(0.0f, 0.0f, -1.0f));
    ProjZ = voxelize_pMat * vctm::lookAt(vec3(0.0f, 0.0f, size), vec3(0.0f, 0.0f, 0.0f), vec3(0.0f, 1.0f, 0.0f));

    DrawDepthTexture();
    DrawVoxelTexture();
  }

  // host_rgba: optional H*W*4 buffer that receives the frame (the reference presents it with glfwSwapBuffers)
  void Render(uint8_t* host_rgba = nullptr) {
    SetRenderUniforms();
    check(vct_render(device, host_rgba));      // model.Draw(VoxelConeTracingShader)
  }

  // voxel view (no reference counterpart): mip `level` of the voxel pyramid drawn as cubes from the camera of Render()
  void RenderVoxels(int level, uint8_t* host_rgba = nullptr) {
    SetRenderUniforms();
    check(vct_render_voxels(device, level, host_rgba, nullptr));
  }

  // irradiance probes (no reference counterpart): indirect light and occlusion of the current pyramid at n world points
  // (xyz: n*3) for a surface facing +X, -X, +Y, -Y, +Z, -Z; out: n*6*4 (r, g, b, occlusion), steps: n*6 or NULL
  void BakeProbes(const float* xyz, size_t n, float* out, uint32_t* steps = nullptr) {
    check(vct_bake_probes(device, n, xyz, out, steps, 0));
  }

  // ray casts (no reference counterpart): the first occupied texel of mip `level` of the current pyramid along n
  // world-space segments (segments: n*6, a.xyz b.xyz); voxel: n texel indices (0xFFFFFFFF = miss); t, face (1..6 =
  // +X, -X, +Y, -Y, +Z, -Z), rgba (n*4) and steps may be NULL
  void CastRays(int level, const float* segments, size_t n, uint32_t* voxel, float* t = nullptr, uint8_t* face = nullptr,
                uint8_t* rgba = nullptr, uint32_t* steps = nullptr) {
    check(vct_cast_rays(device, level, n, segments, voxel, t, face, rgba, steps, 0));
  }

  // the uniform block of Render() (Voxel_Cone_Tracing.h:161-187), separated so that a sharded frame can set it too
  void SetRenderUniforms() {
    mat4 vMat = camera.GetViewMatrix();
    mat4 pMat = vctm::perspective(vctm::radians(camera.Zoom), (float)screen_width / (float)screen_height, 0.1f, 1000.0f);
    vec3 camera_Position = camera.position;
    check(vct_set_i(device, "screen_width", screen_width));
    check(vct_set_i(device, "screen_height", screen_height));
    check(vct_set_3f(device, "CameraPosition", camera_Position.x, camera_Position.y, camera_Position.z));
    check(vct_set_3f(device, "LightDirection", lightDirection.x, lightDirection.y, lightDirection.z));
    check(vct_set_f(device, "VoxelGridWorldSize", VoxelGridWorldSize));
    check(vct_set_i(device, "VoxelDimensions", VoxelDimensions));
    check(vct_set_f(device, "ambientFactor", AmbientFactor));
    check(vct_set_i(device, "ShadowMapSize", (int)ShadowMapSize));
    check(vct_set_i(device, "ShadowMap", 5));
    check(vct_set_i(device, "VoxelTexture", 6));
    mat4 mMat = vctm::translate(vctm::scale(mat4(1.0f), vec3(0.05f, 0.05f, 0.05f)), vec3(0.0f, 0.0f, 0.0f));
    check(vct_set_mat4(device, "ModelMatrix", mMat.data()));
    check(vct_set_mat4(device, "ModelViewMatrix", (vMat * mMat).data()));
    check(vct_set_mat4(device, "ProjectionMatrix", pMat.data()));
    check(vct_set_mat4(device, "DepthModelViewProjectionMatrix", (DepthViewProjectionMatrix * mMat).data()));
  }

  void DrawDepthTexture() {
    mat4 mMat = vctm::translate(vctm::scale(mat4(1.0f), vec3(0.05f, 0.05f, 0.05f)), vec3(0.0f, 0.0f, 0.0f));
    check(vct_set_mat4(device, "DepthModelViewProjectionMatrix", (DepthViewProjectionMatrix * mMat).data()));
    check(vct_draw_depth(device));             // model.Draw(ShadowShader)
  }

  void DrawVoxelTexture() {
    check(vct_set_i(device, "VoxelDimensions", VoxelDimensions));
    check(vct_set_mat4(device, "ProjX", ProjX.data()));
    check(vct_set_mat4(device, "ProjY", ProjY.data()));
    check(vct_set_mat4(device, "ProjZ", ProjZ.data()));
    check(vct_set_i(device, "ShadowMap", 5));
    check(vct_set_i(device, "VoxelTexture", 6));
    mat4 mMat = vctm::translate(vctm::scale(mat4(1.0f), vec3(0.05f, 0.05f, 0.05f)), vec3(0.0f, 0.0f, 0.0f));
    check(vct_set_mat4(device, "ModelMatrix", mMat.data()));
    check(vct_set_mat4(device, "DepthModelViewProjectionMatrix", (DepthViewProjectionMatrix * mMat).data()));
    check(vct_set_i(device, "ShadowMapSize", (int)ShadowMapSize));
    check(vct_set_i(device, "CoveragePolicy", CoveragePolicy));
    check(vct_draw_voxels(device));            // model.Draw(VoxelizeShader) + glGenerateMipmap(GL_TEXTURE_3D)
  }
};

// Several GPUs, one host thread: one Voxel_Cone_Tracing per device, joined by the library's own multi-GPU layer
// (vct_comm_init_multi: symmetric segments + NVSwitch multicast + device-side barriers).  Render() produces ONE frame:
// every device voxelises its share of the triangles, exchanges the voxels it touched, traces its band of rows and
// writes it into device 0's frame; the assembled frame arrives in host_rgba.  Unlike the single-GPU Render(), the
// sharded frame re-voxelises every time (it is the reference's whole loop body, main.cpp:81-92, for dynamic scenes).
struct Voxel_Cone_Tracing_Sharded {
  std::vector<Voxel_Cone_Tracing*> ranks;
  std::vector<vct_handle> handles;

  Voxel_Cone_Tracing_Sharded(int screen_width, int screen_height, const std::vector<int>& cuda_devices) {
    for (int d : cuda_devices) ranks.push_back(new Voxel_Cone_Tracing(screen_width, screen_height, nullptr, d));
    for (auto* r : ranks) handles.push_back(r->device);
  }
  ~Voxel_Cone_Tracing_Sharded() { for (auto* r : ranks) delete r; }
  Voxel_Cone_Tracing_Sharded(const Voxel_Cone_Tracing_Sharded&) = delete;
  Voxel_Cone_Tracing_Sharded& operator=(const Voxel_Cone_Tracing_Sharded&) = delete;

  void init_voxel_cone_tracing(const Model& m, int VoxelDimensions) {
    for (auto* r : ranks) {
      r->VoxelDimensions = VoxelDimensions;
      r->init_voxel_cone_tracing(m);
      r->SetRenderUniforms();            // the segment is sized from VoxelDimensions and the screen size
    }
    if (vct_comm_init_multi(handles.data(), (int)handles.size(), 0) != VCT_OK) ranks[0]->check(VCT_ERR_STATE);
  }

  void Render(uint8_t* host_rgba) {
    for (auto* r : ranks) r->SetRenderUniforms();
    if (vct_frame_sharded_multi(handles.data(), (int)handles.size(), host_rgba) != VCT_OK) ranks[0]->check(VCT_ERR_STATE);
    for (auto* r : ranks) r->check(vct_frame_sharded_wait(r->device));
  }
};

#endif  // !_VOXEL_CONE_TRACING_H_
