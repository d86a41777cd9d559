// facade_demo.cpp -- the reference's main.cpp:23-94 with the window stripped: construct, init, render a few frames.
// Builds a small Cornell-style room in code, renders it through the C++ facade and prints a checksum per frame.
// Needs a CUDA device to run; compiling and linking it is part of build().
//   facade_demo [dump_dir]   with a directory: also writes the flattened scene (verts.f32, idx.u32, trimat.u16), the
//   uniforms of every frame (uniforms_<f>.f32: ModelView, Projection, DepthMVP, ProjX, ProjY, ProjZ, camera) and the
//   frames (frame_<f>.rgba), voxel views of mip level 1 (voxels_<f>.rgba) and, after the frames, the irradiance probes
//   of the cell centres of an 8x8x8 lattice over the grid (probe_xyz.f32, probes.f32) and the level-0 ray casts of a
//   fan of 16x16 segments from the grid's centre to the cell centres of its -Z face (rays_seg.f32, rays_voxel.u32,
//   rays_t.f32), so that a test can replay the same inputs through another binding and compare bytes.
//   facade_demo <dump_dir> sharded [second_device]   also renders the views as sharded frames over two ranks.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "Voxel_Cone_Tracing.h"

static void add_quad(Model& m, const float p[4][3], int mat) {
  unsigned base = (unsigned)m.vertices.size();
  float e1[3], e2[3], n[3];
  for (int k = 0; k < 3; ++k) { e1[k] = p[1][k] - p[0][k]; e2[k] = p[3][k] - p[0][k]; }
  n[0] = e1[1] * e2[2] - e1[2] * e2[1]; n[1] = e1[2] * e2[0] - e1[0] * e2[2]; n[2] = e1[0] * e2[1] - e1[1] * e2[0];
  float ln = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]), l1 = std::sqrt(e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]),
        l2 = std::sqrt(e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2]);
  const float uv[4][2] = {{0, 0}, {1, 0}, {1, 1}, {0, 1}};
  for (int v = 0; v < 4; ++v) {
    Vertex x{};
    for (int k = 0; k < 3; ++k) {
      x.Position[k] = p[v][k] * 20.0f;   // model units: the reference draws with ModelMatrix = scale(0.05)
      x.Normal[k] = n[k] / ln; x.Tangents[k] = e1[k] / l1; x.Bi_Tangents[k] = e2[k] / l2;
    }
    x.TexCoords[0] = uv[v][0]; x.TexCoords[1] = uv[v][1];
    m.vertices.push_back(x);
  }
  const unsigned idx[6] = {0, 1, 2, 0, 2, 3};
  for (unsigned i : idx) m.indices.push_back(base + i);
  m.triangle_material.push_back((uint16_t)mat);
  m.triangle_material.push_back((uint16_t)mat);
}

static void dump(const std::string& path, const void* p, size_t bytes) {
  if (FILE* f = std::fopen(path.c_str(), "wb")) { std::fwrite(p, 1, bytes, f); std::fclose(f); }
}

int main(int argc, char** argv) {
  const std::string dir = argc > 1 ? std::string(argv[1]) + "/" : std::string();
  Model m;
  const float s = 60.0f;
  const float floor_[4][3] = {{-s, -s, s}, {s, -s, s}, {s, -s, -s}, {-s, -s, -s}};
  const float back[4][3] = {{-s, -s, -s}, {s, -s, -s}, {s, s, -s}, {-s, s, -s}};
  const float left[4][3] = {{-s, -s, s}, {-s, -s, -s}, {-s, s, -s}, {-s, s, s}};
  const float right[4][3] = {{s, -s, -s}, {s, -s, s}, {s, s, s}, {s, s, -s}};
  add_quad(m, floor_, 0); add_quad(m, back, 0); add_quad(m, left, 1); add_quad(m, right, 2);
  m.textures = {{1, 1, 3, {200, 200, 200}}, {1, 1, 3, {200, 30, 30}}, {1, 1, 3, {30, 200, 30}}, {1, 1, 1, {128}}, {1, 1, 3, {128, 128, 128}}};
  m.materials = {{0, 3, 4, 20.0f}, {1, 3, 4, 20.0f}, {2, 3, 4, 20.0f}};

  try {
    Voxel_Cone_Tracing voxel_cone_tracing(256, 256, nullptr);
    voxel_cone_tracing.VoxelDimensions = 64;
    camera = Camera(vec3(0.0f, 0.0f, 205.0f));
    voxel_cone_tracing.init_voxel_cone_tracing(m);
    if (!dir.empty()) {
      dump(dir + "verts.f32", m.vertices.data(), m.vertices.size() * sizeof(Vertex));
      dump(dir + "idx.u32", m.indices.data(), m.indices.size() * sizeof(unsigned));
      dump(dir + "trimat.u16", m.triangle_material.data(), m.triangle_material.size() * sizeof(uint16_t));
    }
    std::vector<uint8_t> frame(256 * 256 * 4), view(256 * 256 * 4);
    for (int f = 0; f < 3; ++f) {
      camera.Yaw = -90.0f + 2.0f * f;
      voxel_cone_tracing.Render(frame.data());
      unsigned long long sum = 0;
      for (uint8_t b : frame) sum += b;
      std::printf("frame %d checksum %llu\n", f, sum);
      if (!dir.empty()) {
        const mat4 mMat = vctm::scale(mat4(1.0f), vec3(0.05f, 0.05f, 0.05f));
        const mat4 mv = camera.GetViewMatrix() * mMat, pr = vctm::perspective(vctm::radians(camera.Zoom), 1.0f, 0.1f, 1000.0f),
                   dm = voxel_cone_tracing.DepthViewProjectionMatrix * mMat;
        std::vector<float> u;
        const mat4* mats[6] = {&mv, &pr, &dm, &voxel_cone_tracing.ProjX, &voxel_cone_tracing.ProjY, &voxel_cone_tracing.ProjZ};
        for (const mat4* q : mats)
          u.insert(u.end(), q->data(), q->data() + 16);
        u.push_back(camera.position.x); u.push_back(camera.position.y); u.push_back(camera.position.z);
        dump(dir + "uniforms_" + std::to_string(f) + ".f32", u.data(), u.size() * sizeof(float));
        dump(dir + "frame_" + std::to_string(f) + ".rgba", frame.data(), frame.size());
        voxel_cone_tracing.RenderVoxels(1, view.data());
        dump(dir + "voxels_" + std::to_string(f) + ".rgba", view.data(), view.size());
      }
    }
    if (!dir.empty()) {
      const int k = 8;
      const float G = voxel_cone_tracing.VoxelGridWorldSize, cell = G / (float)k;
      std::vector<float> xyz, probes((size_t)k * k * k * 6 * 4);
      for (int z = 0; z < k; ++z)
        for (int y = 0; y < k; ++y)
          for (int x = 0; x < k; ++x) {
            xyz.push_back(((float)x + 0.5f) * cell - 0.5f * G);
            xyz.push_back(((float)y + 0.5f) * cell - 0.5f * G);
            xyz.push_back(((float)z + 0.5f) * cell - 0.5f * G);
          }
      voxel_cone_tracing.BakeProbes(xyz.data(), (size_t)k * k * k, probes.data());
      dump(dir + "probe_xyz.f32", xyz.data(), xyz.size() * sizeof(float));
      dump(dir + "probes.f32", probes.data(), probes.size() * sizeof(float));
      const int r = 16;
      const float rcell = G / (float)r;
      std::vector<float> seg;
      for (int y = 0; y < r; ++y)
        for (int x = 0; x < r; ++x) {
          const float b[3] = {((float)x + 0.5f) * rcell - 0.5f * G, ((float)y + 0.5f) * rcell - 0.5f * G, -0.5f * G};
          seg.insert(seg.end(), {0.0f, 0.0f, 0.0f, b[0], b[1], b[2]});
        }
      std::vector<uint32_t> ray_voxel((size_t)r * r);
      std::vector<float> ray_t((size_t)r * r);
      voxel_cone_tracing.CastRays(0, seg.data(), (size_t)r * r, ray_voxel.data(), ray_t.data());
      dump(dir + "rays_seg.f32", seg.data(), seg.size() * sizeof(float));
      dump(dir + "rays_voxel.u32", ray_voxel.data(), ray_voxel.size() * sizeof(uint32_t));
      dump(dir + "rays_t.f32", ray_t.data(), ray_t.size() * sizeof(float));
    }
    // The same three views as ONE sharded frame stream over two ranks (two GPUs if the machine has them, else two
    // handles on GPU 0): the frames must equal the single-GPU ones byte for byte.
    if (argc > 2 && std::string(argv[2]) == "sharded") {
      const int second = std::atoi(argc > 3 ? argv[3] : "0");
      Voxel_Cone_Tracing_Sharded sharded(256, 256, {0, second});
      sharded.init_voxel_cone_tracing(m, 64);
      std::vector<uint8_t> single(256 * 256 * 4), both(256 * 256 * 4);
      for (int f = 0; f < 3; ++f) {
        camera.Yaw = -90.0f + 2.0f * f;
        voxel_cone_tracing.Render(single.data());
        sharded.Render(both.data());
        const bool same = std::memcmp(single.data(), both.data(), single.size()) == 0;
        std::printf("sharded frame %d over devices {0,%d}: %s\n", f, second, same ? "identical" : "DIFFERENT");
        if (!same) return 2;
      }
    }
  } catch (const std::exception& e) {
    std::printf("error: %s\n", e.what());
    return 1;
  }
  return 0;
}
