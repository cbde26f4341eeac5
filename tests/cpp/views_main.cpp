// A program that renders the frames of a turntable: the camera orbits the scene's lookat about the vertical axis.
// "loop" renders frame after frame with camera::render, "batch" renders all of them with one rtb200::render_views call;
// both must write the same files and the same stdout.  Used by the GPU test of render_views and tools/views_bench.py.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <memory>
#include <string>
#include <vector>

#include "common/rtweekend.hpp"
#include "accelerator/bvh_node.hpp"
#include "core/camera.hpp"
#include "core/material.hpp"
#include "core/texture.hpp"
#include "hittable/hittable.hpp"
#include "hittable/hittable_list.hpp"
#include "hittable/sphere.hpp"
#include "hittable/quad.hpp"
#include "scenes.hpp"

int main(int argc, char* argv[]) {
  if (argc < 7) {
    fprintf(stderr, "usage: views <scene> <out prefix> <width> <spp> <frames> loop|batch\n");
    return 2;
  }
  const int frames = atoi(argv[5]);
  const bool batch = std::strcmp(argv[6], "batch") == 0;
  rtb200_scenes::scene_setup s;
  if (!rtb200_scenes::build_scene(argv[1], s)) return 2;
  if (atoi(argv[3]) > 0) s.cam.image_width = atoi(argv[3]);
  if (atoi(argv[4]) > 0) s.cam.samples_per_pixel = atoi(argv[4]);

  std::vector<camera> cams(size_t(frames), s.cam);
  std::vector<std::string> paths;
  for (int i = 0; i < frames; i++) {
    const double a = 2.0 * pi * i / frames, c = std::cos(a), sn = std::sin(a);
    const vec3 r = s.cam.lookfrom - s.cam.lookat;
    cams[size_t(i)].lookfrom = s.cam.lookat + vec3(c * r.x() + sn * r.z(), r.y(), -sn * r.x() + c * r.z());
    char name[32];
    std::snprintf(name, sizeof name, "_%03d.ppm", i);
    paths.push_back(std::string(argv[2]) + name);
  }
  std::vector<std::unique_ptr<std::ofstream>> files;
  for (const std::string& p : paths) {
    files.emplace_back(new std::ofstream(p.c_str()));
    if (!*files.back()) {
      fprintf(stderr, "Error: could not open file %s for writing.\n", p.c_str());
      return 1;
    }
  }
  if (batch) {
    std::vector<const camera*> cp;
    std::vector<std::ostream*> outs;
    for (int i = 0; i < frames; i++) cp.push_back(&cams[size_t(i)]), outs.push_back(files[size_t(i)].get());
    rtb200::render_views(s.world, cp, outs);
  } else {
    for (int i = 0; i < frames; i++) cams[size_t(i)].render(*files[size_t(i)], s.world);
  }
  for (auto& f : files) f->close();
  return 0;
}
