// rtb200_host.hpp — host-side mirror of the reference's C++ scene-building API.
//
// Same class names, constructors and public members as jooo0922/raytracing-practice
// (SURVEY.md Appendix D), so scene code such as the reference's src/main.cpp compiles
// unchanged with `-I raytracing-practice_b200/host`.  The difference: these classes only
// RECORD parameters.  There is no CPU intersection / shading code here — camera::render
// flattens the shared_ptr graph into the POD arrays of include/rt_b200.h and hands them
// to the CUDA library (rt_upload_scene / rt_render / rt_download).  No CPU fallback.
//
// Arithmetic that decides scene CONTENT (rand() draws, bounding boxes, BVH topology) is
// done in double with the reference's operation order, so that the flattened scene is
// bit-identical to what the reference would have built from the same rand() stream.
#ifndef RTB200_HOST_HPP
#define RTB200_HOST_HPP

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <fstream>
#include <iostream>
#include <limits>
#include <map>
#include <memory>
#include <set>
#include <string>
#include <system_error>
#include <thread>
#include <vector>

#include "rt_b200.h"
#include "rtb200_jpeg.hpp"

// ---------------------------------------------------------------------------------------
// common/rtweekend.hpp:14-39
const double infinity = std::numeric_limits<double>::infinity();
const double pi = 3.1415926535897932385;

inline double degrees_to_radians(double degrees) { return degrees * pi / 180.0f; }

// int / float division exactly as rtweekend.hpp:26 (24-bit granularity, may return 1.0).
inline double random_double() { return std::rand() / (RAND_MAX + 1.0f); }
inline double random_double(double lo, double hi) { return lo + (hi - lo) * random_double(); }
inline int random_int(int lo, int hi) { return int(random_double(lo, hi + 1)); }

// ---------------------------------------------------------------------------------------
// common/vec3.hpp:8-226.  Division is "multiply by 1/t" as in the reference (:55,:133).
class vec3 {
 public:
  double e[3];
  vec3() : e{0, 0, 0} {}
  vec3(double a, double b, double c) : e{a, b, c} {}
  double x() const { return e[0]; }
  double y() const { return e[1]; }
  double z() const { return e[2]; }
  vec3 operator-() const { return vec3(-e[0], -e[1], -e[2]); }
  double operator[](int i) const { return e[i]; }
  double& operator[](int i) { return e[i]; }
  vec3& operator+=(const vec3& o) {
    for (int i = 0; i < 3; i++) e[i] += o.e[i];
    return *this;
  }
  vec3& operator*=(double t) {
    for (int i = 0; i < 3; i++) e[i] *= t;
    return *this;
  }
  vec3& operator/=(double t) { return *this *= 1 / t; }
  double length_squared() const { return e[0] * e[0] + e[1] * e[1] + e[2] * e[2]; }
  double length() const { return std::sqrt(length_squared()); }
  bool near_zero() const {  // the intended test (the reference's :76 has a paren slip)
    const double s = 1e-8;
    return std::fabs(e[0]) < s && std::fabs(e[1]) < s && std::fabs(e[2]) < s;
  }
  // Same expression shape as vec3.hpp:82,87 so the compiler orders the three rand()
  // draws the same way it does for the reference (g++: right to left).
  static vec3 random() { return vec3(random_double(), random_double(), random_double()); }
  static vec3 random(double lo, double hi) {
    return vec3(random_double(lo, hi), random_double(lo, hi), random_double(lo, hi));
  }
};
using point3 = vec3;
using color = vec3;

inline std::ostream& operator<<(std::ostream& o, const vec3& v) {
  return o << v.e[0] << ' ' << v.e[1] << ' ' << v.e[2];
}
inline vec3 operator+(const vec3& a, const vec3& b) { return vec3(a.e[0] + b.e[0], a.e[1] + b.e[1], a.e[2] + b.e[2]); }
inline vec3 operator-(const vec3& a, const vec3& b) { return vec3(a.e[0] - b.e[0], a.e[1] - b.e[1], a.e[2] - b.e[2]); }
inline vec3 operator*(const vec3& a, const vec3& b) { return vec3(a.e[0] * b.e[0], a.e[1] * b.e[1], a.e[2] * b.e[2]); }
inline vec3 operator*(double t, const vec3& v) { return vec3(t * v.e[0], t * v.e[1], t * v.e[2]); }
inline vec3 operator*(const vec3& v, double t) { return t * v; }
inline vec3 operator/(vec3 v, double t) { return (1 / t) * v; }
inline double dot(const vec3& a, const vec3& b) { return a.e[0] * b.e[0] + a.e[1] * b.e[1] + a.e[2] * b.e[2]; }
inline vec3 cross(const vec3& a, const vec3& b) {
  return vec3(a.e[1] * b.e[2] - a.e[2] * b.e[1], a.e[2] * b.e[0] - a.e[0] * b.e[2],
              a.e[0] * b.e[1] - a.e[1] * b.e[0]);
}
inline vec3 unit_vector(vec3 v) { return v / v.length(); }
inline vec3 random_in_unit_disk() {
  for (;;) {
    vec3 p = vec3(random_double(-1.0f, 1.0f), random_double(-1.0f, 1.0f), 0.0f);
    if (p.length_squared() < 1.0f) return p;
  }
}
inline vec3 random_unit_vector() {
  for (;;) {
    vec3 p = vec3::random(-1, 1);
    double l2 = p.length_squared();
    if (1e-160 < l2 && l2 <= 1) return p / std::sqrt(l2);
  }
}
inline vec3 random_on_hemisphere(const vec3& n) {
  vec3 s = random_unit_vector();
  return dot(s, n) > 0.0f ? s : -s;
}
inline vec3 reflect(const vec3& v, const vec3& n) { return v - 2.0f * dot(v, n) * n; }
inline vec3 refract(const vec3& uv, const vec3& n, double eta_ratio) {
  double c = std::fmin(dot(-uv, n), 1.0f);
  vec3 perp = eta_ratio * (uv + c * n);
  vec3 par = -std::sqrt(std::fabs(1.0f - perp.length_squared())) * n;
  return perp + par;
}

// common/ray.hpp:7-32
class ray {
 public:
  ray() {}
  ray(const point3& o, const vec3& d, double t) : orig(o), dir(d), tm(t) {}
  ray(const point3& o, const vec3& d) : ray(o, d, 0.0f) {}
  point3 origin() const { return orig; }
  vec3 direction() const { return dir; }
  double time() const { return tm; }
  point3 at(double t) const { return orig + t * dir; }

 private:
  point3 orig;
  vec3 dir;
  double tm = 0;
};

// common/interval.hpp:10-80
class interval {
 public:
  double min, max;
  interval() : min(+infinity), max(-infinity) {}
  interval(double lo, double hi) : min(lo), max(hi) {}
  interval(const interval& a, const interval& b)
      : min(a.min <= b.min ? a.min : b.min), max(a.max >= b.max ? a.max : b.max) {}
  double size() const { return max - min; }
  bool contains(double x) const { return min <= x && x <= max; }
  bool surrounds(double x) const { return min < x && x < max; }
  double clamp(double x) const { return x < min ? min : (x > max ? max : x); }
  interval expand(double delta) const {
    double pad = delta / 2.0f;
    return interval(min - pad, max + pad);
  }
  static const interval empty, universe;
};
inline interval operator+(const interval& i, double d) { return interval(i.min + d, i.max + d); }
inline interval operator+(double d, const interval& i) { return i + d; }
// One definition per program in C++11 (the reference's rule too: the whole API is a
// single-TU header set, interval.hpp:79-80); `inline` variables from C++17 on.
#if __cplusplus >= 201703L
#define RTB200_INLINE_VAR inline
#else
#define RTB200_INLINE_VAR
#endif
RTB200_INLINE_VAR const interval interval::empty = interval(+infinity, -infinity);
RTB200_INLINE_VAR const interval interval::universe = interval(-infinity, +infinity);

// common/color.hpp:14-58
inline double linear_to_gamma(double x) { return x > 0.0f ? std::sqrt(x) : 0.0f; }
inline void write_color(std::ostream& out, const color& c) {
  const interval intensity(0.000f, 0.999f);
  int r = int(256 * intensity.clamp(linear_to_gamma(c.x())));
  int g = int(256 * intensity.clamp(linear_to_gamma(c.y())));
  int b = int(256 * intensity.clamp(linear_to_gamma(c.z())));
  out << r << ' ' << g << ' ' << b << '\n';
}

// ---------------------------------------------------------------------------------------
// accelerator/aabb.hpp:12-173 — only construction (padding rules) is needed on the host.
class aabb {
 public:
  interval x, y, z;
  aabb() {}
  aabb(const interval& ix, const interval& iy, const interval& iz) : x(ix), y(iy), z(iz) { pad_to_minimums(); }
  aabb(const point3& a, const point3& b) {
    x = (a[0] <= b[0]) ? interval(a[0], b[0]) : interval(b[0], a[0]);
    y = (a[1] <= b[1]) ? interval(a[1], b[1]) : interval(b[1], a[1]);
    z = (a[2] <= b[2]) ? interval(a[2], b[2]) : interval(b[2], a[2]);
    pad_to_minimums();
  }
  aabb(const aabb& a, const aabb& b) : x(a.x, b.x), y(a.y, b.y), z(a.z, b.z) {}  // no re-pad (:42-48)
  const interval& axis_interval(int n) const { return n == 1 ? y : (n == 2 ? z : x); }
  int longest_axis() const {  // ties go to the later axis (:116-127)
    if (x.size() > y.size()) return x.size() > z.size() ? 0 : 2;
    return y.size() > z.size() ? 1 : 2;
  }
  static const aabb empty, universe;

 private:
  void pad_to_minimums() {
    const double delta = 0.0001;
    if (x.size() < delta) x = x.expand(delta);
    if (y.size() < delta) y = y.expand(delta);
    if (z.size() < delta) z = z.expand(delta);
  }
};
RTB200_INLINE_VAR const aabb aabb::empty = aabb(interval::empty, interval::empty, interval::empty);
RTB200_INLINE_VAR const aabb aabb::universe = aabb(interval::universe, interval::universe, interval::universe);
inline aabb operator+(const aabb& b, const vec3& o) { return aabb(b.x + o.x(), b.y + o.y(), b.z + o.z()); }
inline aabb operator+(const vec3& o, const aabb& b) { return b + o; }

// ---------------------------------------------------------------------------------------
// The flattener: walks the graph once and fills the POD arrays of include/rt_b200.h.
namespace rtb200 {

class scene_builder {
 public:
  std::vector<rt_hittable> hittables;
  std::vector<int32_t> child_index;
  std::vector<rt_material> materials;
  std::vector<rt_texture> textures;
  std::vector<rt_image> images;
  std::vector<rt_perlin> perlins;
  std::vector<std::vector<uint8_t>> image_storage;
  int32_t n_prims = 0;
  int32_t root = -1;

  // memoised by object address: shared nodes are emitted (and numbered) once.
  std::map<const void*, int32_t> seen_hittable, seen_material, seen_texture;

  int32_t new_hittable(const void* key, int32_t kind, const aabb& box) {
    rt_hittable h;
    std::memset(&h, 0, sizeof h);
    h.kind = kind;
    h.material = h.child0 = h.child1 = h.prim_id = -1;
    h.bbox[0] = box.x.min, h.bbox[1] = box.x.max;
    h.bbox[2] = box.y.min, h.bbox[3] = box.y.max;
    h.bbox[4] = box.z.min, h.bbox[5] = box.z.max;
    hittables.push_back(h);
    int32_t id = int32_t(hittables.size()) - 1;
    seen_hittable[key] = id;
    return id;
  }

  rt_scene_desc desc() const {
    rt_scene_desc d;
    std::memset(&d, 0, sizeof d);
    d.abi_version = RT_B200_ABI_VERSION;
    d.root = root;
    d.n_hittables = int32_t(hittables.size());
    d.n_child_index = int32_t(child_index.size());
    d.n_materials = int32_t(materials.size());
    d.n_textures = int32_t(textures.size());
    d.n_images = int32_t(images.size());
    d.n_perlins = int32_t(perlins.size());
    d.n_prims = n_prims;
    d.hittables = hittables.data();
    d.child_index = child_index.data();
    d.materials = materials.data();
    d.textures = textures.data();
    d.images = images.data();
    d.perlins = perlins.data();
    return d;
  }
};

[[noreturn]] inline void no_cpu_path(const char* what) {
  std::fprintf(stderr,
               "rtb200: %s was called on the host, but this build has no CPU rendering path "
               "(the hot path runs on the GPU behind camera::render).\n",
               what);
  std::abort();
}

}  // namespace rtb200

// ---------------------------------------------------------------------------------------
// core/rtw_stb_image.hpp:28-178.  stb_image is not vendored by the reference (FetchContent,
// _cmake/stb.cmake:6-9) and is not available offline, so loading goes through our own
// baseline-JPEG decoder (rtb200_jpeg.hpp); binary PPM (P6) is accepted too.  The
// post-decode conventions are stb's + the reference's: linearise with pow(b/255, 2.2)
// (stb's stbi_loadf LDR->float default) then re-quantise with float_to_byte (:137-150).
class rtw_image {
 public:
  rtw_image() {}
  rtw_image(const char* image_filename) {
    std::string filename(image_filename);
    const char* imagedir = std::getenv("RTW_IMAGES");
    if (imagedir && load(std::string(imagedir) + "/" + image_filename)) return;
    if (load(filename)) return;
    std::string prefix = "images/";
    for (int up = 0; up < 7; up++) {  // images/, ../images/, ... six levels (:48-61)
      if (load(prefix + filename)) return;
      prefix = "../" + prefix;
    }
    std::cerr << "ERROR: Could not load image file '" << image_filename << "'\n";
  }
  bool load(const std::string& filename) {
    std::vector<uint8_t> rgb;
    int w = 0, h = 0;
    if (!rtb200::load_image_rgb8(filename, rgb, w, h)) return false;
    image_width = w, image_height = h;
    bdata.resize(rgb.size());
    for (size_t i = 0; i < rgb.size(); i++) {
      float f = float(std::pow(rgb[i] / 255.0f, 2.2f));  // stbi__ldr_to_hdr, gamma 2.2, scale 1
      bdata[i] = float_to_byte(f);
    }
    return true;
  }
  int width() const { return bdata.empty() ? 0 : image_width; }
  int height() const { return bdata.empty() ? 0 : image_height; }
  const unsigned char* pixel_data(int px, int py) const {
    static unsigned char magenta[] = {255, 0, 255};
    if (bdata.empty()) return magenta;
    px = clamp(px, 0, image_width);
    py = clamp(py, 0, image_height);
    return bdata.data() + size_t(py) * image_width * 3 + size_t(px) * 3;
  }
  const std::vector<uint8_t>& bytes() const { return bdata; }

 private:
  static int clamp(int v, int lo, int hi) { return v < lo ? lo : (v < hi ? v : hi - 1); }
  static unsigned char float_to_byte(float v) {
    if (v <= 0.0f) return 0;
    if (v >= 1.0f) return 255;
    return static_cast<unsigned char>(256.0f * v);
  }
  std::vector<uint8_t> bdata;
  int image_width = 0, image_height = 0;
};

// core/perlin.hpp:9-31,162-188 — table construction only (draws rand() exactly as the
// reference: 256 x unit_vector(vec3::random(-1,1)) then three Fisher-Yates permutes).
class perlin {
 public:
  static const int point_count = 256;
  perlin() {
    for (int i = 0; i < point_count; i++) randvec[i] = unit_vector(vec3::random(-1.0f, 1.0f));
    generate_perm(perm_x);
    generate_perm(perm_y);
    generate_perm(perm_z);
  }
  double noise_perlin(const point3&) const { rtb200::no_cpu_path("perlin::noise_perlin"); }
  double turb(const point3&, int) const { rtb200::no_cpu_path("perlin::turb"); }
  void export_tables(rt_perlin& out) const {
    for (int i = 0; i < point_count; i++) {
      for (int c = 0; c < 3; c++) out.randvec[i][c] = randvec[i][c];
      out.perm_x[i] = perm_x[i], out.perm_y[i] = perm_y[i], out.perm_z[i] = perm_z[i];
    }
  }

 private:
  static void generate_perm(int* p) {
    for (int i = 0; i < point_count; i++) p[i] = i;
    for (int i = point_count - 1; i > 0; i--) {
      int target = random_int(0, i);
      if (target > i) target = i;  // random_double() can return exactly 1.0 (SURVEY A.11):
                                   // the reference would read out of bounds here.
      std::swap(p[i], p[target]);
    }
  }
  vec3 randvec[point_count];
  int perm_x[point_count], perm_y[point_count], perm_z[point_count];
};

// core/texture.hpp:11-156
class texture {
 public:
  virtual ~texture() = default;
  virtual color value(double, double, const point3&) const { rtb200::no_cpu_path("texture::value"); }
  virtual int32_t flatten(rtb200::scene_builder& b) const = 0;

 protected:
  static int32_t emit(rtb200::scene_builder& b, const void* key, const rt_texture& t) {
    b.textures.push_back(t);
    return b.seen_texture[key] = int32_t(b.textures.size()) - 1;
  }
  static rt_texture blank(int32_t kind) {
    rt_texture t;
    std::memset(&t, 0, sizeof t);
    t.kind = kind;
    t.even = t.odd = t.image = t.perlin = -1;
    return t;
  }
};

inline int32_t rtb200_flatten_texture(rtb200::scene_builder& b, const texture* t) {
  auto it = b.seen_texture.find(t);
  return it != b.seen_texture.end() ? it->second : t->flatten(b);
}

class solid_color : public texture {
 public:
  solid_color(const color& a) : albedo(a) {}
  solid_color(double r, double g, double bl) : solid_color(color(r, g, bl)) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    rt_texture t = blank(RT_T_SOLID);
    for (int c = 0; c < 3; c++) t.color[c] = albedo[c];
    return emit(b, this, t);
  }

 private:
  color albedo;
};

class checker_texture : public texture {
 public:
  checker_texture(double scale, std::shared_ptr<texture> e, std::shared_ptr<texture> o)
      : inv_scale(1.0f / scale), even(e), odd(o) {}
  checker_texture(double scale, const color& c1, const color& c2)
      : checker_texture(scale, std::make_shared<solid_color>(c1), std::make_shared<solid_color>(c2)) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    rt_texture t = blank(RT_T_CHECKER);
    t.scale = inv_scale;
    t.even = rtb200_flatten_texture(b, even.get());
    t.odd = rtb200_flatten_texture(b, odd.get());
    return emit(b, this, t);
  }

 private:
  double inv_scale;
  std::shared_ptr<texture> even, odd;
};

class image_texture : public texture {
 public:
  image_texture(const char* filename) : image(filename) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    rt_texture t = blank(RT_T_IMAGE);
    b.image_storage.push_back(image.bytes());
    rt_image im;
    im.width = image.width();
    im.height = image.height();
    im.rgb = nullptr;  // patched after all storage is final (vector moves): see finalize()
    b.images.push_back(im);
    t.image = int32_t(b.images.size()) - 1;
    return emit(b, this, t);
  }

 private:
  rtw_image image;
};

class noise_texture : public texture {
 public:
  noise_texture(double s) : scale(s) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    rt_texture t = blank(RT_T_NOISE);
    t.scale = scale;
    rt_perlin p;
    noise.export_tables(p);
    b.perlins.push_back(p);
    t.perlin = int32_t(b.perlins.size()) - 1;
    return emit(b, this, t);
  }

 private:
  perlin noise;
  double scale;
};

// ---------------------------------------------------------------------------------------
// hittable/hittable.hpp:16-50
class material;
class hit_record {
 public:
  point3 p;
  vec3 normal;
  std::shared_ptr<material> mat;
  double t, u, v;
  bool front_face;
  void set_face_normal(const ray& r, const vec3& outward_normal) {
    front_face = dot(r.direction(), outward_normal) < 0;
    normal = front_face ? outward_normal : -outward_normal;
  }
};

// core/material.hpp:21-240 (+ isotropic, SURVEY.md App. B.3)
class material {
 public:
  virtual ~material() = default;
  virtual color emitted(double, double, const point3&) const { rtb200::no_cpu_path("material::emitted"); }
  virtual bool scatter(const ray&, const hit_record&, color&, ray&) const { rtb200::no_cpu_path("material::scatter"); }
  virtual int32_t flatten(rtb200::scene_builder& b) const = 0;

 protected:
  static int32_t emit(rtb200::scene_builder& b, const void* key, int32_t kind, int32_t tex, const color& albedo,
                      double fuzz, double ior) {
    rt_material m;
    std::memset(&m, 0, sizeof m);
    m.kind = kind;
    m.texture = tex;
    for (int c = 0; c < 3; c++) m.albedo[c] = albedo[c];
    m.fuzz = fuzz;
    m.ior = ior;
    b.materials.push_back(m);
    return b.seen_material[key] = int32_t(b.materials.size()) - 1;
  }
};

inline int32_t rtb200_flatten_material(rtb200::scene_builder& b, const material* m) {
  auto it = b.seen_material.find(m);
  return it != b.seen_material.end() ? it->second : m->flatten(b);
}

class lambertian : public material {
 public:
  lambertian(const color& albedo) : tex(std::make_shared<solid_color>(albedo)) {}
  lambertian(std::shared_ptr<texture> t) : tex(t) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    return emit(b, this, RT_M_LAMBERTIAN, rtb200_flatten_texture(b, tex.get()), color(), 0, 0);
  }

 private:
  std::shared_ptr<texture> tex;
};

class metal : public material {
 public:
  metal(const color& a, double f) : albedo(a), fuzz(f < 1.0f ? f : 1.0f) {}
  int32_t flatten(rtb200::scene_builder& b) const override { return emit(b, this, RT_M_METAL, -1, albedo, fuzz, 0); }

 private:
  color albedo;
  double fuzz;
};

class dielectric : public material {
 public:
  dielectric(double ri) : refraction_index(ri) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    return emit(b, this, RT_M_DIELECTRIC, -1, color(), 0, refraction_index);
  }

 private:
  double refraction_index;
};

class diffuse_light : public material {
 public:
  diffuse_light(std::shared_ptr<texture> t) : tex(t) {}
  diffuse_light(const color& emit_color) : tex(std::make_shared<solid_color>(emit_color)) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    return emit(b, this, RT_M_DIFFUSE_LIGHT, rtb200_flatten_texture(b, tex.get()), color(), 0, 0);
  }

 private:
  std::shared_ptr<texture> tex;
};

class isotropic : public material {
 public:
  isotropic(const color& albedo) : tex(std::make_shared<solid_color>(albedo)) {}
  isotropic(std::shared_ptr<texture> t) : tex(t) {}
  int32_t flatten(rtb200::scene_builder& b) const override {
    return emit(b, this, RT_M_ISOTROPIC, rtb200_flatten_texture(b, tex.get()), color(), 0, 0);
  }

 private:
  std::shared_ptr<texture> tex;
};

// ---------------------------------------------------------------------------------------
class hittable {
 public:
  virtual ~hittable() = default;
  virtual bool hit(const ray&, interval, hit_record&) const { rtb200::no_cpu_path("hittable::hit"); }
  virtual aabb bounding_box() const = 0;
  // A user subclass that is not one of the known concrete types cannot be flattened:
  // fail loudly rather than silently dropping geometry (SURVEY.md Appendix D note).
  virtual int32_t flatten(rtb200::scene_builder&) const {
    std::fprintf(stderr, "rtb200: unknown hittable subclass cannot be uploaded to the GPU\n");
    std::abort();
  }
};

inline int32_t rtb200_flatten_hittable(rtb200::scene_builder& b, const hittable* h) {
  auto it = b.seen_hittable.find(h);
  return it != b.seen_hittable.end() ? it->second : h->flatten(b);
}

// hittable/hittable.hpp:74-117
class translate : public hittable {
 public:
  translate(std::shared_ptr<hittable> obj, const vec3& off) : object(obj), offset(off) {
    bbox = object->bounding_box() + offset;
  }
  aabb bounding_box() const override { return bbox; }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_TRANSLATE, bbox);
    for (int c = 0; c < 3; c++) b.hittables[id].p[c] = offset[c];
    int32_t child = rtb200_flatten_hittable(b, object.get());
    b.hittables[id].child0 = child;
    return id;
  }

 private:
  std::shared_ptr<hittable> object;
  vec3 offset;
  aabb bbox;
};

// Not in the reference: "The Next Week" rotate_y (SURVEY.md Appendix B.1).
class rotate_y : public hittable {
 public:
  rotate_y(std::shared_ptr<hittable> obj, double angle) : object(obj), angle_degrees(angle) {
    double radians = degrees_to_radians(angle);
    sin_theta = std::sin(radians);
    cos_theta = std::cos(radians);
    bbox = object->bounding_box();
    point3 lo(infinity, infinity, infinity), hi(-infinity, -infinity, -infinity);
    for (int i = 0; i < 2; i++)
      for (int j = 0; j < 2; j++)
        for (int k = 0; k < 2; k++) {
          double px = i * bbox.x.max + (1 - i) * bbox.x.min;
          double py = j * bbox.y.max + (1 - j) * bbox.y.min;
          double pz = k * bbox.z.max + (1 - k) * bbox.z.min;
          double nx = cos_theta * px + sin_theta * pz;
          double nz = -sin_theta * px + cos_theta * pz;
          vec3 corner(nx, py, nz);
          for (int c = 0; c < 3; c++) {
            lo[c] = std::fmin(lo[c], corner[c]);
            hi[c] = std::fmax(hi[c], corner[c]);
          }
        }
    bbox = aabb(lo, hi);
  }
  aabb bounding_box() const override { return bbox; }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_ROTATE_Y, bbox);
    b.hittables[id].p[0] = angle_degrees;
    b.hittables[id].p[1] = sin_theta;
    b.hittables[id].p[2] = cos_theta;
    int32_t child = rtb200_flatten_hittable(b, object.get());
    b.hittables[id].child0 = child;
    return id;
  }

 private:
  std::shared_ptr<hittable> object;
  double angle_degrees, sin_theta, cos_theta;
  aabb bbox;
};

// hittable/hittable_list.hpp:21-76
class hittable_list : public hittable {
 public:
  std::vector<std::shared_ptr<hittable>> objects;
  hittable_list() {}
  hittable_list(std::shared_ptr<hittable> object) { add(object); }
  void clear() { objects.clear(); }
  void add(std::shared_ptr<hittable> object) {
    objects.push_back(object);
    bbox = aabb(bbox, object->bounding_box());
  }
  aabb bounding_box() const override { return bbox; }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_LIST, bbox);
    std::vector<int32_t> kids;
    for (const auto& o : objects) kids.push_back(rtb200_flatten_hittable(b, o.get()));
    b.hittables[id].child0 = int32_t(b.child_index.size());
    b.hittables[id].child1 = int32_t(kids.size());
    b.child_index.insert(b.child_index.end(), kids.begin(), kids.end());
    return id;
  }

 private:
  aabb bbox;
};

// hittable/sphere.hpp:7-119
class sphere : public hittable {
 public:
  sphere(point3 static_center, double r, std::shared_ptr<material> m)
      : center(static_center, vec3(0.0f, 0.0f, 0.0f)), radius(r), mat(m) {
    vec3 rvec(radius, radius, radius);
    bbox = aabb(static_center - rvec, static_center + rvec);
  }
  sphere(point3 c1, point3 c2, double r, std::shared_ptr<material> m) : center(c1, c2 - c1), radius(r), mat(m) {
    vec3 rvec(radius, radius, radius);
    aabb box1(center.at(0.0f) - rvec, center.at(0.0f) + rvec);
    aabb box2(center.at(1.0f) - rvec, center.at(1.0f) + rvec);
    bbox = aabb(box1, box2);
  }
  aabb bounding_box() const override { return bbox; }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_SPHERE, bbox);
    b.hittables[id].prim_id = b.n_prims++;
    for (int c = 0; c < 3; c++) {
      b.hittables[id].p[c] = center.origin()[c];
      b.hittables[id].p[3 + c] = center.direction()[c];
    }
    b.hittables[id].p[6] = radius;
    int32_t m = rtb200_flatten_material(b, mat.get());
    b.hittables[id].material = m;
    return id;
  }

 private:
  ray center;
  double radius;
  std::shared_ptr<material> mat;
  aabb bbox;
};

// hittable/quad.hpp:8-159
class quad : public hittable {
 public:
  quad(const point3& q, const vec3& eu, const vec3& ev, std::shared_ptr<material> m) : Q(q), u(eu), v(ev), mat(m) {
    vec3 n = cross(u, v);
    normal = unit_vector(n);
    D = dot(normal, Q);
    w = n / dot(n, n);
    set_bounding_box();
  }
  virtual void set_bounding_box() {
    aabb d1(Q, Q + u + v);
    aabb d2(Q + u, Q + v);
    bbox = aabb(d1, d2);
  }
  aabb bounding_box() const override { return bbox; }
  virtual bool is_interior(double a, double b, hit_record& rec) const {
    interval unit(0.0f, 1.0f);
    if (!unit.contains(a) || !unit.contains(b)) return false;
    rec.u = a, rec.v = b;
    return true;
  }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_QUAD, bbox);
    b.hittables[id].prim_id = b.n_prims++;
    for (int c = 0; c < 3; c++) {
      b.hittables[id].p[c] = Q[c];
      b.hittables[id].p[3 + c] = u[c];
      b.hittables[id].p[6 + c] = v[c];
    }
    int32_t m = rtb200_flatten_material(b, mat.get());
    b.hittables[id].material = m;
    return id;
  }

 private:
  point3 Q;
  vec3 u, v, w;
  std::shared_ptr<material> mat;
  aabb bbox;
  vec3 normal;
  double D;
};

// quad.hpp:129-159 — six sides in the order +z, +x, -z, -x, +y, -y.
inline std::shared_ptr<hittable_list> box(const point3& a, const point3& b, std::shared_ptr<material> mat) {
  auto sides = std::make_shared<hittable_list>();
  point3 lo(std::fmin(a.x(), b.x()), std::fmin(a.y(), b.y()), std::fmin(a.z(), b.z()));
  point3 hi(std::fmax(a.x(), b.x()), std::fmax(a.y(), b.y()), std::fmax(a.z(), b.z()));
  vec3 dx(hi.x() - lo.x(), 0.0f, 0.0f), dy(0.0f, hi.y() - lo.y(), 0.0f), dz(0.0f, 0.0f, hi.z() - lo.z());
  sides->add(std::make_shared<quad>(point3(lo.x(), lo.y(), hi.z()), dx, dy, mat));
  sides->add(std::make_shared<quad>(point3(hi.x(), lo.y(), hi.z()), -dz, dy, mat));
  sides->add(std::make_shared<quad>(point3(hi.x(), lo.y(), lo.z()), -dx, dy, mat));
  sides->add(std::make_shared<quad>(point3(lo.x(), lo.y(), lo.z()), dz, dy, mat));
  sides->add(std::make_shared<quad>(point3(lo.x(), hi.y(), hi.z()), dx, -dz, mat));
  sides->add(std::make_shared<quad>(point3(lo.x(), lo.y(), lo.z()), dx, dz, mat));
  return sides;
}

// Not in the reference: "The Next Week" constant_medium (SURVEY.md Appendix B.2).
class constant_medium : public hittable {
 public:
  constant_medium(std::shared_ptr<hittable> b, double density, std::shared_ptr<texture> tex)
      : boundary(b), dens(density), neg_inv_density(-1 / density), phase_function(std::make_shared<isotropic>(tex)) {}
  constant_medium(std::shared_ptr<hittable> b, double density, const color& albedo)
      : boundary(b), dens(density), neg_inv_density(-1 / density), phase_function(std::make_shared<isotropic>(albedo)) {}
  aabb bounding_box() const override { return boundary->bounding_box(); }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_MEDIUM, boundary->bounding_box());
    b.hittables[id].p[0] = dens;
    b.hittables[id].p[1] = neg_inv_density;
    int32_t child = rtb200_flatten_hittable(b, boundary.get());
    b.hittables[id].child0 = child;
    int32_t m = rtb200_flatten_material(b, phase_function.get());
    b.hittables[id].material = m;
    return id;
  }

 private:
  std::shared_ptr<hittable> boundary;
  double dens, neg_inv_density;
  std::shared_ptr<material> phase_function;
};

// accelerator/bvh_node.hpp:16-134.  The topology is kept (the CPU oracle replays the
// reference's left-then-right traversal over it); the GPU builds its own SAH tree over
// the leaves.  Same split rule and the same std::sort call as the reference, so the same
// libstdc++ produces the same tree.
class bvh_node : public hittable {
 public:
  bvh_node(hittable_list list) : bvh_node(list.objects, 0, list.objects.size()) {}
  bvh_node(std::vector<std::shared_ptr<hittable>>& objects, size_t start, size_t end) {
    bbox = aabb::empty;
    for (size_t i = start; i < end; i++) bbox = aabb(bbox, objects[i]->bounding_box());
    const int axis = bbox.longest_axis();
    const size_t span = end - start;
    if (span == 1) {
      left = right = objects[start];
    } else if (span == 2) {
      left = objects[start];
      right = objects[start + 1];
    } else {
      std::sort(std::begin(objects) + start, std::begin(objects) + end,
                axis == 0 ? before<0> : (axis == 1 ? before<1> : before<2>));
      size_t mid = start + span / 2;
      left = std::make_shared<bvh_node>(objects, start, mid);
      right = std::make_shared<bvh_node>(objects, mid, end);
    }
  }
  aabb bounding_box() const override { return bbox; }
  int32_t flatten(rtb200::scene_builder& b) const override {
    int32_t id = b.new_hittable(this, RT_H_BVH, bbox);
    int32_t l = rtb200_flatten_hittable(b, left.get());
    int32_t r = rtb200_flatten_hittable(b, right.get());
    b.hittables[id].child0 = l;
    b.hittables[id].child1 = r;
    return id;
  }

 private:
  template <int AXIS>
  static bool before(const std::shared_ptr<hittable> a, const std::shared_ptr<hittable> b) {
    return a->bounding_box().axis_interval(AXIS).min < b->bounding_box().axis_interval(AXIS).min;
  }
  std::shared_ptr<hittable> left, right;
  aabb bbox;
};

// ---------------------------------------------------------------------------------------
namespace rtb200 {

// Flatten a world into an owning scene_builder (desc() gives the C-ABI view).
inline std::unique_ptr<scene_builder> flatten_world(const hittable& world) {
  std::unique_ptr<scene_builder> b(new scene_builder);
  b->root = rtb200_flatten_hittable(*b, &world);
  for (size_t i = 0; i < b->images.size(); i++)
    b->images[i].rgb = b->image_storage[i].empty() ? nullptr : b->image_storage[i].data();
  return b;
}

}  // namespace rtb200

// ---------------------------------------------------------------------------------------
// core/camera.hpp:10-245 — same public fields, same render(std::ostream&, world) signature,
// same PPM text (header :36-37, one "r g b\n" per pixel, color.hpp:57) and the same stdout
// progress strings (:47,:70).  The pixel/sample/bounce loops run on the GPU.
class camera {
 public:
  double aspect_ratio = 1.0f;
  int image_width = 100;
  int samples_per_pixel = 10;
  int max_depth = 10;
  color background;
  double vfov = 90.0f;
  point3 lookfrom = point3(0.0f, 0.0f, 0.0f);
  point3 lookat = point3(0.0f, 0.0f, -1.0f);
  vec3 vup = vec3(0.0f, 1.0f, 0.0f);
  double defocus_angle = 0.0f;
  double focus_dist = 10.0f;

  rt_camera_desc desc() const {
    rt_camera_desc c;
    std::memset(&c, 0, sizeof c);
    c.aspect_ratio = aspect_ratio;
    c.image_width = image_width;
    c.samples_per_pixel = samples_per_pixel;
    c.max_depth = max_depth;
    c.vfov = vfov;
    c.defocus_angle = defocus_angle;
    c.focus_dist = focus_dist;
    for (int i = 0; i < 3; i++) {
      c.background[i] = background[i];
      c.lookfrom[i] = lookfrom[i];
      c.lookat[i] = lookat[i];
      c.vup[i] = vup[i];
    }
    return c;
  }

  void render(std::ostream& output_stream, const hittable& world);
};

#ifndef RTB200_NO_RENDER_IMPL
namespace rtb200 {
inline void die(rt_ctx* ctx, const char* where, int rc) {
  std::fprintf(stderr, "rtb200: %s failed (%d): %s\n", where, rc, rt_last_error(ctx));
  std::exit(1);
}
// Fast integer formatting of the P3 body: at GPU speed the iostream << of W*H lines is a
// visible share of wall time (SURVEY.md §8(f) rank 2).
inline void write_ppm_p3(std::ostream& out, int w, int h, const uint8_t* rgb) {
  out << "P3\n" << w << ' ' << h << "\n255\n";
  std::string buf;
  buf.reserve(size_t(w) * 12 * 64);
  char num[256][4];
  int len[256];
  for (int v = 0; v < 256; v++) len[v] = std::snprintf(num[v], 4, "%d", v);
  for (int j = 0; j < h; j++) {
    for (int i = 0; i < w; i++) {
      const uint8_t* p = rgb + (size_t(j) * w + i) * 3;
      buf.append(num[p[0]], len[p[0]]);
      buf.push_back(' ');
      buf.append(num[p[1]], len[p[1]]);
      buf.push_back(' ');
      buf.append(num[p[2]], len[p[2]]);
      buf.push_back('\n');
    }
    if (buf.size() > (1u << 20)) {
      out.write(buf.data(), std::streamsize(buf.size()));
      buf.clear();
    }
  }
  out.write(buf.data(), std::streamsize(buf.size()));
}
// Binary side output (SURVEY.md §8(f) rank 2): the same bytes the P3 text spells out, as a P6 file.
inline bool write_ppm_p6(const char* path, int w, int h, const uint8_t* rgb) {
  std::FILE* f = std::fopen(path, "wb");
  if (!f) return false;
  std::fprintf(f, "P6\n%d %d\n255\n", w, h);
  const size_t n = size_t(w) * h * 3;
  const bool ok = std::fwrite(rgb, 1, n, f) == n;
  return (std::fclose(f) == 0) && ok;
}

// ---- checkpointed progressive rendering (SURVEY.md §8(f) rank 4) ---------------------------------------------
// camera::render's sample loop (camera.hpp:55-61) is a plain sum, the device keeps it as exact int64 fixed-point
// sums, and sample s of pixel p draws from Philox counter (p, s, bounce): a render can therefore stop after any
// number of samples and continue later — in another process, on another number of GPUs — and the finished image
// has the bits of an uninterrupted one.  The file holds a header and the W x H x 3 int64 sums.
struct checkpoint_header {
  char magic[8];  // "RTB2CKPT"
  uint32_t version, width, height, spp_total, spp_done, max_depth;
  uint64_t seed, scene_hash;  // FNV-1a over the camera and the flattened scene description
};
inline uint64_t fnv1a(uint64_t h, const void* data, size_t bytes) {
  const unsigned char* p = static_cast<const unsigned char*>(data);
  for (size_t i = 0; i < bytes; i++) h = (h ^ p[i]) * 1099511628211ull;
  return h;
}
inline uint64_t scene_hash(const rt_scene_desc& d, const rt_camera_desc& cam) {
  uint64_t h = 1469598103934665603ull;
  h = fnv1a(h, &cam, sizeof cam);
  h = fnv1a(h, &d.root, sizeof d.root);
  h = fnv1a(h, d.hittables, size_t(d.n_hittables) * sizeof(rt_hittable));
  h = fnv1a(h, d.child_index, size_t(d.n_child_index) * sizeof(int32_t));
  h = fnv1a(h, d.materials, size_t(d.n_materials) * sizeof(rt_material));
  h = fnv1a(h, d.textures, size_t(d.n_textures) * sizeof(rt_texture));
  h = fnv1a(h, d.perlins, size_t(d.n_perlins) * sizeof(rt_perlin));
  for (int i = 0; i < d.n_images; i++) {
    h = fnv1a(h, &d.images[i].width, 4);
    h = fnv1a(h, &d.images[i].height, 4);
    if (d.images[i].rgb) h = fnv1a(h, d.images[i].rgb, size_t(d.images[i].width) * d.images[i].height * 3);
  }
  return h;
}
// Reads `path` into `sums`; returns the samples per pixel it holds, 0 when there is no file, and exits loudly when
// the file belongs to another scene / camera / sample count (continuing it would silently mix two images).
inline int checkpoint_load(const char* path, const checkpoint_header& want, std::vector<int64_t>& sums) {
  std::FILE* f = std::fopen(path, "rb");
  if (!f) return 0;
  checkpoint_header h;
  const bool head = std::fread(&h, sizeof h, 1, f) == 1;
  const bool match = head && std::memcmp(h.magic, want.magic, 8) == 0 && h.version == want.version && h.width == want.width && h.height == want.height &&
                     h.spp_total == want.spp_total && h.max_depth == want.max_depth && h.seed == want.seed && h.scene_hash == want.scene_hash &&
                     h.spp_done <= h.spp_total;
  const bool body = match && std::fread(sums.data(), 8, sums.size(), f) == sums.size();
  std::fclose(f);
  if (!body) {
    std::fprintf(stderr, "rtb200: checkpoint %s %s; remove it to start over.\n", path,
                 !head ? "is truncated" : (!match ? "was written for another scene, camera or sample count" : "is truncated"));
    std::exit(1);
  }
  return int(h.spp_done);
}
inline void checkpoint_save(const char* path, checkpoint_header h, int spp_done, const std::vector<int64_t>& sums) {
  h.spp_done = uint32_t(spp_done);
  const std::string tmp = std::string(path) + ".tmp";  // write-then-rename: a kill mid-write leaves the old file intact
  std::FILE* f = std::fopen(tmp.c_str(), "wb");
  bool ok = f != nullptr;
  if (f) {
    ok = std::fwrite(&h, sizeof h, 1, f) == 1 && std::fwrite(sums.data(), 8, sums.size(), f) == sums.size();
    ok = (std::fclose(f) == 0) && ok;
  }
  if (!ok || std::rename(tmp.c_str(), path) != 0) {
    std::fprintf(stderr, "rtb200: could not write checkpoint %s\n", path);
    std::exit(1);
  }
}
}  // namespace rtb200

namespace rtb200 {
// RT_B200_TIMING=1: camera::render prints where its wall time went (one JSON line on stderr)
struct phase_timer {
  std::chrono::steady_clock::time_point last = std::chrono::steady_clock::now();
  std::vector<std::pair<const char*, double>> parts;
  void mark(const char* name) {
    const auto now = std::chrono::steady_clock::now();
    parts.emplace_back(name, std::chrono::duration<double, std::milli>(now - last).count());
    last = now;
  }
  void report(int w, int h, int spp, int devices) const {
    const char* e = std::getenv("RT_B200_TIMING");
    if (!e || !*e || *e == '0') return;
    double total = 0;
    for (const auto& p : parts) total += p.second;
    std::fprintf(stderr, "RTB200_TIMING {\"width\": %d, \"height\": %d, \"spp\": %d, \"devices\": %d, \"total_ms\": %.3f", w, h, spp, devices, total);
    for (const auto& p : parts) std::fprintf(stderr, ", \"%s_ms\": %.3f", p.first, p.second);
    std::fprintf(stderr, "}\n");
  }
};

// The process-level context cache of camera::render: slot r of RT_B200_DEVICES keeps its rt_ctx (and, through it, its
// arena, accumulator, reduce buffer and peer mappings) until the process exits.
class context_cache {
 public:
  static context_cache& get() {
    static context_cache c;
    return c;
  }
  rt_ctx* acquire(int slot, int device) {
    if (size_t(slot) >= slots_.size()) slots_.resize(size_t(slot) + 1);
    entry& e = slots_[size_t(slot)];
    if (e.ctx && e.device != device) {  // the slot moved to another device: start over for it
      rt_shutdown(e.ctx);
      e = entry();
      for (auto it = peers_.begin(); it != peers_.end();) it = (it->first == slot || it->second == slot) ? peers_.erase(it) : std::next(it);
    }
    if (!e.ctx) {
      int rc = rt_init(device, &e.ctx);
      if (rc != RT_OK) die(nullptr, "rt_init", rc);
      e.device = device;
      // released at exit — registered AFTER the first rt_init, i.e. after the CUDA runtime registered its own exit handler,
      // so that (handlers run in reverse order) the contexts are shut down while the runtime is still up
      if (!registered_) registered_ = true, std::atexit(&context_cache::shutdown_all);
    }
    return e.ctx;
  }
  // all slots of one camera::render at once: the contexts that do not exist yet are created CONCURRENTLY, one thread per
  // device — creating a CUDA context takes 0.4-1.7 s and eight of them in a row would outlast the headline render eight times
  std::vector<rt_ctx*> acquire_all(const std::vector<int>& devices) {
    const size_t R = devices.size();
    if (slots_.size() < R) slots_.resize(R);
    std::vector<size_t> missing;
    for (size_t r = 0; r < R; r++) {
      entry& e = slots_[r];
      if (e.ctx && e.device != devices[r]) acquire(int(r), devices[r]);  // the slot moved: the serial path replaces it
      if (!slots_[r].ctx) missing.push_back(r);
    }
    if (missing.size() > 1) {
      std::vector<int> rc(R, RT_OK);
      std::vector<std::thread> workers;
      for (size_t r : missing) {
        auto job = [this, r, &devices, &rc] { rc[r] = rt_init(devices[r], &slots_[r].ctx); };
        try {
          workers.emplace_back(job);
        } catch (const std::system_error&) {  // a program linked without thread support (old glibc, no -pthread): serially
          job();
        }
      }
      for (std::thread& w : workers) w.join();
      for (size_t r : missing) {
        if (rc[r] != RT_OK) die(nullptr, "rt_init", rc[r]);
        slots_[r].device = devices[r];
      }
      if (!registered_) registered_ = true, std::atexit(&context_cache::shutdown_all);
    }
    std::vector<rt_ctx*> out(R, nullptr);
    for (size_t r = 0; r < R; r++) out[r] = acquire(int(r), devices[r]);
    return out;
  }
  static void shutdown_all() {
    context_cache& c = get();
    for (entry& e : c.slots_)
      if (e.ctx) rt_shutdown(e.ctx), e.ctx = nullptr;
    c.peers_.clear();
  }
  bool peer_enable(int slot, int with) {
    if (peers_.count({slot, with})) return true;
    if (rt_peer_enable(slots_[size_t(slot)].ctx, slots_[size_t(with)].ctx) != RT_OK) return false;
    peers_.insert({slot, with});
    return true;
  }

 private:
  bool registered_ = false;
  struct entry {
    rt_ctx* ctx = nullptr;
    int device = -1;
  };
  std::vector<entry> slots_;
  std::set<std::pair<int, int>> peers_;
};

// RT_B200_DEVICES as a list of CUDA ordinals (default {0}), at most `limit` of them (and at least one)
inline std::vector<int> device_list(int limit) {
  std::vector<int> devices;
  const char* env = std::getenv("RT_B200_DEVICES");
  std::string spec = env ? env : "0";
  for (size_t pos = 0; pos < spec.size();) {
    size_t comma = spec.find(',', pos);
    if (comma == std::string::npos) comma = spec.size();
    if (comma > pos) devices.push_back(std::atoi(spec.substr(pos, comma - pos).c_str()));
    pos = comma + 1;
  }
  if (devices.empty()) devices.push_back(0);
  if (int(devices.size()) > limit) devices.resize(size_t(std::max(1, limit)));
  return devices;
}

// The scene on every context; several are built and uploaded concurrently (rt_upload_scene is synchronous)
inline void upload_all(const std::vector<rt_ctx*>& ctx, const rt_scene_desc& sd) {
  const int R = int(ctx.size());
  if (R == 1) {
    int rc = rt_upload_scene(ctx[0], &sd);
    if (rc != RT_OK) die(ctx[0], "rt_upload_scene", rc);
    return;
  }
  std::vector<int> rcs(size_t(R), RT_OK);
  std::vector<std::thread> workers;
  for (int r = 0; r < R; r++) {
    auto job = [&, r] { rcs[size_t(r)] = rt_upload_scene(ctx[size_t(r)], &sd); };
    try {
      workers.emplace_back(job);
    } catch (const std::system_error&) {
      job();
    }
  }
  for (std::thread& w : workers) w.join();
  for (int r = 0; r < R; r++)
    if (rcs[size_t(r)] != RT_OK) die(ctx[size_t(r)], "rt_upload_scene", rcs[size_t(r)]);
}
}  // namespace rtb200

// Environment (the reference's camera has no such fields, and the drop-in keeps its class as it is):
//   RT_B200_DEVICES         comma-separated CUDA ordinals (default "0"); samples are sharded over them
//   RT_B200_P6              path of a binary P6 copy of the image
//   RT_B200_CHECKPOINT      path of a checkpoint file: resumed when present, rewritten after every pass
//   RT_B200_CHECKPOINT_SPP  samples per pixel per pass (default 256)
//   RT_B200_STOP_AFTER_SPP  stop (exit code 3, no image) once that many samples are checkpointed — an interrupted run
inline void camera::render(std::ostream& output_stream, const hittable& world) {
  rt_camera_desc cam = desc();
  rt_camera_frame frame;
  rt_camera_initialize(&cam, &frame);
  std::printf("\rScanlines remaining: %d ", frame.image_height);
  std::fflush(stdout);

  auto scene = rtb200::flatten_world(world);
  rt_scene_desc sd = scene->desc();

  std::vector<int> devices = rtb200::device_list(samples_per_pixel);

  const int R = int(devices.size());
  rtb200::phase_timer timing;
  timing.mark("flatten");
  // Contexts (CUDA context, stream, scene arena, accumulator, reduce buffer, peer mappings) come from a process-level
  // cache and are released at exit: a program that renders several scenes or frames — main.cpp's switch run in a loop —
  // pays rt_init once per device, not once per camera::render (0.2-0.3 s each, more than most of the shipped scenes take
  // to render).
  std::vector<rt_ctx*> ctx = rtb200::context_cache::get().acquire_all(devices);
  timing.mark("init");
  rtb200::upload_all(ctx, sd);
  timing.mark("upload");
  // Several devices: the exchange step (the per-pixel sum of camera.hpp:61) is done on the devices — every context
  // adds its accumulator into the first one's reduce buffer over peer memory (rt_render_opts.push_accum), no host sum.
  // Devices without peer access to the first one fall back to the exact integer sum on the host.
  bool on_device = R > 1;
  for (int r = 1; r < R && on_device; r++) on_device = rtb200::context_cache::get().peer_enable(r, 0);
  timing.mark("peer");

  const size_t npix = size_t(frame.image_width) * frame.image_height;
  std::vector<int64_t> host_sum;  // the pass's sums when the devices cannot reduce among themselves
  // One pass = sample indices [begin, begin + count) of every pixel, count >= R, sharded over the devices.  Afterwards
  // the pass's sums sit in the first context's accumulator or, without peer access, in host_sum.
  auto run_pass = [&](int begin, int count) {
    void* reduce = nullptr;
    if (on_device) {  // (re-)zeroed for this pass
      int rc = rt_reduce_buffer(ctx[0], &cam, &reduce, nullptr);
      if (rc != RT_OK) rtb200::die(ctx[0], "rt_reduce_buffer", rc);
    }
    for (int r = 0; r < R; r++) {  // asynchronous: all devices render concurrently
      rt_render_opts o;
      std::memset(&o, 0, sizeof o);
      o.seed = 0;
      o.sample_begin = begin + int32_t((int64_t(count) * r) / R);
      o.sample_count = begin + int32_t((int64_t(count) * (r + 1)) / R) - o.sample_begin;
      o.clear = 1;
      o.push_accum = reduce;
      int rc = rt_render(ctx[size_t(r)], &cam, &o);
      if (rc != RT_OK) rtb200::die(ctx[size_t(r)], "rt_render", rc);
    }
    if (on_device) {
      for (int r = 0; r < R; r++) {
        int rc = rt_synchronize(ctx[size_t(r)]);
        if (rc != RT_OK) rtb200::die(ctx[size_t(r)], "rt_synchronize", rc);
      }
      int rc = rt_adopt_reduce_buffer(ctx[0]);
      if (rc != RT_OK) rtb200::die(ctx[0], "rt_adopt_reduce_buffer", rc);
    } else if (R > 1) {
      // exact integer reduction on the host side of the boundary (order-independent)
      std::vector<int64_t> part(npix * 3);
      host_sum.assign(npix * 3, 0);
      for (int r = 0; r < R; r++) {
        int rc = rt_download(ctx[size_t(r)], RT_BUF_ACCUM_I64, samples_per_pixel, part.data(), part.size() * 8);
        if (rc != RT_OK) rtb200::die(ctx[size_t(r)], "rt_download", rc);
        for (size_t i = 0; i < host_sum.size(); i++) host_sum[i] += part[i];
      }
    }
  };

  const char* ckpt = std::getenv("RT_B200_CHECKPOINT");
  if (ckpt && !*ckpt) ckpt = nullptr;
  bool sums_on_host = false;
  if (!ckpt) {
    run_pass(0, samples_per_pixel);
    sums_on_host = R > 1 && !on_device;
  } else {
    rtb200::checkpoint_header head;
    std::memset(&head, 0, sizeof head);
    std::memcpy(head.magic, "RTB2CKPT", 8);
    head.version = 1, head.width = uint32_t(frame.image_width), head.height = uint32_t(frame.image_height);
    head.spp_total = uint32_t(samples_per_pixel), head.max_depth = uint32_t(max_depth);
    head.seed = 0, head.scene_hash = rtb200::scene_hash(sd, cam);
    const char* e_pass = std::getenv("RT_B200_CHECKPOINT_SPP");
    const char* e_stop = std::getenv("RT_B200_STOP_AFTER_SPP");
    const int per_pass = std::max(R, e_pass ? std::atoi(e_pass) : 256);
    const int stop_after = e_stop ? std::atoi(e_stop) : 0;
    host_sum.assign(npix * 3, 0);
    std::vector<int64_t> total(npix * 3, 0), part(npix * 3);
    int done = rtb200::checkpoint_load(ckpt, head, total);
    while (done < samples_per_pixel) {
      int n = std::min(per_pass, samples_per_pixel - done);
      if (samples_per_pixel - done - n < R) n = samples_per_pixel - done;  // no pass smaller than the device count
      run_pass(done, n);
      const int64_t* pass = host_sum.data();
      if (R == 1 || on_device) {
        int rc = rt_download(ctx[0], RT_BUF_ACCUM_I64, samples_per_pixel, part.data(), part.size() * 8);
        if (rc != RT_OK) rtb200::die(ctx[0], "rt_download", rc);
        pass = part.data();
      }
      for (size_t i = 0; i < total.size(); i++) total[i] += pass[i];
      done += n;
      rtb200::checkpoint_save(ckpt, head, done, total);
      std::printf("\rSamples remaining: %d ", samples_per_pixel - done);
      std::fflush(stdout);
      if (stop_after > 0 && done >= stop_after && done < samples_per_pixel) {
        std::printf("\rStopped after %d of %d samples per pixel; checkpoint in %s\n", done, samples_per_pixel, ckpt);
        std::exit(3);
      }
    }
    host_sum.swap(total);
    // write_color on the device from the restored sums — the same finalize kernel as an uninterrupted render
    int rc = rt_upload_accum(ctx[0], &cam, host_sum.data(), host_sum.size() * 8);
    if (rc != RT_OK) rtb200::die(ctx[0], "rt_upload_accum", rc);
  }

  std::vector<uint8_t> rgb(npix * 3);
  if (!ckpt && (R == 1 || on_device)) {  // (the device passes above are asynchronous when nothing had to wait for them)
    for (int r = 0; r < R; r++) rt_synchronize(ctx[size_t(r)]);
  }
  timing.mark("render");
  if (!sums_on_host) {
    int rc = rt_download(ctx[0], RT_BUF_RGB8, samples_per_pixel, rgb.data(), rgb.size());
    if (rc != RT_OK) rtb200::die(ctx[0], "rt_download", rc);
  } else {
    // write_color (common/color.hpp:26-58) in double, operation for operation what the device's finalize kernel does
    const double scale = double(1.0f / float(samples_per_pixel));  // pixel_samples_scale, camera.hpp:83
    const double hi = double(0.999f);
    for (size_t i = 0; i < host_sum.size(); i++) {
      const double lin = double(host_sum[i]) * (1.0 / 4294967296.0) * scale;
      double g = lin > 0.0 ? std::sqrt(lin) : 0.0;
      g = g < 0.0 ? 0.0 : (g > hi ? hi : g);
      rgb[i] = uint8_t(int(256 * g));
    }
  }
  timing.mark("download");

  rtb200::write_ppm_p3(output_stream, frame.image_width, frame.image_height, rgb.data());
  output_stream.flush();
  if (const char* p6 = std::getenv("RT_B200_P6")) {
    if (*p6 && !rtb200::write_ppm_p6(p6, frame.image_width, frame.image_height, rgb.data()))
      std::fprintf(stderr, "rtb200: could not write %s\n", p6);
  }
  timing.mark("ppm");
  timing.report(frame.image_width, frame.image_height, samples_per_pixel, R);
  std::printf("\rDone.                       \n");
  std::fflush(stdout);
}

namespace rtb200 {
// Several frames of one world — a turntable, an animation's frames: outs[i] receives the P3 text camera::render writes for
// *cams[i], and stdout the same progress lines, frame after frame, so the program's output is that of a loop of
// camera::render calls.  The world is flattened and uploaded once per device; every device of RT_B200_DEVICES renders a
// contiguous range of the frames in one rt_render_views launch (no reduce: each frame is rendered whole on one device).
// The cameras must share image_width, image height and samples_per_pixel.  RT_B200_CHECKPOINT / RT_B200_P6 do not apply.
inline void render_views(const hittable& world, const std::vector<const camera*>& cams, const std::vector<std::ostream*>& outs) {
  if (cams.size() != outs.size()) {
    std::fprintf(stderr, "rtb200::render_views: %zu cameras but %zu output streams\n", cams.size(), outs.size());
    std::exit(1);
  }
  if (cams.empty()) return;
  const int V = int(cams.size());
  std::vector<rt_camera_desc> desc(cams.size());
  for (int v = 0; v < V; v++) desc[size_t(v)] = cams[size_t(v)]->desc();
  rt_camera_frame frame;
  rt_camera_initialize(&desc[0], &frame);
  const int spp = desc[0].samples_per_pixel;

  auto scene = flatten_world(world);
  rt_scene_desc sd = scene->desc();
  std::vector<int> devices = device_list(V);
  const int R = int(devices.size());
  std::vector<rt_ctx*> ctx = context_cache::get().acquire_all(devices);
  upload_all(ctx, sd);

  const size_t image = size_t(frame.image_width) * frame.image_height * 3;
  std::vector<uint8_t> rgb(image * size_t(V));
  for (int r = 0; r < R; r++) {  // asynchronous: all devices render concurrently
    const int begin = int((int64_t(V) * r) / R), end = int((int64_t(V) * (r + 1)) / R);
    rt_render_opts o;
    std::memset(&o, 0, sizeof o);
    o.seed = 0;
    o.clear = 1;
    int rc = rt_render_views(ctx[size_t(r)], end - begin, desc.data() + begin, &o);
    if (rc != RT_OK) die(ctx[size_t(r)], "rt_render_views", rc);
  }
  for (int r = 0; r < R; r++) {
    const int begin = int((int64_t(V) * r) / R), end = int((int64_t(V) * (r + 1)) / R);
    int rc = rt_download(ctx[size_t(r)], RT_BUF_RGB8, spp, rgb.data() + image * size_t(begin), image * size_t(end - begin));
    if (rc != RT_OK) die(ctx[size_t(r)], "rt_download", rc);
  }
  for (int v = 0; v < V; v++) {
    std::printf("\rScanlines remaining: %d ", frame.image_height);
    write_ppm_p3(*outs[size_t(v)], frame.image_width, frame.image_height, rgb.data() + image * size_t(v));
    outs[size_t(v)]->flush();
    std::printf("\rDone.                       \n");
  }
  std::fflush(stdout);
}
}  // namespace rtb200
#endif  // RTB200_NO_RENDER_IMPL

#endif  // RTB200_HOST_HPP
