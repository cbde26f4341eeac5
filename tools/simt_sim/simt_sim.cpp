// simt_sim.cpp — CPU simulator of SIMT scheduling policies for the render kernel (a design tool, not product code).
//
// It compiles csrc/rt_device.cuh for the host (shim/cuda_runtime.h) and runs the SAME per-lane routines the kernels run
// (node_step, hit_sphere / hit_box / hit_quad, medium_sample, surface_at, scatter_ray) on the SAME flattened scene and
// BVH (csrc/scene_build.hpp), but under a model of the warp: 32 lanes in lock step, a code block costs its instruction
// count once per warp if ANY lane executes it.  Output per policy: warp instructions and thread instructions per ray by
// phase, i.e. the "active lanes per instruction" ncu reports — so a scheduling design (lane refill from a queue, warp
// specialisation, refill thresholds ...) can be compared on the CPU before it is written in CUDA and measured on a B200.
//   policy mega : render_kernel as shipped in round 1 (a lane owns a path; while-while traversal; shade in place)
//   policy wq   : trace warps whose lanes take rays from a CTA-wide queue the moment enough of them are idle,
//                 shade in dense batches of 32 finished rays
//   policy inplace : the megakernel with in-place lane refill (the warp leaves the traversal once `shade_thr` lanes wait)
//   policy sym  : symmetric warps over CTA-wide queues
// Build: make -C tools/simt_sim      Run: tools/simt_sim/simt_sim book2_final mega|wq|sym|inplace [key=value ...]
//
// REALITY CHECK (round 2, profiles/r2_session_experiments.md).  The model reproduces the megakernel well (8.16 node visits per
// ray, 7.4 lanes in node_step against ncu's 6.8, 117 warp instructions per ray against 143) and its LANE predictions hold up
// on the GPU (in-place refill: 16-18 lanes predicted in node_step, 13.9 measured).  Its TIME predictions do not: it gave the
// refill schedule 1.30x, a node-step threshold 1.06x and the queue-fed kernel 1.45x fewer instructions; measured speeds are
// 0.83x, 0.81-0.89x and 0.46x.  What it lacks: (1) a shade round is charged per material group that is present, but on the GPU
// the long divergent shade costs ~1,350 warp instructions almost regardless of how many lanes take part, so every schedule
// that shades more often pays in full; (2) a leaf phase is charged 10 + 30..55 per primitive, the real one (six-way type
// dispatch at ~4 lanes, dependent shared-memory reads, the pop that follows) costs several times that, so schedules that
// multiply leaf phases lose; (3) it counts issued instructions only — the kernel is bound by the ALU pipe and by latency at 28
// warps per SM, and the reordered schedules drop issue utilisation from 75 % to 43-62 %.  Use it for lane statistics and ray
// census, not for speed-ups.
#include <cuda_runtime.h>  // the shim
#include <cstdio>
#include <cstdlib>
#include <deque>
#include <map>
#include <string>
#include <vector>

#include "../../raytracing-practice_b200/csrc/device_scene.h"
inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }
inline float2 make_float2(float x, float y) { return float2{x, y}; }
inline float2 __ffma2_rn(float2 a, float2 b, float2 c) { return float2{std::fma(a.x, b.x, c.x), std::fma(a.y, b.y, c.y)}; }
#include "../../raytracing-practice_b200/csrc/rt_device.cuh"
#include "../../raytracing-practice_b200/csrc/scene_build.hpp"

extern "C" {
struct rth_scene;
rth_scene* rth_scene_build(const char* name, long rand_seed);
const rt_scene_desc* rth_scene_desc(rth_scene* s);
rt_camera_desc* rth_scene_camera(rth_scene* s);
}
using namespace rtb200;

// ---- instruction-cost model (SASS instruction counts of the r15 build, rounded) -----------------------------------
struct Costs {
  double node = 52, pop_iter = 8, vote = 6, leaf_iter = 10, sph_miss = 30, sph_hit = 50, box = 55, quad = 30, medium = 120, medium_rng = 65;
  double gm = 130, regen = 110, item_fetch = 40, shade_base = 30, philox = 45, surf_sph = 45, surf_box = 50, surf_quad = 25, surf_med = 10;
  double scat_common = 35, lamb = 15, metal = 30, diel = 60, iso = 5, light = 5, tex_checker = 25, tex_image = 85, tex_noise = 1500, deposit = 20;
  double set_ray = 25;
  // wq only
  double fin = 14, refill = 40, qbook = 16, shade_load = 14, shade_store = 18;
} C;

struct Phase {
  double W = 0, T = 0;  // warp instructions, thread instructions
  void add(double cost, int lanes) { if (lanes > 0) W += cost, T += cost * lanes; }
};
static std::map<std::string, Phase> g_ph;
static inline void charge(const char* phase, double cost, int lanes) { g_ph[phase].add(cost, lanes); }

struct Cam {
  float3 center, p00c, du, dv, ddu, ddv, bg;
  int W, H, max_depth, defocus;
};
static void camera_frame(const rt_camera_desc* c, Cam& o) {  // camera::initialize, as rt_camera_initialize + fill_camera
  using namespace build_detail;
  const double pi = 3.1415926535897932385;
  int W = c->image_width, H = int(c->image_width / c->aspect_ratio);
  H = H < 1 ? 1 : H;
  double theta = c->vfov * pi / 180.0, h = std::tan(theta / 2), vh = 2 * h * c->focus_dist, vw = vh * (double(W) / H);
  d3 from = ld(c->lookfrom), at = ld(c->lookat), vup = ld(c->vup);
  auto unit = [](d3 v) { return (1 / std::sqrt(v.x * v.x + v.y * v.y + v.z * v.z)) * v; };
  d3 w = unit(from - at), u = unit(cross(vup, w)), v = cross(w, u);
  d3 vu = vw * u, vv = vh * d3{-v.x, -v.y, -v.z}, du = (1 / double(W)) * vu, dv = (1 / double(H)) * vv;
  d3 ul = from - (c->focus_dist * w) - 0.5 * vu - 0.5 * vv, p00 = ul + 0.5 * (du + dv);
  double dr = c->focus_dist * std::tan((c->defocus_angle * pi / 180.0) / 2.0);
  d3 ddu = dr * u, ddv = dr * v;
  auto f = [](d3 a) { return make_float3(float(a.x), float(a.y), float(a.z)); };
  o.center = f(from), o.p00c = f(p00 - from), o.du = f(du), o.dv = f(dv), o.ddu = f(ddu), o.ddv = f(ddv);
  o.bg = make_float3(float(c->background[0]), float(c->background[1]), float(c->background[2]));
  o.W = W, o.H = H, o.max_depth = c->max_depth, o.defocus = c->defocus_angle > 0;
}

// ---- the job: work items as in render_range -------------------------------------------------------------------------
struct Job {
  DeviceScene sc;
  Cam cam;
  uint2 key{7u, 0u};
  int chunk = 32, n_chunks = 1, tiles_x, tiles_y, tile_stride = 16;
  unsigned long long next_item = 0, n_items = 0;
  unsigned long long rays = 0, samples = 0;
  double radiance = 0;
  // a work item or false when the image is used up
  bool take(int& pixel, int& s0) {
    for (;;) {
      if (next_item >= n_items) return false;
      unsigned long long it = next_item++;
      unsigned per_chunk = unsigned(tiles_x) * tiles_y * 32u;
      unsigned chunkid = unsigned(it / per_chunk), q = unsigned(it % per_chunk);
      unsigned tile = q >> 5, lane = q & 31u;
      if (tile % unsigned(tile_stride) != 0) { next_item = it - lane + 32; continue; }  // subsample: every tile_stride-th tile
      int px = int(tile % unsigned(tiles_x)) * 8 + int(lane & 7u), py = int(tile / unsigned(tiles_x)) * 4 + int(lane >> 3);
      if (px < cam.W && py < cam.H) {
        pixel = py * cam.W + px, s0 = int(chunkid) * chunk;
        return true;
      }
    }
  }
};

struct Path {
  float3 o, d, beta;
  float time = 0;
  uint32_t skip = REF_NONE;
  int depth = 0, pixel = -1, s = 0, s_end = 0;
  Hit best{0, REF_NONE};  // seeded by the scene-enclosing media, then the closest hit
  bool alive = false, done = false;
};

// camera::get_ray for the next sample of p's item (fetching an item when needed).  Returns false when out of work.
static bool regenerate(Job& J, Path& p, bool& fetched) {
  fetched = false;
  if (p.pixel < 0 || p.s >= p.s_end) {
    int pixel, s0;
    fetched = true;
    if (!J.take(pixel, s0)) { p.done = true; return false; }
    p.pixel = pixel, p.s = s0, p.s_end = s0 + J.chunk;
  }
  PathKey key{J.key, uint32_t(p.pixel), uint32_t(p.s++)};
  const Cam& cam = J.cam;
  const int py = p.pixel / cam.W, px = p.pixel - py * cam.W;
  uint4 r0 = rng_block(key, 0u, 0u);
  float ox = u01(r0.x) - 0.5f, oy = u01(r0.y) - 0.5f;
  p.time = u01(r0.z);
  float3 dir = fma3(float(px) + ox, cam.du, fma3(float(py) + oy, cam.dv, cam.p00c));
  p.o = cam.center;
  if (cam.defocus) {
    uint4 r1 = rng_block(key, 0u, 1u);
    float rr = sqrtf(u01(r1.x)), sn, cs;
    sincos_2pi(u01(r1.y), sn, cs);
    float3 off = fma3(rr * cs, cam.ddu, (rr * sn) * cam.ddv);
    p.o = p.o + off, dir = dir - off;
  }
  p.d = dir, p.beta = f3(1, 1, 1), p.depth = cam.max_depth, p.skip = REF_NONE, p.alive = cam.max_depth > 0;
  J.samples++;
  return true;
}

// what a shade of one finished query costs, by divergence group
struct ShadeTag {
  int hit_type;  // -1 miss, else REF_*
  int mat;       // MAT_*
  int tex;       // 0 none/solid, TEX_*
  bool needs_uv;
};
static int root_texture_kind(const DeviceScene& sc, int tex, float3 p, bool& checker) {
  checker = false;
  for (int g = 0; g < 16 && tex >= 0; g++) {
    float4 t0 = sc.textures[2 * tex], t1 = sc.textures[2 * tex + 1];
    int kind = __float_as_int(t1.x), a = __float_as_int(t1.y), b = __float_as_int(t1.z);
    if (kind == TEX_CHECKER) {
      checker = true;
      int s = int(floorf(t0.w * p.x)) + int(floorf(t0.w * p.y)) + int(floorf(t0.w * p.z));
      tex = (s & 1) ? b : a;
      continue;
    }
    return kind;
  }
  return TEX_SOLID;
}
// the tail of ray_color for the query whose answer is p.best; returns the tag, updates the path (next ray or dead)
static ShadeTag shade_path(Job& J, Path& p) {
  const DeviceScene& sc = J.sc;
  ShadeTag tag{-1, 0, 0, false};
  J.rays++;
  Hit h = p.best;
  float3 L = f3(0, 0, 0);
  if (h.ref == REF_NONE) {
    L = p.beta * J.cam.bg;
    p.alive = false;
  } else {
    const PathKey key{J.key, uint32_t(p.pixel), uint32_t(p.s - 1)};
    const uint32_t bounce = uint32_t(J.cam.max_depth - p.depth) + 1u;
    const uint4 rnd = rng_block(key, bounce, 0u);
    Surface sf = surface_at(sc, h, p.o, p.d, p.time);
    float4 m1 = sc.materials[2 * sf.material + 1];
    tag.hit_type = int(h.ref >> 30), tag.mat = __float_as_int(m1.x);
    tag.needs_uv = (__float_as_int(m1.z) & MATF_NEEDS_UV) != 0;
    bool chk;
    int tex = __float_as_int(m1.y);
    tag.tex = tex >= 0 ? root_texture_kind(sc, tex, sf.p, chk) + (chk ? 16 : 0) : 0;
    float3 emit, atten, d_out;
    bool cont = scatter_ray<false>(sc, sf, p.d, rnd, emit, atten, d_out, nullptr);
    L = p.beta * emit;
    if (cont) {
      p.beta = p.beta * atten, p.o = sf.p, p.d = d_out;
      p.skip = (h.ref >> 30) == REF_MEDIUM ? REF_NONE : h.ref;
      p.alive = --p.depth > 0;
    } else {
      p.alive = false;
    }
  }
  if (!p.alive) J.radiance += L.x + L.y + L.z;
  return tag;
}
static void charge_shade(const char* ph, const std::vector<ShadeTag>& tags) {
  const int n = int(tags.size());
  if (!n) return;
  charge(ph, C.shade_base, n);
  int hits = 0, cnt_type[4] = {0, 0, 0, 0}, cnt_mat[8] = {0}, chk = 0, img = 0, noise = 0;
  for (const ShadeTag& t : tags) {
    if (t.hit_type < 0) continue;
    hits++, cnt_type[t.hit_type]++, cnt_mat[t.mat]++;
    if (t.tex & 16) chk++;
    if ((t.tex & 15) == TEX_IMAGE) img++;
    if ((t.tex & 15) == TEX_NOISE) noise++;
  }
  charge(ph, C.philox + C.scat_common, hits);
  charge(ph, C.surf_sph, cnt_type[REF_SPHERE]), charge(ph, C.surf_quad, cnt_type[REF_QUAD]), charge(ph, C.surf_box, cnt_type[REF_BOX]),
      charge(ph, C.surf_med, cnt_type[REF_MEDIUM]);
  charge(ph, C.lamb, cnt_mat[MAT_LAMBERTIAN]), charge(ph, C.metal, cnt_mat[MAT_METAL]), charge(ph, C.diel, cnt_mat[MAT_DIELECTRIC]),
      charge(ph, C.light, cnt_mat[MAT_LIGHT]), charge(ph, C.iso, cnt_mat[MAT_ISOTROPIC]);
  charge(ph, C.tex_checker, chk), charge(ph, C.tex_image, img);
  charge("perlin", C.tex_noise, noise);
  int dead = 0;
  (void)dead;
}

// ---- per-lane traversal engine --------------------------------------------------------------------------------------
struct Engine {
  TravState ts;
  TravStack st;
  int slot = -1;  // wq: the pool slot whose ray this lane traces
  int nodes_this_ray = 0;
};
static NodeSource g_ns;
static long g_kind_n[6][2], g_kind_nodes[6][2], g_bounce_n[41];
static std::vector<long> g_hist_nodes(512, 0);
static long g_pushes = 0, g_pop_iters = 0, g_pops_ok = 0, g_max_sp = 0;
static std::vector<long> g_hist_sp(40, 0);

// node steps for the lanes with cur >= 0; returns how many lanes took one
static int sim_node_step(std::vector<Engine*>& lanes, const char* ph) {
  int n = 0, pops_max = 0, pops_sum = 0, pop_lanes = 0;
  for (Engine* e : lanes) {
    if (e->ts.cur < 0) continue;
    n++;
    e->nodes_this_ray++;
    const int sp0 = e->ts.sp;
    node_step<false, false>(e->ts, e->st, g_ns, nullptr);
    if (e->ts.sp > sp0) g_pushes++, g_max_sp = std::max<long>(g_max_sp, e->ts.sp), g_hist_sp[size_t(e->ts.sp)]++;
    if (e->ts.sp < sp0 || e->ts.cur == kTravDone) g_pop_iters += sp0 - e->ts.sp, g_pops_ok += e->ts.cur != kTravDone;
    if (e->ts.sp < sp0 || (e->ts.cur == kTravDone)) {  // popped (both children missed)
      int it = std::max(1, sp0 - e->ts.sp);
      pops_max = std::max(pops_max, it), pops_sum += it, pop_lanes++;
    }
  }
  charge(ph, C.node, n);
  if (pop_lanes) g_ph[std::string(ph) + "_pop"].W += C.pop_iter * pops_max, g_ph[std::string(ph) + "_pop"].T += C.pop_iter * pops_sum;
  return n;
}
// leaf step for lanes sitting on a leaf (cur < 0 and != done)
static int sim_leaf_step(Job& J, std::vector<Engine*>& lanes, std::vector<Path*>& paths, const char* ph) {
  const DeviceScene& sc = J.sc;
  int n = 0, maxcount = 0;
  for (Engine* e : lanes)
    if (e->ts.cur < 0 && e->ts.cur != kTravDone) n++, maxcount = std::max(maxcount, ((~e->ts.cur) & 7) + 1);
  if (!n) return 0;
  for (int k = 0; k < maxcount; k++) {
    int c_iter = 0, c_sph_miss = 0, c_sph_hit = 0, c_box = 0, c_quad = 0, c_med = 0, c_med_rng = 0;
    for (size_t li = 0; li < lanes.size(); li++) {
      Engine* e = lanes[li];
      if (!(e->ts.cur < 0 && e->ts.cur != kTravDone)) continue;
      const int code = ~e->ts.cur, first = code >> 3, count = (code & 7) + 1;
      if (k >= count) continue;
      c_iter++;
      TravState& ts = e->ts;
      Path& p = *paths[li];
      uint32_t ref = sc.leaf_refs[first + k];
      uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
      float t = -1.0f;
      if (type == REF_SPHERE) {
        t = hit_sphere(sc.spheres[2 * idx], sc.spheres[2 * idx + 1], ts.o, ts.d, p.time, ts.tmin, ts.best.t, ref == p.skip);
        (t != -1.0f ? c_sph_hit : c_sph_miss)++;
      } else if (type == REF_QUAD) {
        if (ref != p.skip) t = hit_quad(sc.quads[3 * idx], sc.quads[3 * idx + 1], sc.quads[3 * idx + 2], ts.o, ts.d, ts.tmin, ts.best.t);
        c_quad++;
      } else if (type == REF_BOX) {
        if (ref != REF_NONE) {
          const uint32_t b = idx >> 3;
          const int self_face = ((p.skip >> 30) == REF_BOX && p.skip != REF_NONE && ((p.skip & 0x3FFFFFFFu) >> 3) == b) ? int(p.skip & 7u) : -1;
          int face = 0;
          t = hit_box(sc.boxes[3 * b], sc.boxes[3 * b + 1], sc.boxes[3 * b + 2], ts.o, ts.d, ts.inv, -ts.nood, ts.tmin, ts.best.t, self_face, face);
          ref = make_ref(REF_BOX, (b << 3) | uint32_t(face));
          c_box++;
        }
      } else {
        const DMedium m = sc.media[idx];
        PathKey key{J.key, uint32_t(p.pixel), uint32_t(p.s - 1)};
        const uint32_t bounce = uint32_t(J.cam.max_depth - p.depth) + 1u;
        float t1, t2;
        bool span = medium_span(sc, m, ts.o, ts.d, p.time, t1, t2) && fmaxf(t1, ts.tmin) < fminf(t2, ts.best.t);
        t = medium_sample(sc, m, int(idx), ts.o, ts.d, p.time, ts.tmin, ts.best.t, key, bounce);
        c_med++;
        if (span) c_med_rng++;
      }
      if (t != -1.0f) ts.best = Hit{t, ref};
    }
    charge(ph, C.leaf_iter, c_iter);
    charge(ph, C.sph_miss, c_sph_miss + c_sph_hit), charge(ph, C.sph_hit - C.sph_miss, c_sph_hit);
    charge(ph, C.box, c_box), charge(ph, C.quad, c_quad), charge("leaf_medium", C.medium, c_med), charge("leaf_medium", C.medium_rng, c_med_rng);
  }
  int pops_max = 0, pops_sum = 0;
  for (Engine* e : lanes) {
    if (!(e->ts.cur < 0 && e->ts.cur != kTravDone)) continue;
    const int sp0 = e->ts.sp;
    trav_pop(e->ts, e->st);
    g_pop_iters += sp0 - e->ts.sp, g_pops_ok += e->ts.cur != kTravDone;
    int it = std::max(1, sp0 - e->ts.sp);
    pops_max = std::max(pops_max, it), pops_sum += it;
  }
  g_ph[std::string(ph) + "_pop"].W += C.pop_iter * pops_max, g_ph[std::string(ph) + "_pop"].T += C.pop_iter * pops_sum;
  return n;
}
static void begin_ray(Job& J, Engine& e, Path& p, bool with_media) {
  trav_set_ray(e.ts, p.o, p.d, p.time, 0.001f, p.skip);
  const float INF = __int_as_float(0x7f800000);
  e.ts.best = Hit{INF, REF_NONE};
  if (with_media && J.sc.n_global_media) {
    PathKey key{J.key, uint32_t(p.pixel), uint32_t(p.s - 1)};
    const uint32_t bounce = uint32_t(J.cam.max_depth - p.depth) + 1u;
    e.ts.best = sample_global_media<false>(J.sc, p.o, p.d, p.time, 0.001f, INF, key, bounce, nullptr);
  }
  e.ts.sp = 0, e.ts.cur = 0, e.nodes_this_ray = 0;
}

// ---- policy: megakernel ---------------------------------------------------------------------------------------------
static void run_mega(Job& J, int n_warps, int node_unroll) {
  struct Warp {
    Path p[32];
    Engine e[32];
    bool finished = false;
  };
  std::vector<Warp> warps(static_cast<size_t>(n_warps));
  int live_warps = n_warps;
  while (live_warps) {
    for (Warp& w : warps) {
      if (w.finished) continue;
      int n_regen = 0, n_fetch = 0;
      for (int l = 0; l < 32; l++)
        if (!w.p[l].alive && !w.p[l].done) {
          bool fetched;
          if (regenerate(J, w.p[l], fetched)) n_regen++;
          n_fetch += fetched;
        }
      charge("regen", C.regen, n_regen), charge("regen", C.item_fetch, n_fetch);
      charge("loop", C.vote, 32);
      int alive = 0;
      bool all_done = true;
      for (int l = 0; l < 32; l++) alive += w.p[l].alive, all_done = all_done && w.p[l].done;
      if (!alive) {
        if (all_done) w.finished = true, live_warps--;
        continue;
      }
      std::vector<Engine*> lanes;
      std::vector<Path*> paths;
      for (int l = 0; l < 32; l++) {
        w.e[l].ts.cur = kTravDone;
        if (w.p[l].alive) begin_ray(J, w.e[l], w.p[l], true);
        lanes.push_back(&w.e[l]), paths.push_back(&w.p[l]);
      }
      charge("set_ray", C.set_ray, alive);
      if (J.sc.n_global_media) charge("global_media", C.gm * J.sc.n_global_media, alive);
      for (;;) {
        for (;;) {
          charge("trav_vote", C.vote, 32);
          bool any = false;
          for (Engine* e : lanes) any = any || e->ts.cur >= 0;
          if (!any) break;
          for (int u = 0; u < node_unroll; u++) sim_node_step(lanes, "node");
        }
        charge("trav_vote", C.vote, 32);
        if (!sim_leaf_step(J, lanes, paths, "leaf")) break;
      }
      std::vector<ShadeTag> tags;
      int n_dead = 0;
      for (int l = 0; l < 32; l++)
        if (w.p[l].alive) {
          g_hist_nodes[size_t(std::min(511, w.e[l].nodes_this_ray))]++;
          w.p[l].best = w.e[l].ts.best;
          {
            const Hit hb = w.e[l].ts.best;
            int kind = hb.ref == REF_NONE ? 0 : 1 + int(hb.ref >> 30);
            if (kind == 1 + int(REF_MEDIUM) && J.sc.n_global_media && int(hb.ref & 0x3FFFFFFFu) == J.sc.global_media[0]) kind = 5;
            const float3 o = w.p[l].o;
            const bool inside = o.x >= J.sc.bounds_lo[0] && o.x <= J.sc.bounds_hi[0] && o.y >= J.sc.bounds_lo[1] && o.y <= J.sc.bounds_hi[1] && o.z >= J.sc.bounds_lo[2] && o.z <= J.sc.bounds_hi[2];
            g_kind_n[kind][inside]++, g_kind_nodes[kind][inside] += w.e[l].nodes_this_ray;
            g_bounce_n[std::min(40, J.cam.max_depth - w.p[l].depth)]++;
          }
          tags.push_back(shade_path(J, w.p[l]));
          n_dead += !w.p[l].alive;
        }
      charge_shade("shade", tags);
      charge("shade", C.deposit, n_dead);
    }
  }
}

// ---- policy: CTA-wide queues, trace warps with lane refill, dense shade batches ---------------------------------------
struct WqOpts {
  int n_slots = 1024, n_trace_warps = 20, refill_thr = 8, node_unroll = 2;
  int node_thr = 1;  // keep taking node steps while at least this many lanes want one (1 = classic while-while)
};
static void run_wq(Job& J, const WqOpts& O) {
  std::vector<Path> slots(static_cast<size_t>(O.n_slots));
  std::deque<int> traceQ, shadeQ;
  for (int i = 0; i < O.n_slots; i++) shadeQ.push_back(i);  // fresh slots: their first shade is a regeneration
  int dead_slots = 0;
  struct TW {
    Engine e[32];
    double clock = 0;
  };
  std::vector<TW> tw(static_cast<size_t>(O.n_trace_warps));
  for (TW& w : tw)
    for (Engine& e : w.e) e.ts.cur = kTravDone, e.slot = -1;
  const float INF = __int_as_float(0x7f800000);
  (void)INF;
  auto shade_batch = [&]() {
    std::vector<ShadeTag> tags;
    int n = 0, n_regen = 0, n_fetch = 0, n_dead = 0, n_gm = 0;
    std::vector<int> batch;
    while (n < 32 && !shadeQ.empty()) batch.push_back(shadeQ.front()), shadeQ.pop_front(), n++;
    charge("shade_q", C.shade_load + C.shade_store, n);
    for (int s : batch) {
      Path& p = slots[size_t(s)];
      if (p.pixel >= 0 && p.alive) {
        tags.push_back(shade_path(J, p));
        n_dead += !p.alive;
      }
      if (!p.alive) {
        bool fetched;
        bool ok = regenerate(J, p, fetched);
        n_fetch += fetched;
        if (!ok) { dead_slots++; continue; }
        n_regen++;
      }
      // the next ray: scene-enclosing media here, 32 wide
      if (J.sc.n_global_media) {
        Engine tmp;
        begin_ray(J, tmp, p, true);
        p.best = tmp.ts.best;
        n_gm++;
      } else {
        p.best = Hit{INF, REF_NONE};
      }
      traceQ.push_back(s);
    }
    charge_shade("shade", tags);
    charge("shade", C.deposit, n_dead);
    charge("regen", C.regen, n_regen), charge("regen", C.item_fetch, n_fetch);
    charge("global_media", C.gm * J.sc.n_global_media, n_gm);
  };
  for (;;) {
    // shade whenever a full batch waits, or the tracers would starve
    while (shadeQ.size() >= 32 || (!shadeQ.empty() && traceQ.empty())) shade_batch();
    // the trace warp that is furthest behind runs one outer iteration
    TW* w = nullptr;
    for (TW& x : tw)
      if (!w || x.clock < w->clock) w = &x;
    double W0 = 0;
    for (auto& kv : g_ph) W0 += kv.second.W;
    std::vector<Engine*> lanes;
    std::vector<Path*> paths;
    int idle = 0, busy = 0;
    for (Engine& e : w->e) idle += e.ts.cur == kTravDone, busy += e.ts.cur != kTravDone;
    charge("trace_vote", C.vote, 32);
    if ((idle >= O.refill_thr || busy == 0) ) {
      int n_fin = 0, n_ref = 0;
      for (Engine& e : w->e)
        if (e.ts.cur == kTravDone) {
          if (e.slot >= 0) {
            g_hist_nodes[size_t(std::min(511, e.nodes_this_ray))]++;
            slots[size_t(e.slot)].best = e.ts.best;
            shadeQ.push_back(e.slot);
            e.slot = -1, n_fin++;
          }
          if (!traceQ.empty()) {
            e.slot = traceQ.front(), traceQ.pop_front();
            Path& p = slots[size_t(e.slot)];
            begin_ray(J, e, p, false);
            e.ts.best = p.best;
            n_ref++;
          }
        }
      charge("trace_q", C.qbook, 32), charge("trace_q", C.fin, n_fin), charge("trace_q", C.refill, n_ref);
    }
    busy = 0;
    for (Engine& e : w->e) {
      busy += e.ts.cur != kTravDone;
      lanes.push_back(&e), paths.push_back(e.slot >= 0 ? &slots[size_t(e.slot)] : nullptr);
    }
    if (!busy) {
      if (traceQ.empty() && shadeQ.empty()) {
        bool any = false;
        for (TW& x : tw)
          for (Engine& e : x.e) any = any || e.slot >= 0;
        if (!any) break;
      }
      w->clock += 50;  // idle poll
      continue;
    }
    for (;;) {
      charge("trav_vote", C.vote, 32);
      int want = 0;
      for (Engine* e : lanes) want += e->ts.cur >= 0;
      if (want < std::max(1, std::min(O.node_thr, busy)) ) {
        bool leafs = false;
        for (Engine* e : lanes) leafs = leafs || (e->ts.cur < 0 && e->ts.cur != kTravDone);
        if (want == 0 || leafs) break;
      }
      for (int u = 0; u < O.node_unroll; u++) sim_node_step(lanes, "node");
    }
    sim_leaf_step(J, lanes, paths, "leaf");
    double W1 = 0;
    for (auto& kv : g_ph) W1 += kv.second.W;
    w->clock += W1 - W0;
  }
}


// ---- policy: symmetric warps over CTA-wide queues ---------------------------------------------------------------------
// Every warp alternates between TRACE (lanes = traversal engines refilled from traceQ) and SHADE (a dense batch of 32
// finished rays from shadeQ); a tracer leaves for SHADE only with a batch already reserved, its unfinished traversals
// stay suspended in its lanes.  Warps advance on virtual clocks (warp instructions issued).
struct SymOpts {
  int n_slots = 1024, n_warps = 24, refill_thr = 8, node_unroll = 1, node_thr = 10, shade_min = 32;
  double alpha = 0;  // > 0: node step iff want >= alpha * leafs (majority rule) instead of the fixed threshold
  double switch_cost = 40;
};
static void run_sym(Job& J, const SymOpts& O) {
  std::vector<Path> slots(static_cast<size_t>(O.n_slots));
  std::deque<int> traceQ, shadeQ;
  for (int i = 0; i < O.n_slots; i++) shadeQ.push_back(i);
  struct SW {
    Engine e[32];
    double clock = 0;
    std::vector<int> batch;  // a reserved shade batch
  };
  std::vector<SW> ws(static_cast<size_t>(O.n_warps));
  for (SW& w : ws)
    for (Engine& e : w.e) e.ts.cur = kTravDone, e.slot = -1;
  const float INF = __int_as_float(0x7f800000);
  long n_batches = 0, n_batch_lanes = 0, starved_polls = 0, refills = 0, refill_lanes = 0;
  auto totalW = [&]() { double W = 0; for (auto& kv : g_ph) W += kv.second.W; return W; };
  auto reserve = [&](SW& w, bool starving) {
    if (shadeQ.size() >= size_t(O.shade_min) || (starving && !shadeQ.empty())) {
      while (w.batch.size() < 32 && !shadeQ.empty()) w.batch.push_back(shadeQ.front()), shadeQ.pop_front();
      return true;
    }
    return false;
  };
  auto shade_batch = [&](SW& w) {
    std::vector<ShadeTag> tags;
    int n = int(w.batch.size()), n_regen = 0, n_fetch = 0, n_dead = 0, n_gm = 0;
    n_batches++, n_batch_lanes += n;
    charge("shade_q", C.shade_load + C.shade_store, n);
    charge("switch", O.switch_cost, 32);
    for (int s : w.batch) {
      Path& p = slots[size_t(s)];
      if (p.pixel >= 0 && p.alive) {
        tags.push_back(shade_path(J, p));
        n_dead += !p.alive;
      }
      if (!p.alive) {
        bool fetched;
        bool ok = regenerate(J, p, fetched);
        n_fetch += fetched;
        if (!ok) continue;  // dead slot
        n_regen++;
      }
      if (J.sc.n_global_media) {
        Engine tmp;
        begin_ray(J, tmp, p, true);
        p.best = tmp.ts.best;
        n_gm++;
      } else {
        p.best = Hit{INF, REF_NONE};
      }
      traceQ.push_back(s);
    }
    w.batch.clear();
    charge_shade("shade", tags);
    charge("shade", C.deposit, n_dead);
    charge("regen", C.regen, n_regen), charge("regen", C.item_fetch, n_fetch);
    charge("global_media", C.gm * J.sc.n_global_media, n_gm);
  };
  for (;;) {
    SW* w = nullptr;
    for (SW& x : ws)
      if (!w || x.clock < w->clock) w = &x;
    const double W0 = totalW();
    int idle = 0, busy = 0;
    for (Engine& e : w->e) idle += e.ts.cur == kTravDone, busy += e.ts.cur != kTravDone;
    charge("trace_vote", C.vote, 32);
    if (idle >= O.refill_thr || busy == 0) {
      // finish + refill; poll the shade queue
      int n_fin = 0, n_ref = 0;
      for (Engine& e : w->e)
        if (e.ts.cur == kTravDone && e.slot >= 0) {
          g_hist_nodes[size_t(std::min(511, e.nodes_this_ray))]++;
          slots[size_t(e.slot)].best = e.ts.best;
          shadeQ.push_back(e.slot);
          e.slot = -1, n_fin++;
        }
      charge("trace_q", C.qbook, 32), charge("trace_q", C.fin, n_fin);
      if (reserve(*w, traceQ.empty())) {
        shade_batch(*w);
        w->clock += totalW() - W0;
        continue;
      }
      for (Engine& e : w->e)
        if (e.ts.cur == kTravDone && !traceQ.empty()) {
          e.slot = traceQ.front(), traceQ.pop_front();
          Path& p = slots[size_t(e.slot)];
          begin_ray(J, e, p, false);
          e.ts.best = p.best;
          n_ref++;
        }
      charge("trace_q", C.refill, n_ref);
      refills++, refill_lanes += n_ref;
    }
    std::vector<Engine*> lanes;
    std::vector<Path*> paths;
    busy = 0;
    for (Engine& e : w->e) {
      busy += e.ts.cur != kTravDone;
      lanes.push_back(&e), paths.push_back(e.slot >= 0 ? &slots[size_t(e.slot)] : nullptr);
    }
    if (!busy) {
      bool any = !traceQ.empty() || !shadeQ.empty();
      for (SW& x : ws)
        for (Engine& e : x.e) any = any || e.slot >= 0;
      if (!any) break;
      starved_polls++;
      w->clock += 50;
      charge("starve", 50, 32);
      continue;
    }
    // node steps while enough lanes want one, else a leaf step
    for (;;) {
      charge("trav_vote", C.vote, 32);
      int want = 0, leafs = 0;
      for (Engine* e : lanes) want += e->ts.cur >= 0, leafs += (e->ts.cur < 0 && e->ts.cur != kTravDone);
      if (O.alpha > 0 ? (want == 0 || (leafs > 0 && want < O.alpha * leafs)) : (want == 0 || (want < O.node_thr && leafs > 0))) break;
      for (int u = 0; u < O.node_unroll; u++) sim_node_step(lanes, "node");
    }
    sim_leaf_step(J, lanes, paths, "leaf");
    w->clock += totalW() - W0;
  }
  printf("sym: %ld shade batches, %.1f lanes each; %ld refills, %.1f lanes each; %ld starved polls\n", n_batches, double(n_batch_lanes) / n_batches, refills,
         double(refill_lanes) / std::max(1L, refills), starved_polls);
}


// ---- policy: megakernel with IN-PLACE lane refill ---------------------------------------------------------------------
// A lane still owns its path, but the warp leaves the traversal as soon as `shade_thr` lanes have finished their ray:
// those lanes shade / regenerate / seed the next ray while the others keep their traversal suspended (state parked in
// shared memory: `switch_cost` instructions per transition for the whole warp), then everybody traverses again.
struct InplaceOpts {
  int n_warps = 28, node_thr = 10, shade_thr = 16, node_unroll = 2;
  double switch_cost = 40;
};
static void run_inplace(Job& J, const InplaceOpts& O) {
  struct Warp {
    Path p[32];
    Engine e[32];
    bool finished = false;
  };
  std::vector<Warp> warps(static_cast<size_t>(O.n_warps));
  for (Warp& w : warps)
    for (Engine& e : w.e) e.ts.cur = kTravDone;
  int live_warps = O.n_warps;
  long n_shade_rounds = 0, n_shade_lanes = 0;
  while (live_warps) {
    for (Warp& w : warps) {
      if (w.finished) continue;
      // ---- SHADE: every lane whose traversal is over ----
      std::vector<ShadeTag> tags;
      int n_dead = 0, n_regen = 0, n_fetch = 0, n_new = 0, n_lanes = 0;
      for (int l = 0; l < 32; l++) {
        if (w.e[l].ts.cur != kTravDone || w.p[l].done) continue;
        n_lanes++;
        if (w.p[l].alive) {
          g_hist_nodes[size_t(std::min(511, w.e[l].nodes_this_ray))]++;
          w.p[l].best = w.e[l].ts.best;
          tags.push_back(shade_path(J, w.p[l]));
          n_dead += !w.p[l].alive;
        }
        if (!w.p[l].alive) {
          bool fetched;
          if (regenerate(J, w.p[l], fetched)) n_regen++;
          n_fetch += fetched;
        }
        if (w.p[l].alive) begin_ray(J, w.e[l], w.p[l], true), n_new++;
      }
      n_shade_rounds++, n_shade_lanes += n_lanes;
      charge("switch", O.switch_cost, 32);
      charge_shade("shade", tags);
      charge("shade", C.deposit, n_dead);
      charge("regen", C.regen, n_regen), charge("regen", C.item_fetch, n_fetch);
      charge("set_ray", C.set_ray, n_new);
      if (J.sc.n_global_media) charge("global_media", C.gm * J.sc.n_global_media, n_new);
      std::vector<Engine*> lanes;
      std::vector<Path*> paths;
      int tracing = 0;
      for (int l = 0; l < 32; l++) lanes.push_back(&w.e[l]), paths.push_back(&w.p[l]), tracing += w.e[l].ts.cur != kTravDone;
      if (!tracing) {
        bool all_done = true;
        for (int l = 0; l < 32; l++) all_done = all_done && w.p[l].done;
        if (all_done) w.finished = true, live_warps--;
        continue;
      }
      // ---- TRACE until shade_thr lanes wait for a shade (or nobody is tracing) ----
      for (;;) {
        charge("trav_vote", C.vote, 32);
        int want = 0, leafs = 0, waiting = 0;
        for (int l = 0; l < 32; l++) {
          const int c = w.e[l].ts.cur;
          want += c >= 0, leafs += (c < 0 && c != kTravDone), waiting += (c == kTravDone && !w.p[l].done);
        }
        if (want + leafs == 0 || waiting >= O.shade_thr) break;
        if (want >= O.node_thr || leafs == 0) {
          for (int u = 0; u < O.node_unroll; u++) sim_node_step(lanes, "node");
        } else {
          sim_leaf_step(J, lanes, paths, "leaf");
        }
      }
    }
  }
  printf("inplace: %ld shade rounds, %.1f lanes each\n", n_shade_rounds, double(n_shade_lanes) / n_shade_rounds);
}

int main(int argc, char** argv) {
  std::string scene = argc > 1 ? argv[1] : "book2_final", policy = argc > 2 ? argv[2] : "mega";
  std::map<std::string, double> kv;
  for (int i = 3; i < argc; i++) {
    std::string a = argv[i];
    size_t eq = a.find('=');
    if (eq != std::string::npos) kv[a.substr(0, eq)] = atof(a.c_str() + eq + 1);
  }
  auto opt = [&](const char* k, double d) { return kv.count(k) ? kv[k] : d; };
  rth_scene* s = rth_scene_build(scene.c_str(), 1);
  if (!s) { fprintf(stderr, "unknown scene\n"); return 1; }
  HostScene h;
  if (!build_host_scene(rth_scene_desc(s), h)) { fprintf(stderr, "build failed: %s\n", h.error.c_str()); return 1; }
  Job J;
  DeviceScene& d = J.sc;
  memset(&d, 0, sizeof d);
  d.nodes = h.nodes.data(), d.leaf_refs = h.leaf_refs.data(), d.spheres = h.spheres.data(), d.sph_meta = h.sph_meta.data();
  d.quads = h.quads.data(), d.quad_mat = h.quad_mat.data(), d.boxes = h.boxes.data(), d.box_meta = h.box_meta.data();
  d.media = h.media.data(), d.medium_brefs = h.medium_brefs.data(), d.materials = h.materials.data(), d.textures = h.textures.data();
  d.texels = h.texels.data(), d.images = h.images.data(), d.perlin_vec = h.perlin_vec.data(), d.perlin_perm = h.perlin_perm.data();
  d.rotations = h.rotations.data();
  d.n_nodes = int(h.nodes.size() / 4), d.n_spheres = int(h.spheres.size() / 2), d.n_quads = int(h.quads.size() / 3), d.n_boxes = int(h.boxes.size() / 3);
  d.n_leaf_refs = int(h.leaf_refs.size()), d.n_media = int(h.media.size()), d.n_materials = int(h.materials.size() / 2), d.n_textures = int(h.textures.size() / 2);
  for (int a = 0; a < 3; a++) d.bounds_lo[a] = h.bounds_lo[a], d.bounds_hi[a] = h.bounds_hi[a];
  d.n_global_media = int(h.global_media.size());
  for (int i = 0; i < 4; i++) d.global_media[i] = i < d.n_global_media ? h.global_media[size_t(i)] : -1;
  g_ns = NodeSource{nullptr, d.nodes, 0, 0u};
  rt_camera_desc cam = *rth_scene_camera(s);
  if (kv.count("width")) cam.image_width = int(kv["width"]);
  camera_frame(&cam, J.cam);
  J.chunk = int(opt("chunk", 32)), J.n_chunks = int(opt("chunks", 1)), J.tile_stride = int(opt("stride", 16));
  J.tiles_x = (J.cam.W + 7) / 8, J.tiles_y = (J.cam.H + 3) / 4;
  J.n_items = (unsigned long long)J.tiles_x * J.tiles_y * 32ull * J.n_chunks;
  printf("scene %s: %d nodes depth %d, %d spheres %d boxes %d quads %d media (%d global), image %dx%d depth %d\n", scene.c_str(), d.n_nodes, h.bvh_depth,
         d.n_spheres, d.n_boxes, d.n_quads, d.n_media, d.n_global_media, J.cam.W, J.cam.H, J.cam.max_depth);
  if (policy == "mega") {
    run_mega(J, int(opt("warps", 28)), int(opt("unroll", 2)));
  } else if (policy == "inplace") {
    InplaceOpts O;
    O.n_warps = int(opt("warps", 28)), O.node_thr = int(opt("node_thr", 10)), O.shade_thr = int(opt("shade_thr", 16)), O.node_unroll = int(opt("unroll", 2));
    O.switch_cost = opt("switch", 40);
    run_inplace(J, O);
  } else if (policy == "sym") {
    SymOpts O;
    O.n_slots = int(opt("slots", 1024)), O.n_warps = int(opt("warps", 24)), O.refill_thr = int(opt("refill", 8)), O.node_unroll = int(opt("unroll", 1));
    O.node_thr = int(opt("node_thr", 10)), O.shade_min = int(opt("shade_min", 32)), O.alpha = opt("alpha", 0);
    run_sym(J, O);
  } else {
    WqOpts O;
    O.n_slots = int(opt("slots", 1024)), O.n_trace_warps = int(opt("twarps", 20)), O.refill_thr = int(opt("refill", 8)), O.node_unroll = int(opt("unroll", 2));
    O.node_thr = int(opt("node_thr", 1));
    run_wq(J, O);
  }
  double W = 0, T = 0;
  for (auto& kvp : g_ph) W += kvp.second.W, T += kvp.second.T;
  printf("policy %s: %llu samples, %llu rays (%.2f rays/sample), mean radiance %.5f\n", policy.c_str(), J.samples, J.rays, double(J.rays) / J.samples,
         J.radiance / (3.0 * J.samples));
  printf("%-14s %10s %10s %7s %7s\n", "phase", "winst/ray", "tinst/ray", "lanes", "winst%");
  for (auto& kvp : g_ph)
    printf("%-14s %10.2f %10.1f %7.2f %6.1f%%\n", kvp.first.c_str(), kvp.second.W / J.rays, kvp.second.T / J.rays, kvp.second.T / kvp.second.W,
           100 * kvp.second.W / W);
  printf("%-14s %10.2f %10.1f %7.2f\n", "TOTAL", W / J.rays, T / J.rays, T / W);
  {
    const char* kn[6] = {"none", "sphere", "quad", "medium", "box", "gmedium"};
    for (int k = 0; k < 6; k++)
      for (int in = 0; in < 2; in++)
        if (g_kind_n[k][in]) printf("hit %-8s origin %s: %6.2f%% of rays, %.2f nodes\n", kn[k], in ? "inside " : "outside", 100.0 * g_kind_n[k][in] / J.rays, double(g_kind_nodes[k][in]) / g_kind_n[k][in]);
    printf("rays by bounce:");
    for (int b = 0; b < 41; b++) printf(" %.3f", double(g_bounce_n[b]) / J.samples);
    printf("\n");
  }
  long tot = 0, acc = 0;
  for (long v : g_hist_nodes) tot += v;
  printf("node visits per ray: ");
  double mean = 0;
  for (size_t i = 0; i < g_hist_nodes.size(); i++) mean += double(i) * g_hist_nodes[i];
  printf("mean %.2f; percentiles:", mean / tot);
  const double qs[] = {0.25, 0.5, 0.75, 0.9, 0.95, 0.99, 0.999};
  size_t qi = 0;
  for (size_t i = 0; i < g_hist_nodes.size() && qi < 7; i++) {
    acc += g_hist_nodes[i];
    while (qi < 7 && acc >= qs[qi] * tot) printf(" p%g=%zu", qs[qi] * 100, i), qi++;
  }
  printf("\n");
  printf("stack: pushes/ray %.3f, pop iterations/ray %.3f, pops taken/ray %.3f (culled %.3f), max depth %ld\n", double(g_pushes) / J.rays, double(g_pop_iters) / J.rays,
         double(g_pops_ok) / J.rays, double(g_pop_iters - g_pops_ok) / J.rays, g_max_sp);
  printf("stack depth after push histogram:");
  for (size_t i = 1; i < g_hist_sp.size(); i++) if (g_hist_sp[i]) printf(" %zu:%.4f", i, double(g_hist_sp[i]) / g_pushes);
  printf("\n");
  return 0;
}
