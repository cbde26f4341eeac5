// rt_b200.cu — kernels + the C-ABI of include/rt_b200.h (librt_b200.so), sm_100a only.
//
// The hot path — camera::render's pixel x sample loop with its recursive ray_color
// (src/core/camera.hpp:29-72, 180-232) — is ONE persistent megakernel:
//   * grid = #SMs CTAs (one per SM), each staging the top of the BVH in shared memory;
//   * work item = (pixel, chunk of consecutive sample indices); lanes pull items from a global
//     atomic counter and REGENERATE a camera path the moment theirs ends, so a warp never
//     idles on its longest path: every loop iteration is "trace one segment + shade" for all
//     32 lanes (the recursion of ray_color is a pure tail product, SURVEY.md §3.3);
//   * every sample is quantised to 2^-32 fixed point and summed as int64: integer addition is
//     associative, so the image is bit-identical for any split of samples over lanes, CTAs,
//     launches and GPUs (the multi-GPU reduce is an exact ncclInt64 sum or peer red.add.u64).
// There is no CPU fallback: rt_init fails without a device.
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/rt_b200.h"
#include "device_scene.h"
#include "rt_device.cuh"
#include "scene_build.hpp"

namespace rtb200 {

struct CameraDev {
  float3 center, p00c, du, dv, ddu, ddv, bg;
  int W, H, max_depth, defocus;
};

// Shared-memory plan of the streaming kernel (rt_stream.cuh), byte offsets into its dynamic shared memory.
struct StreamLayout {
  uint32_t node_plane;             // bytes per node plane = 16 * n_nodes: planes A, B, C at 0, 1x, 2x; the (child, child) pairs (8 B) at 3x
  uint32_t off_sph, off_box, off_refs;
  uint32_t off_slots, slot_plane;  // path pool: 4 planes of 16 B x n_slots
  uint32_t off_stack;              // traversal stacks: [level][thread] x 4 B
  uint32_t off_tq, off_sq, ring_mask;  // trace / shade queues: rings of (ring_mask + 1) 16-bit slot numbers
  uint32_t off_ctl;
  uint32_t n_slots;
  uint32_t total;
};

struct RenderParams {
  DeviceScene sc;
  CameraDev cam;
  uint2 key;
  int sample_begin, sample_count, chunk, n_chunks;
  int tiles_x, tiles_y;
  unsigned int per_chunk;  // work items per sample chunk = tiles_x * tiles_y * 32
  unsigned int n_items;
  unsigned long long* accum;     // 3 x int64 per pixel (two's complement adds)
  unsigned long long* push;      // peer reduce: a reduce buffer (possibly another GPU's) that push_kernel adds `accum` into
  unsigned long long n_values;   // 3 * W * H
  unsigned long long* counters;  // [0] next work item, [1] rays, [2] samples
  int smem_nodes;
  unsigned int state_off;  // byte offset of the per-thread shade-state records in dynamic shared memory
  unsigned int stack_off;  // byte offset of the shared-memory traversal stacks (kernels instantiated with SSTACK)
  unsigned int stack_levels;  // levels reserved per thread at stack_off (checks builds test against it)
  int* aov_id;             // render_kernel<.., AOV>: primitive id, t and shading normal of every pixel-centre ray
  float* aov_t;
  float* aov_n;
  float* aov_b;            // render_kernel<.., AOV> with max_depth 2: the bounce segment, kAovBounce floats per pixel
  StreamLayout sl;   // streaming kernel only
  // render_kernel<.., VIEWS> (rt_render_views): one camera per view; `cam` above carries the size all views share.
  // A work item's global pixel is view * view_pixels + in-view pixel, and per_chunk covers all views.
  const CameraDev* cams;
  int n_views;
  unsigned int view_items;   // work items per view and sample chunk = tiles_x * tiles_y * 32
  unsigned int view_pixels;  // W * H
};

#ifndef RT_THREADS
#define RT_THREADS 896  // 28 warps x 72 registers: +6 % over 1024 x 64 on the Book-2 scene since the box primitive (gpurun_out/ab_threads.log)
#endif
constexpr int kRenderThreads = RT_THREADS;
#ifndef RT_SMEM_STACK_BUDGET_KB
#define RT_SMEM_STACK_BUDGET_KB 164  // shared memory a launch may use and still take the stacks in: leaves L1 >= 64 KB of the 228 KB
#endif
#ifndef RT_SMEM_STACK
#define RT_SMEM_STACK 1  // traversal stacks in shared memory when the launch has the room (rt_device.cuh, TravStackS)
#endif
constexpr size_t kSmemStackBudget = size_t(RT_SMEM_STACK_BUDGET_KB) * 1024;
#ifndef RT_DEFAULT_STREAM
#define RT_DEFAULT_STREAM 0
#endif
constexpr bool kDefaultStreamKernel = RT_DEFAULT_STREAM != 0;
enum : int { KERNEL_MEGA = 0, KERNEL_STREAM = 1, KERNEL_REFILL = 2 };
constexpr int RT_RENDER_POOL_REMOVED = 4;  // rt_b200.h: the bit of the removed path-pool kernel
#ifndef RT_DEFAULT_REFILL
#define RT_DEFAULT_REFILL 0
#endif
constexpr bool kDefaultRefillKernel = RT_DEFAULT_REFILL != 0;
constexpr float kFixScale = 4294967296.0f;  // 2^32
constexpr int kAovBounce = 12;              // floats per pixel of the bounce AOV record (render_kernel)

__device__ __forceinline__ long long to_fixed(float v) {
  // NaN -> 0 (a NaN sample would poison the pixel).  The clamp bounds one sample at 2^16 = 65,536 (the brightest
  // emitter of the shipped scenes is 15; write_color clips the pixel MEAN at 0.999 anyway), so a sample is < 2^48 in
  // fixed point and the signed 64-bit sum holds 2^15 = 32,768 samples AT the clamp — and 2^31 samples of radiance <= 1
  // — without wrapping; the headline 10,000 spp fits with every sample at the clamp.
  v = (v == v) ? fminf(fmaxf(v, 0.0f), 65536.0f) : 0.0f;
  return __float2ll_rn(v * kFixScale);
}

// The multi-GPU exchange step (the per-pixel sum of camera.hpp:61 across ranks) without a collective call: stream-
// ordered right behind the render kernel, every rank adds its accumulator into rank 0's reduce buffer — its own memory
// or another GPU's, peer-mapped over NVLink — with system-scope red.add.u64.  Integer adds commute, so the reduced
// image has the bits of a single-GPU render.  15 MB per rank once per multi-second render.
// (Doing this from the render kernel's own epilogue — grid-wide arrival counter, cooperative launch — was built and
// worked, but the mere presence of that code cost the main loop 11 % on the headline scene through ptxas' scheduling:
// 948 vs 1,073 Msamples/s, gpurun_out/ab_push.log.  A separate 20-microsecond kernel costs nothing.)
__global__ void push_kernel(const unsigned long long* __restrict__ accum, unsigned long long* __restrict__ push, unsigned long long n_values) {
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_values; i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long v = __ldcg(accum + i);  // L2: the sums were made by red.add at L2
    if (v) atomicAdd_system(push + i, v);
  }
}

// AOV = true is the parity instantiation (rt_primary_visibility with RT_TRACE_RENDER_KERNEL): the SAME kernel — staging,
// work distribution, camera ray arithmetic, closest_hit_keyfn with the same node / leaf steps and stack — traces the
// jitter-free pixel-centre ray of every pixel (no defocus, time 0, media transparent) and, instead of shading, writes
// the primitive id, t and normal it found, so that the traversal rt_render runs is itself under the id / t / normal gate
// (camera.hpp:192, hittable_list.hpp:40-64).  With P.aov_b (rt_bounce_visibility, max_depth 2) a pixel-centre ray that
// hits is shaded as rt_render shades it (surface_at + scatter_ray, sample 0, bounce 1), its scattered ray takes the
// start primitive exactly as below (`skip`) and goes through the same traversal in the next iteration; that second hit
// is written as the record {origin1.xyz, dir1.xyz, normal.xyz, t, id bits, front}.
// COOP = true evaluates Perlin turbulence warp-cooperatively (below); chosen per scene by the launch plan — only where a
// good share of the primitives carries a noise texture: the hoisted hit record it needs costs the other scenes 3 %.
// VIEWS = true renders a batch of views of one scene (rt_render_views): the work items of a sample chunk run over
// (view, tile, lane), and a path's global pixel — the one its state record holds — is view * W * H + its in-view pixel.
// Its camera, its Philox pixel (the in-view one) and its bounce numbering are derived from that index where they are
// needed, so nothing more is live across the traversal; the sums go to view-major images.  Every path is the path
// rt_render(cams[view]) traces, so view v has the bits of that render.
template <bool COUNT, bool ALL_SMEM, bool SSTACK = false, bool AOV = false, bool COOP = false, bool VIEWS = false>
__global__ void __launch_bounds__(kRenderThreads, 1) render_kernel(const __grid_constant__ RenderParams P) {
  extern __shared__ float4 s_nodes[];
  stage_nodes<ALL_SMEM>(s_nodes, P.sc.nodes, P.smem_nodes);
  LeafSource ls{0u, 0u, 0u};
  if (ALL_SMEM) {  // ... and the leaves' data: [nodes][spheres 2 x float4][boxes 3 x float4][leaf refs u32]
    float4* s_sph = s_nodes + 4 * P.smem_nodes;
    float4* s_box = s_sph + 2 * P.sc.n_spheres;
    uint32_t* s_ref = reinterpret_cast<uint32_t*>(s_box + 3 * P.sc.n_boxes);
    for (int i = threadIdx.x; i < 2 * P.sc.n_spheres; i += blockDim.x) s_sph[i] = P.sc.spheres[i];
    for (int i = threadIdx.x; i < 3 * P.sc.n_boxes; i += blockDim.x) s_box[i] = P.sc.boxes[i];
    for (int i = threadIdx.x; i < P.sc.n_leaf_refs; i += blockDim.x) s_ref[i] = P.sc.leaf_refs[i];
    ls.spheres = opaque_u32(uint32_t(__cvta_generic_to_shared(s_sph)));
    ls.boxes = opaque_u32(uint32_t(__cvta_generic_to_shared(s_box)));
    ls.refs = opaque_u32(uint32_t(__cvta_generic_to_shared(s_ref)));
  }
  __syncthreads();
  const NodeSource ns = node_source(s_nodes, P.sc.nodes, P.smem_nodes, P.sc.n_nodes);
  const DeviceScene& sc = P.sc;
  const float INF = __int_as_float(0x7f800000);
  // the camera of a global pixel index, and its in-view pixel (the pixel of its Philox counter); one camera without VIEWS
  auto cam_of = [&](int pixel) -> const CameraDev& {
    if constexpr (VIEWS) {
      RT_CHECK(unsigned(pixel) / P.view_pixels < unsigned(P.n_views), CHK_VIEW);
      return P.cams[unsigned(pixel) / P.view_pixels];
    } else {
      return P.cam;
    }
  };
  auto view_pixel = [&](int pixel) -> int {
    if constexpr (VIEWS) return int(unsigned(pixel) % P.view_pixels);
    else return pixel;
  };

  // Per-lane path state, kept small on purpose: the kernel runs 896 threads per SM (72 registers; 1024 x 64 and 768 x 80
  // are slower, gpurun_out/ab_lean2.log) and it is very sensitive to what is live across the traversal — two more
  // values cost 16-24 % (profiles/r15_fastforward_rejected.patch), the diet below gained 6-9 % (gpurun_out/ab_lean*.log):
  // no running radiance sum, a warp-uniform ray counter, no end-of-item / next-item registers, and
  // what only SHADE needs — throughput, depth, pixel, next sample — lives in shared memory between shades, not in
  // registers across the traversal, and so do the ray's time and the primitive it starts on, which only leaves look at:
  // two float4 records per thread, {beta.xyz, depth} and {pixel, s, time, skip}, read with volatile LDS so that the
  // compiler cannot carry a loaded value across the traversal instead.
  const uint32_t st_a = opaque_u32(uint32_t(__cvta_generic_to_shared(s_nodes)) + P.state_off) + 16u * threadIdx.x;
  constexpr uint32_t kStB = 16u * kRenderThreads;
  auto sts_f4 = [](uint32_t addr, float4 v) { asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory"); };
  sts_f4(st_a, make_float4(1.0f, 1.0f, 1.0f, __int_as_float(0)));
  sts_f4(st_a + kStB, make_float4(__int_as_float(-1), __int_as_float(P.sample_begin), 0.0f, __uint_as_float(REF_NONE)));
  const int s_last = P.sample_begin + P.sample_count;
  bool alive = false;
  unsigned int n_rays = 0;
  unsigned int cn[COUNT ? CN_COUNT : 1];
  if (COUNT)
    for (int i = 0; i < CN_COUNT; i++) cn[i] = 0;
  float3 o = f3(0, 0, 0), d = f3(0, 0, 1);

  // Every iteration = (regenerate dead lanes) + (one path segment for all lanes).  The iteration
  // boundary is a warp vote, so the 32 lanes reconverge here; lanes that ran out of work idle
  // until the whole warp is done (only at the very end of the render).
  // (Two finer-grained alternatives were measured and lost, see profiles/r03_render_phase_sched.md:
  //  every lane a NODE/LEAF/SHADE state machine with the warp executing the most populated phase, and a
  //  resumable traversal that breaks out to shade/refill finished lanes once < 8..24 lanes still traverse.
  //  Shading a half-empty warp twice costs more than the shallow traversal saves.)
  const unsigned FULL = 0xFFFFFFFFu;
  const bool media = !AOV && sc.n_media != 0;
  bool done = false;
  // the traversal stack: local memory, or — when the launch has the room — one 32-bit entry per level in shared memory
  typename std::conditional<SSTACK, TravStackS, TravStack>::type st;
  if constexpr (SSTACK) {
    st.base = opaque_u32(uint32_t(__cvta_generic_to_shared(s_nodes)) + P.stack_off) + 4u * threadIdx.x;
    st.stride = 4u * kRenderThreads;
#if RT_CHECKS
    st.levels = P.stack_levels;
#endif
  }
  for (;;) {
    if (!alive && !done) {
      const float4 B0 = lds_f4(st_a + kStB);
      int pixel = __float_as_int(B0.x), s = __float_as_int(B0.y);
      PathKey key{P.key, uint32_t(pixel), 0u};
      // a work item holds a power-of-two number of samples (the host rounds P.chunk down): "my item is used up" is a
      // mask test on the next sample index — no end-of-item register; initially s == sample_begin, which reads as used up
      if ((((unsigned)(s - P.sample_begin)) & (unsigned)(P.chunk - 1)) == 0u || s >= s_last) {
        done = true;
        for (;;) {
          const unsigned long long it = atomicAdd(P.counters, 1ull);  // taken when needed: no prefetched candidate to keep
          if (it >= (unsigned long long)P.n_items) break;
          const unsigned int item = (unsigned int)it;
          const unsigned int chunk = item / P.per_chunk, q = item - chunk * P.per_chunk;
          unsigned int view = 0u, vq = q;  // VIEWS: (view, tile, lane) within the chunk, a warp's 32 items = one tile of one view
          if constexpr (VIEWS) view = q / P.view_items, vq = q - view * P.view_items;
          const unsigned int tile = vq >> 5, lane = vq & 31u;
          const int px = int(tile % (unsigned)P.tiles_x) * 8 + int(lane & 7u);
          const int py = int(tile / (unsigned)P.tiles_x) * 4 + int(lane >> 3);
          // (a view with max_depth <= 0 traces nothing, as rt_render launches nothing for it: its items are skipped)
          if (px < P.cam.W && py < P.cam.H && (!VIEWS || cam_of(int(view * P.view_pixels)).max_depth > 0)) {
            s = P.sample_begin + int(chunk) * P.chunk;
            if (s < s_last) {
              pixel = py * P.cam.W + px;
              if constexpr (VIEWS) pixel += int(view * P.view_pixels);
              key.pixel = uint32_t(pixel);
              done = false;
              break;
            }
          }
        }
      }
      if (!done) {
        // ---- camera::get_ray (camera.hpp:139-162): jitter, defocus disk, shutter time ----
        key.sample = uint32_t(s++);
        const CameraDev& cam = cam_of(pixel);
        const int vpixel = view_pixel(pixel);
        if constexpr (VIEWS) key.pixel = uint32_t(vpixel);
        const int py = vpixel / P.cam.W, px = vpixel - py * P.cam.W;
        uint4 r0 = rng_block(key, 0u, 0u);
        float ox = u01(r0.x) - 0.5f, oy = u01(r0.y) - 0.5f;
        float time = u01(r0.z);
        if (AOV) ox = oy = time = 0.0f;
        float3 dir = fma3(float(px) + ox, cam.du, fma3(float(py) + oy, cam.dv, cam.p00c));
        o = cam.center;
        if (!AOV && cam.defocus) {  // uniform disk: r = sqrt(u), phi = 2 pi v (== rejection sampling in law)
          uint4 r1 = rng_block(key, 0u, 1u);
          float rr = sqrtf(u01(r1.x)), sn, cs;
          sincos_2pi(u01(r1.y), sn, cs);
          float3 off = fma3(rr * cs, cam.ddu, (rr * sn) * cam.ddv);
          o = o + off;
          dir = dir - off;
        }
        d = dir;
        sts_f4(st_a, make_float4(1.0f, 1.0f, 1.0f, __int_as_float(cam.max_depth)));
        sts_f4(st_a + kStB, make_float4(__int_as_float(pixel), __int_as_float(s), time, __uint_as_float(REF_NONE)));
        alive = cam.max_depth > 0;
      }
    }
    const unsigned live = __ballot_sync(FULL, alive);
    if (live == 0u) {
      if (__all_sync(FULL, done)) break;
      continue;
    }
    n_rays += __popc(live);  // warp-uniform: the count lives in the uniform datapath, not in a lane register
    // ---- one segment of ray_color (camera.hpp:180-232) -----------------------------------
    // the ray's Philox counter, read back for the scene-enclosing media (every ray) and — lazily — for a medium leaf
    auto key_of = [&](PathKey& k, uint32_t& b) {
      const float4 A = lds_f4(st_a), B = lds_f4(st_a + kStB);
      if constexpr (VIEWS) {
        k = PathKey{P.key, uint32_t(view_pixel(__float_as_int(B.x))), uint32_t(__float_as_int(B.y) - 1)};
        b = uint32_t(cam_of(__float_as_int(B.x)).max_depth - __float_as_int(A.w)) + 1u;
      } else {
        k = PathKey{P.key, uint32_t(__float_as_int(B.x)), uint32_t(__float_as_int(B.y) - 1)};
        b = uint32_t(P.cam.max_depth - __float_as_int(A.w)) + 1u;
      }
    };
    auto aux_of = [&](float& t, uint32_t& sk) {
      float tt, ss;
      asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(tt), "=f"(ss) : "r"(st_a + kStB + 8u));
      t = tt, sk = __float_as_uint(ss);
    };
    Hit h = closest_hit_keyfn<COUNT, ALL_SMEM>(sc, ns, o, d, 0.001f, INF, media, key_of, aux_of, cn, alive, ls, st);
    if constexpr (AOV) {
      if (alive) {
        const float4 A = lds_f4(st_a), B = lds_f4(st_a + kStB);
        const int pixel = __float_as_int(B.x);
        const bool first = __float_as_int(A.w) == P.cam.max_depth;
        int pid = -1;
        float t = INF;
        Surface sf;
        sf.n = f3(0.0f, 0.0f, 0.0f), sf.front = false;
        if (h.ref != REF_NONE) {
          sf = surface_at(sc, h, o, d, 0.0f);
          const uint32_t type = h.ref >> 30, idx = h.ref & 0x3FFFFFFFu;
          if (type == REF_BOX) {  // the reference quad behind this face of the box (scene_build.hpp, box_meta)
            const int4 meta = sc.box_meta[idx >> 3];
            pid = sc.xquads[meta.y + int((uint32_t(meta.z) >> (4u * (idx & 7u))) & 7u)].pid;
          } else {
            pid = type == REF_SPHERE ? sc.xspheres[idx].pid : (type == REF_QUAD ? sc.xquads[idx].pid : -2 - int(idx));
          }
          t = sf.t;
        }
        alive = false;
        if (first) {
          P.aov_id[pixel] = pid, P.aov_t[pixel] = t;
          P.aov_n[3 * pixel] = sf.n.x, P.aov_n[3 * pixel + 1] = sf.n.y, P.aov_n[3 * pixel + 2] = sf.n.z;
          if (P.aov_b) {
            float* r = P.aov_b + kAovBounce * pixel;
            bool cont = false;
            float3 d_out = f3(0.0f, 0.0f, 0.0f);
            if (h.ref != REF_NONE) {  // the shade of rt_render's first segment (below), sample 0
              const uint4 rnd = rng_block(PathKey{P.key, uint32_t(pixel), uint32_t(__float_as_int(B.y) - 1)}, 1u, 0u);
              float3 emit, atten;
              cont = scatter_ray<false>(sc, sf, d, rnd, emit, atten, d_out, nullptr);
            }
            for (int k = 0; k < kAovBounce; k++) r[k] = 0.0f;
            r[10] = __int_as_float(RT_NO_BOUNCE);
            if (cont) {
              o = sf.p;
              d = d_out;
              r[0] = o.x, r[1] = o.y, r[2] = o.z, r[3] = d.x, r[4] = d.y, r[5] = d.z;
              const uint32_t skip = (h.ref >> 30) == REF_MEDIUM ? REF_NONE : h.ref;
              sts_f4(st_a, make_float4(A.x, A.y, A.z, __int_as_float(__float_as_int(A.w) - 1)));
              asm volatile("st.shared.u32 [%0], %1;" ::"r"(st_a + kStB + 12u), "r"(skip) : "memory");
              alive = true;
            }
          }
        } else {
          float* r = P.aov_b + kAovBounce * pixel;
          r[6] = sf.n.x, r[7] = sf.n.y, r[8] = sf.n.z, r[9] = t, r[10] = __int_as_float(pid), r[11] = sf.front ? 1.0f : 0.0f;
        }
      }
      continue;
    }
    // COOP: world.hit's record for the lanes that hit something (hit_record, face normal, uv: surface_at) is built BEFORE
    // the shade, where the warp is still converged, and the lanes whose hit lands on a noise texture get their Perlin
    // turbulence evaluated by the whole warp (rt_device.cuh, coop_noise_turb: seven lanes per requester, one octave each)
    // instead of one lane after the other inside the divergent shade below.  Same bits as the serial loop.
    Surface sf;
    float turb_pre = -1.0f;  // a turbulence is |.| >= 0: negative = not evaluated here
    if constexpr (COOP) {
      const bool hit_something = alive && h.ref != REF_NONE;
      if (hit_something) {
        float tm, sk;
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(tm), "=f"(sk) : "r"(st_a + kStB + 8u));
        sf = surface_at(sc, h, o, d, tm);
      }
      const int want = hit_something ? noise_request(sc, sf.material, sf.p) : -1;
      turb_pre = coop_noise_turb(sc, want, hit_something ? sf.p : f3(0.0f, 0.0f, 0.0f), threadIdx.x & 31u);
    }
    if (alive) {
      const float4 A = lds_f4(st_a), B = lds_f4(st_a + kStB);
      float3 beta = f3(A.x, A.y, A.z);
      int depth = __float_as_int(A.w);
      const int pixel = __float_as_int(B.x);
      const float time = B.z;
      const CameraDev& cam = cam_of(pixel);
      const PathKey key{P.key, uint32_t(view_pixel(pixel)), uint32_t(__float_as_int(B.y) - 1)};
      const uint32_t bounce = uint32_t(cam.max_depth - depth) + 1u;
      // The radiance of a path is beta x (emission | background) at its LAST vertex: no material of the reference both
      // emits and scatters (diffuse_light::scatter is false, material.hpp:36; every other emitted() is black), so no
      // running sum lives across the traversal.
      float3 L = f3(0.0f, 0.0f, 0.0f);
      if (h.ref == REF_NONE) {
        L = L + beta * cam.bg;
        alive = false;
      } else {
        const uint4 rnd = rng_block(key, bounce, 0u);
        if constexpr (!COOP) sf = surface_at(sc, h, o, d, time);
        float3 emit, atten, d_out;
        bool cont = scatter_ray<COUNT>(sc, sf, d, rnd, emit, atten, d_out, cn, turb_pre);
        L = L + beta * emit;
        if (cont) {
          beta = beta * atten;
          o = sf.p;
          d = d_out;
          const uint32_t skip = (h.ref >> 30) == REF_MEDIUM ? REF_NONE : h.ref;
          alive = --depth > 0;
          sts_f4(st_a, make_float4(beta.x, beta.y, beta.z, __int_as_float(depth)));
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(st_a + kStB + 12u), "r"(skip) : "memory");
        } else {
          alive = false;
        }
      }
      if (!alive) {
        // the finished sample, quantised to 2^-32, straight into the int64 accumulator (red.add.u64:
        // fire-and-forget, ~3 per 5 rays).  Integer adds commute, so the image does not depend on
        // which lane / CTA / launch / GPU contributed which sample.
        RT_CHECK(pixel >= 0 && (unsigned long long)pixel * 3ull + 2ull < P.n_values, CHK_PIXEL);
        unsigned long long* dst = P.accum + 3ull * (unsigned long long)pixel;
        const long long fr = to_fixed(L.x), fg = to_fixed(L.y), fb = to_fixed(L.z);
        if (fr) atomicAdd(dst + 0, (unsigned long long)fr);
        if (fg) atomicAdd(dst + 1, (unsigned long long)fg);
        if (fb) atomicAdd(dst + 2, (unsigned long long)fb);
      }
    }
  }
  // ---- counters: warp-reduce, one atomic per warp ---------------------------------------
  unsigned int rays = n_rays;
  if ((threadIdx.x & 31) == 0) atomicAdd(P.counters + 1, (unsigned long long)rays);
  if (COUNT)
    for (int i = 0; i < CN_COUNT; i++)
      if (cn[i]) atomicAdd(P.counters + 4 + i, (unsigned long long)cn[i]);
}

}  // namespace rtb200
#include "rt_stream.cuh"
#include "rt_refill.cuh"
namespace rtb200 {

// ---- write_color (common/color.hpp:26-58) on the device, in double like the reference ----
__global__ void finalize_kernel(const long long* __restrict__ accum, long long n_values, double scale, float* __restrict__ radiance,
                                unsigned char* __restrict__ rgb8) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_values) return;
  double lin = double(accum[i]) * (1.0 / 4294967296.0) * scale;
  if (radiance) radiance[i] = float(lin);
  if (rgb8) {
    double g = lin > 0.0 ? sqrt(lin) : 0.0;
    const double hi = double(0.999f);
    g = g < 0.0 ? 0.0 : (g > hi ? hi : g);
    rgb8[i] = (unsigned char)(int(256 * g));
  }
}

// ---- closest-hit queries for the parity harness ---------------------------------------------
struct TraceParams {
  DeviceScene sc;
  long long n;
  const double* origin;
  const double* direction;
  const double* time;
  const uint32_t* skip;  // fp32 mode: the device ref each ray starts on (rt_trace_rays_from), NULL = none
  double tmin, tmax;
  int flags;
  unsigned long long seed;
  int* prim_id;
  double* t;
  double* normal;
  unsigned char* front;
  int smem_nodes;
};

// fp32 conservative traversal; EVERY candidate primitive is evaluated by the fp64 routines that
// follow sphere::hit / quad::hit operation for operation, and the winner is chosen by the
// reference's visit order on exact ties (hittable_list.hpp:47-61, SURVEY.md A.4-A.5).
__device__ void exact_closest(const DeviceScene& sc, const NodeSource& ns, const XRay& r, double tmin, double tmax, int& out_pid, XRec& out_rec) {
  float3 o = f3(float(r.o.x.v), float(r.o.y.v), float(r.o.z.v)), d = f3(float(r.d.x.v), float(r.d.y.v), float(r.d.z.v));
  float3 inv = f3(fabsf(d.x) > 1e-30f ? 1.0f / d.x : copysignf(1e30f, d.x), fabsf(d.y) > 1e-30f ? 1.0f / d.y : copysignf(1e30f, d.y),
                  fabsf(d.z) > 1e-30f ? 1.0f / d.z : copysignf(1e30f, d.z));
  float3 ood = o * inv;
  const float eps = 4e-6f * (sc.scene_abs_max + fabsf(o.x) + fabsf(o.y) + fabsf(o.z));
  const float tminf = float(tmin) - fabsf(float(tmin)) * 1e-5f - 1e-30f;
  double best_t = tmax;
  int best_order = -1, best_is_quad = 0;
  out_pid = -1;
  int stack[kStackDepth];
  int sp = 0, cur = 0;
  for (;;) {
    if (cur >= 0) {
      float4 a, b, c;
      int c0, c1;
      load_node(ns, cur, a, b, c, c0, c1);
      float bestf = best_t < 3e38 ? float(best_t) * (1.0f + 1e-5f) + 1e-30f : __int_as_float(0x7f800000);
      float x0 = fmaf(a.x - eps, inv.x, -ood.x), x1 = fmaf(a.w + eps, inv.x, -ood.x);
      float y0 = fmaf(a.y - eps, inv.y, -ood.y), y1 = fmaf(b.x + eps, inv.y, -ood.y);
      float z0 = fmaf(a.z - eps, inv.z, -ood.z), z1 = fmaf(b.y + eps, inv.z, -ood.z);
      float n0 = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), tminf));
      float f0 = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), bestf));
      x0 = fmaf(b.z - eps, inv.x, -ood.x), x1 = fmaf(c.y + eps, inv.x, -ood.x);
      y0 = fmaf(b.w - eps, inv.y, -ood.y), y1 = fmaf(c.z + eps, inv.y, -ood.y);
      z0 = fmaf(c.x - eps, inv.z, -ood.z), z1 = fmaf(c.w + eps, inv.z, -ood.z);
      float n1 = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), tminf));
      float f1 = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), bestf));
      // an empty child has lo=+inf, hi=-inf: lo-eps = +inf, hi+eps = -inf, still never entered
      bool h0 = n0 <= f0 * (1.0f + 1e-5f) + 1e-30f, h1 = n1 <= f1 * (1.0f + 1e-5f) + 1e-30f;
      if (h0 && h1) {
        if (sp < kStackDepth) stack[sp++] = c1;
        cur = c0;
        continue;
      }
      if (h0) { cur = c0; continue; }
      if (h1) { cur = c1; continue; }
    } else {
      int code = ~cur;
      int first = code >> 3, count = (code & 7) + 1;
      for (int k = 0; k < count; k++) {
        uint32_t ref = sc.leaf_refs[first + k];
        uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
        if (ref == REF_NONE || type == REF_MEDIUM) continue;  // media are transparent here (SURVEY §8(c))
        // a box leaf stands for its six quads (quad.hpp:145-155), evaluated one by one like the reference does
        const int n_sub = type == REF_BOX ? 6 : 1;
        const int sub0 = type == REF_BOX ? sc.box_meta[idx >> 3].y : int(idx);
        for (int j = 0; j < n_sub; j++) {
          XRec rec;
          int order, pid, is_quad = type != REF_SPHERE;
          bool ok;
          if (is_quad) {
            const XQuad& q = sc.xquads[sub0 + j];
            ok = exact_quad(sc, q, r, tmin, tmax, rec);
            order = q.order, pid = q.pid;
          } else {
            const XSphere& q = sc.xspheres[idx];
            ok = exact_sphere(sc, q, r, tmin, tmax, rec);
            order = q.order, pid = q.pid;
          }
          if (!ok) continue;
          bool take;
          if (best_order < 0) {
            take = is_quad ? rec.t.v <= best_t : rec.t.v < best_t;
          } else if (rec.t.v != best_t) {
            take = rec.t.v < best_t;
          } else {  // exact tie: the later visit wins iff it is a quad (contains vs surrounds)
            take = order > best_order ? is_quad != 0 : best_is_quad == 0;
          }
          if (take) best_t = rec.t.v, best_order = order, best_is_quad = is_quad, out_pid = pid, out_rec = rec;
        }
      }
    }
    if (sp == 0) return;
    cur = stack[--sp];
  }
}

__global__ void __launch_bounds__(256) trace_kernel(const __grid_constant__ TraceParams P) {
  extern __shared__ float4 s_nodes[];
  for (int i = threadIdx.x; i < 4 * P.smem_nodes; i += blockDim.x) s_nodes[i] = P.sc.nodes[i];
  __syncthreads();
  const NodeSource ns = node_source(s_nodes, P.sc.nodes, P.smem_nodes, P.sc.n_nodes);
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  const DeviceScene& sc = P.sc;
  double tm = P.time ? P.time[i] : 0.0;
  int pid = -1;
  double t = INFINITY, nx = 0, ny = 0, nz = 0;
  bool front = false;
  if (P.flags & RT_TRACE_EXACT) {
    XRay r{SV(P.origin + 3 * i), SV(P.direction + 3 * i), S(tm)};
    XRec rec;
    exact_closest(sc, ns, r, P.tmin, P.tmax, pid, rec);
    if (pid >= 0) t = rec.t.v, nx = rec.n.x.v, ny = rec.n.y.v, nz = rec.n.z.v, front = rec.front;
  } else {
    float3 o = f3(float(P.origin[3 * i]), float(P.origin[3 * i + 1]), float(P.origin[3 * i + 2]));
    float3 d = f3(float(P.direction[3 * i]), float(P.direction[3 * i + 1]), float(P.direction[3 * i + 2]));
    PathKey key{make_uint2((unsigned)P.seed, (unsigned)(P.seed >> 32)), (uint32_t)i, 0u};
    bool media = sc.n_media && !(P.flags & RT_TRACE_SKIP_MEDIA);
    float tmaxf = P.tmax < 3e38 ? float(P.tmax) : __int_as_float(0x7f800000);
    Hit h = closest_hit<false>(sc, ns, o, d, float(tm), float(P.tmin), tmaxf, P.skip ? P.skip[i] : REF_NONE, media, key, 1u, nullptr);
    if (h.ref != REF_NONE) {
      Surface sf = surface_at(sc, h, o, d, float(tm));
      uint32_t type = h.ref >> 30, idx = h.ref & 0x3FFFFFFFu;
      if (type == REF_BOX) {
        const int4 meta = sc.box_meta[idx >> 3];
        pid = sc.xquads[meta.y + int((uint32_t(meta.z) >> (4u * (idx & 7u))) & 7u)].pid;
      } else {
        pid = type == REF_SPHERE ? sc.xspheres[idx].pid : (type == REF_QUAD ? sc.xquads[idx].pid : -2 - int(idx));
      }
      t = sf.t, nx = sf.n.x, ny = sf.n.y, nz = sf.n.z, front = sf.front;
    }
  }
  if (P.prim_id) P.prim_id[i] = pid;
  if (P.t) P.t[i] = t;
  if (P.normal) P.normal[3 * i] = nx, P.normal[3 * i + 1] = ny, P.normal[3 * i + 2] = nz;
  if (P.front) P.front[i] = front;
}

// pixel-centre rays in double with the operation order of camera::get_ray at zero jitter
// (camera.hpp:147,156): pixel00 + (i * du) + (j * dv), direction = sample - center.
__global__ void center_rays_kernel(rt_camera_frame f, double* origin, double* direction) {
  int i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
  if (i >= f.image_width) return;
  sv p00 = SV(f.pixel00_loc), du = SV(f.pixel_delta_u), dv = SV(f.pixel_delta_v), c = SV(f.center);
  sv ps = p00 + (S(double(i) + 0.0) * du) + (S(double(j) + 0.0) * dv);
  sv dir = ps - c;
  long long p = ((long long)j * f.image_width + i) * 3;
  origin[p] = c.x.v, origin[p + 1] = c.y.v, origin[p + 2] = c.z.v;
  direction[p] = dir.x.v, direction[p + 1] = dir.y.v, direction[p + 2] = dir.z.v;
}

__global__ void medium_spans_kernel(DeviceScene sc, int medium, long long n, const double* origin, const double* direction, const double* time, double* t1,
                                    double* t2) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float3 o = f3(float(origin[3 * i]), float(origin[3 * i + 1]), float(origin[3 * i + 2]));
  float3 d = f3(float(direction[3 * i]), float(direction[3 * i + 1]), float(direction[3 * i + 2]));
  float a = NAN, b = NAN;
  const float INF = __int_as_float(0x7f800000);
  const DMedium m = sc.media[medium];
  float x1, x2;
  bool both = medium_span(sc, m, o, d, time ? float(time[i]) : 0.0f, x1, x2);
  if (x1 != INF) a = x1;
  if (both) b = x2;
  t1[i] = a, t2[i] = b;
}

__global__ void eval_texture_kernel(DeviceScene sc, int tex, long long n, const double* uvp, float* rgb) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* q = uvp + 5 * i;
  float3 c = texture_value<false>(sc, tex, float(q[0]), float(q[1]), f3(float(q[2]), float(q[3]), float(q[4])), nullptr);
  rgb[3 * i] = c.x, rgb[3 * i + 1] = c.y, rgb[3 * i + 2] = c.z;
}

__global__ void eval_scatter_kernel(DeviceScene sc, int material, long long n, unsigned long long seed, const double* dir_in, const double* normal,
                                    const unsigned char* front, float* dir_out, float* atten, unsigned char* scattered) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Surface s;
  s.p = f3(0, 0, 0);
  s.n = f3(float(normal[3 * i]), float(normal[3 * i + 1]), float(normal[3 * i + 2]));
  s.u = s.v = 0.0f;
  s.front = front[i] != 0;
  s.material = material;
  PathKey key{make_uint2((unsigned)seed, (unsigned)(seed >> 32)), (uint32_t)i, (uint32_t)(i >> 32)};
  uint4 rnd = rng_block(key, 1u, 0u);
  float3 emit, a = f3(0, 0, 0), dout = f3(0, 0, 0);
  bool ok = scatter_ray<false>(sc, s, f3(float(dir_in[3 * i]), float(dir_in[3 * i + 1]), float(dir_in[3 * i + 2])), rnd, emit, a, dout, nullptr);
  scattered[i] = ok;
  dir_out[3 * i] = dout.x, dir_out[3 * i + 1] = dout.y, dir_out[3 * i + 2] = dout.z;
  atten[3 * i] = a.x, atten[3 * i + 1] = a.y, atten[3 * i + 2] = a.z;
}

}  // namespace rtb200

// =============================================================================================
// C-ABI
// =============================================================================================
using namespace rtb200;

namespace {
std::mutex g_err_mutex;
std::string g_init_error = "";
// the live contexts of this process: rt_render_opts.peer_accum must be the accumulator of one of them
std::vector<struct ::rt_ctx*> g_contexts;

template <typename T>
struct DevArray {
  T* ptr = nullptr;
  size_t count = 0;
};
}  // namespace

struct rt_ctx {
  int device = 0;
  int sm_count = 0;
  size_t smem_optin = 0;
  float noise_share = 0.0f;  // share of the BVH's primitives whose material can end in a noise texture (rt_upload_scene)
  // Process-environment knobs (experiments and test hooks, none needed for normal use), read ONCE when the context is
  // created: rt_render itself never looks at the environment, its behaviour is a function of its arguments and the context.
  //   RT_B200_KERNEL=mega|stream|refill  default render kernel        RT_B200_NO_STAGING=1   BVH top levels only in shared memory
  //   RT_B200_CHUNK_MAX=n                samples per work item <= n   RT_B200_MAX_CHUNKS=n   launches of <= n sample chunks (test hook)
  //   RT_B200_NO_SMEM_STACK=1            megakernel traversal stacks in local memory (test hook: every plan under one scene)
  struct Knobs {
    int kernel = 0;
    int chunk_max = 0, max_chunks = 0;
    bool no_staging = false, no_smem_stack = false;
  } knobs;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  bool timed = false;
  std::string error;
  // the device scene lives in ONE grow-only arena filled by ONE copy from a pinned staging buffer: re-uploading a scene
  // (bench.py's e2e does it every step) then makes no cudaMalloc / cudaFree at all — those calls synchronise the device
  // and took 60-500 ms per upload inside a process that also holds torch's allocations (gpurun_out/bench_n1_final4.json)
  unsigned char* arena = nullptr;
  size_t arena_bytes = 0;
  unsigned char* staging = nullptr;  // cudaHostAlloc
  size_t staging_bytes = 0;
  DeviceScene sc;
  bool has_scene = false;
  HostScene host;
  unsigned long long* accum = nullptr;
  size_t accum_values = 0;
  int acc_w = 0, acc_h = 0;
  int acc_views = 0;  // images the accumulator holds: 1 after rt_render / rt_upload_accum, n_views after rt_render_views
  // rt_render_views' camera table: one CameraDev per view on the device, filled by a stream-ordered copy from a pinned
  // buffer that outlives it (ev_cams marks when that copy has read it).  Both only grow: with peer access enabled a
  // cudaMalloc costs tens of milliseconds.
  CameraDev* cams_dev = nullptr;
  CameraDev* cams_host = nullptr;
  int cams_cap = 0;
  cudaEvent_t ev_cams = nullptr;
  unsigned long long* counters = nullptr;  // 32 x u64: [0] next item, [1] rays, [2] samples, [4..] census
  unsigned long long rays_total = 0, samples_total = 0;
  int smem_nodes = 0;
  int launches = 0;
  void* scratch = nullptr;  // rt_download's device-side staging buffer
  size_t scratch_bytes = 0;
  unsigned long long* reduce_buf = nullptr;  // fused multi-GPU reduce: peers add their accumulators here
  size_t reduce_values = 0;
};

#define RT_CUDA(ctx, call)                                                                          \
  do {                                                                                              \
    cudaError_t e_ = (call);                                                                        \
    if (e_ != cudaSuccess) {                                                                        \
      (ctx)->error = std::string(#call) + ": " + cudaGetErrorString(e_);                            \
      return RT_ERR_CUDA;                                                                           \
    }                                                                                               \
  } while (0)

// RT_B200_DEBUG=1: entry points report a CUDA error that is already pending when they start / still pending when they
// return, on stderr.  A non-sticky error left by an unrelated earlier call (anywhere in the process) would otherwise be
// blamed on the next cudaGetLastError() after one of OUR launches; every entry point clears it first.
static void debug_error(const char* where, bool clear) {
  cudaError_t e = clear ? cudaGetLastError() : cudaPeekAtLastError();
  if (e != cudaSuccess && std::getenv("RT_B200_DEBUG"))
    std::fprintf(stderr, "[rt_b200] %s: CUDA error '%s' %s\n", where, cudaGetErrorString(e), clear ? "was pending (cleared)" : "left pending");
}
struct DebugScope {
  const char* name;
  explicit DebugScope(const char* n) : name(n) { debug_error(n, true); }
  ~DebugScope() { debug_error(name, false); }
};

static int fail(rt_ctx* ctx, int code, const std::string& msg) {
  ctx->error = msg;
  return code;
}

namespace {
struct ScenePiece {
  const void* src;
  size_t bytes;
  void* field;  // address of the DeviceScene pointer member this array is published through
  size_t offset;
};
}  // namespace

// Packs the pieces (256-byte aligned) into the pinned staging buffer, copies them to the arena in one H2D transfer and
// publishes the device pointers.  Both buffers only ever grow.
static int upload_pieces(rt_ctx* ctx, std::vector<ScenePiece>& pieces) {
  size_t total = 0;
  for (ScenePiece& p : pieces) {
    p.offset = total;
    total += (std::max<size_t>(p.bytes, 1) + 255) & ~size_t(255);
  }
  if (total > ctx->arena_bytes) {
    const size_t want = total + total / 2;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->arena);
    ctx->arena = nullptr, ctx->arena_bytes = 0;
    RT_CUDA(ctx, cudaMalloc(&ctx->arena, want));
    ctx->arena_bytes = want;
  }
  if (total > ctx->staging_bytes) {
    const size_t want = total + total / 2;
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFreeHost(ctx->staging);
    ctx->staging = nullptr, ctx->staging_bytes = 0;
    RT_CUDA(ctx, cudaHostAlloc(&ctx->staging, want, cudaHostAllocDefault));
    ctx->staging_bytes = want;
  }
  for (const ScenePiece& p : pieces) {
    if (p.bytes) std::memcpy(ctx->staging + p.offset, p.src, p.bytes);
    const void* dev = ctx->arena + p.offset;
    std::memcpy(p.field, &dev, sizeof dev);
  }
  RT_CUDA(ctx, cudaMemcpyAsync(ctx->arena, ctx->staging, total, cudaMemcpyHostToDevice, ctx->stream));
  return RT_OK;
}

static void free_scene(rt_ctx* ctx) {  // the arena stays: the next rt_upload_scene overwrites it
  ctx->has_scene = false;
}

// ---- parity-harness entry points -----------------------------------------------------------
namespace {
struct Scratch {
  std::vector<void*> ptrs;
  ~Scratch() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <typename T>
  T* alloc(size_t n) {
    void* p = nullptr;
    if (cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)) != cudaSuccess) return nullptr;
    ptrs.push_back(p);
    return static_cast<T*>(p);
  }
  template <typename T>
  T* to_device(const T* host, size_t n) {
    if (!host) return nullptr;
    T* p = alloc<T>(n);
    if (p && cudaMemcpy(p, host, n * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
    return p;
  }
};

int run_trace(rt_ctx* ctx, long long n, const double* d_origin, const double* d_dir, const double* d_time, const uint32_t* d_skip, double tmin, double tmax,
              int flags, int32_t* prim_id, double* t, double* normal, uint8_t* front_face, Scratch& sx) {
  TraceParams P;
  std::memset(&P, 0, sizeof P);
  P.sc = ctx->sc;
  P.n = n;
  P.origin = d_origin, P.direction = d_dir, P.time = d_time, P.skip = d_skip;
  P.tmin = tmin, P.tmax = tmax, P.flags = flags, P.seed = 0;
  P.prim_id = prim_id ? sx.alloc<int>(size_t(n)) : nullptr;
  P.t = t ? sx.alloc<double>(size_t(n)) : nullptr;
  P.normal = normal ? sx.alloc<double>(size_t(3 * n)) : nullptr;
  P.front = front_face ? sx.alloc<unsigned char>(size_t(n)) : nullptr;
  if ((prim_id && !P.prim_id) || (t && !P.t) || (normal && !P.normal) || (front_face && !P.front)) return fail(ctx, RT_ERR_CUDA, "cudaMalloc failed");
  P.smem_nodes = std::min(ctx->smem_nodes, int((ctx->smem_optin > 8192 ? ctx->smem_optin - 4096 : 0) / 64));
  size_t smem = size_t(P.smem_nodes) * 64;
  RT_CUDA(ctx, cudaFuncSetAttribute(trace_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
  if (n > 0) {
    trace_kernel<<<unsigned((n + 255) / 256), 256, smem, ctx->stream>>>(P);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
  }
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (prim_id) RT_CUDA(ctx, cudaMemcpy(prim_id, P.prim_id, size_t(n) * 4, cudaMemcpyDeviceToHost));
  if (t) RT_CUDA(ctx, cudaMemcpy(t, P.t, size_t(n) * 8, cudaMemcpyDeviceToHost));
  if (normal) RT_CUDA(ctx, cudaMemcpy(normal, P.normal, size_t(n) * 24, cudaMemcpyDeviceToHost));
  if (front_face) RT_CUDA(ctx, cudaMemcpy(front_face, P.front, size_t(n), cudaMemcpyDeviceToHost));
  return RT_OK;
}

// Reference primitive id -> the device ref a ray that starts on it carries into the traversal (the `skip` rt_render sets
// after a scatter): a sphere or quad of the BVH is its own ref; a quad of a box() list is that box with the face bits
// (box_meta's face -> quad nibbles, inverted).  Only primitives the BVH references have one; an id that names two
// different device primitives (a hittable reached twice through the graph) cannot be resolved.  Both are refused.
int start_refs(rt_ctx* ctx, long long n, const int32_t* start_prim, std::vector<uint32_t>& out) {
  const HostScene& h = ctx->host;
  std::vector<uint32_t> ref_of;  // indexed by reference primitive id
  auto add = [&](int pid, uint32_t ref) {
    if (pid < 0) return true;
    if (size_t(pid) >= ref_of.size()) ref_of.resize(size_t(pid) + 1, REF_NONE);
    if (ref_of[size_t(pid)] != REF_NONE && ref_of[size_t(pid)] != ref) return false;
    ref_of[size_t(pid)] = ref;
    return true;
  };
  for (uint32_t ref : h.leaf_refs) {
    if (ref == REF_NONE) continue;
    const uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    bool ok = true;
    if (type == REF_SPHERE) {
      ok = add(h.xspheres[idx].pid, ref);
    } else if (type == REF_QUAD) {
      ok = add(h.xquads[idx].pid, ref);
    } else if (type == REF_BOX) {
      const uint32_t b = idx >> 3;
      const int4 meta = h.box_meta[b];
      for (uint32_t f = 0; f < 6 && ok; f++)
        ok = add(h.xquads[size_t(meta.y) + ((uint32_t(meta.z) >> (4u * f)) & 7u)].pid, make_ref(REF_BOX, (b << 3) | f));
    }
    if (!ok) return fail(ctx, RT_ERR_INVALID, "start_prim: a primitive id names more than one device primitive");
  }
  out.resize(size_t(n));
  for (long long i = 0; i < n; i++) {
    const int32_t pid = start_prim[i];
    if (pid == -1) {
      out[size_t(i)] = REF_NONE;
    } else if (pid < 0 || size_t(pid) >= ref_of.size() || ref_of[size_t(pid)] == REF_NONE) {
      return fail(ctx, RT_ERR_INVALID, "start_prim[" + std::to_string(i) + "] = " + std::to_string(pid) + " is not a primitive of the traversal");
    } else {
      out[size_t(i)] = ref_of[size_t(pid)];
    }
  }
  return RT_OK;
}
}  // namespace

extern "C" {

int rt_abi_sizeof(int which) {
  switch (which) {
    case 0: return int(sizeof(rt_hittable));
    case 1: return int(sizeof(rt_material));
    case 2: return int(sizeof(rt_texture));
    case 3: return int(sizeof(rt_image));
    case 4: return int(sizeof(rt_perlin));
    case 5: return int(sizeof(rt_scene_desc));
    case 6: return int(sizeof(rt_camera_desc));
    case 7: return int(sizeof(rt_camera_frame));
    case 8: return int(sizeof(rt_render_opts));
    case 9: return int(sizeof(rt_stats));
  }
  return -1;
}

// camera::initialize (src/core/camera.hpp:76-136), double, same operation order.
int rt_camera_initialize(const rt_camera_desc* c, rt_camera_frame* f) {
  if (!c || !f) return RT_ERR_INVALID;
  using namespace build_detail;
  const double pi = 3.1415926535897932385;
  int W = c->image_width;
  int H = static_cast<int>(c->image_width / c->aspect_ratio);
  H = H < 1 ? 1 : H;
  f->image_width = W;
  f->image_height = H;
  f->pixel_samples_scale = 1.0f / c->samples_per_pixel;  // float / int -> float (:83)
  double theta = c->vfov * pi / 180.0f;
  double h = std::tan(theta / 2);
  double vh = 2 * h * c->focus_dist;
  double vw = vh * (static_cast<double>(W) / H);
  d3 from = ld(c->lookfrom), at = ld(c->lookat), vup = ld(c->vup);
  auto unit = [](d3 v) { return (1 / std::sqrt(v.x * v.x + v.y * v.y + v.z * v.z)) * v; };
  d3 w = unit(from - at);
  d3 u = unit(cross(vup, w));
  d3 v = cross(w, u);
  d3 vu = vw * u;
  d3 vv = vh * d3{-v.x, -v.y, -v.z};
  d3 du = (1 / double(W)) * vu;
  d3 dv = (1 / double(H)) * vv;
  d3 ul = from - (c->focus_dist * w) - (1 / 2.0) * vu - (1 / 2.0) * vv;
  d3 p00 = ul + 0.5 * (du + dv);
  double dr = c->focus_dist * std::tan((c->defocus_angle * pi / 180.0f) / 2.0f);
  d3 ddu = dr * u, ddv = dr * v;
  const d3* src[9] = {&from, &p00, &du, &dv, &u, &v, &w, &ddu, &ddv};
  double* dst[9] = {f->center, f->pixel00_loc, f->pixel_delta_u, f->pixel_delta_v, f->u, f->v, f->w, f->defocus_disk_u, f->defocus_disk_v};
  for (int i = 0; i < 9; i++) dst[i][0] = src[i]->x, dst[i][1] = src[i]->y, dst[i][2] = src[i]->z;
  return RT_OK;
}

int rt_init(int device, rt_ctx** out) {
  if (!out) return RT_ERR_INVALID;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0 || device < 0 || device >= n) {
    std::lock_guard<std::mutex> g(g_err_mutex);
    g_init_error = e != cudaSuccess ? std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)
                                    : "no such CUDA device " + std::to_string(device) + " (" + std::to_string(n) + " visible); there is no CPU fallback";
    return RT_ERR_NO_DEVICE;
  }
  rt_ctx* ctx = new rt_ctx;
  ctx->device = device;
  std::memset(&ctx->sc, 0, sizeof ctx->sc);
  auto bail = [&](const char* what, cudaError_t err) {
    std::lock_guard<std::mutex> g(g_err_mutex);
    g_init_error = std::string(what) + ": " + cudaGetErrorString(err);
    if (ctx->counters) cudaFree(ctx->counters);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_cams) cudaEventDestroy(ctx->ev_cams);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return RT_ERR_CUDA;
  };
  const bool timing = std::getenv("RT_B200_TIMING") != nullptr;
  auto t_last = std::chrono::steady_clock::now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[rt_init] %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
    t_last = now;
  };
  lap("cudaGetDeviceCount (cuInit)");
  ctx->knobs.kernel = kDefaultStreamKernel ? KERNEL_STREAM : (kDefaultRefillKernel ? KERNEL_REFILL : KERNEL_MEGA);
  if (const char* k = std::getenv("RT_B200_KERNEL")) {
    const std::string v = k;
    ctx->knobs.kernel = v == "stream" ? KERNEL_STREAM : (v == "refill" ? KERNEL_REFILL : (v == "mega" ? KERNEL_MEGA : ctx->knobs.kernel));
  }
  if (const char* k = std::getenv("RT_B200_CHUNK_MAX")) ctx->knobs.chunk_max = std::max(1, std::atoi(k));
  if (const char* k = std::getenv("RT_B200_MAX_CHUNKS")) ctx->knobs.max_chunks = std::max(1, std::atoi(k));
  ctx->knobs.no_staging = std::getenv("RT_B200_NO_STAGING") != nullptr;
  ctx->knobs.no_smem_stack = std::getenv("RT_B200_NO_SMEM_STACK") != nullptr;
  if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
  lap("cudaSetDevice");
  // two attributes, not cudaGetDeviceProperties: the full property query costs tens of milliseconds (it reads clocks
  // and PCI state through the driver) and camera::render pays rt_init once per process
  int sm_count = 0, smem_optin = 0;
  if ((e = cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) return bail("cudaDeviceGetAttribute", e);
  if ((e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device)) != cudaSuccess) return bail("cudaDeviceGetAttribute", e);
  ctx->sm_count = sm_count;
  ctx->smem_optin = size_t(smem_optin);
  lap("cudaDeviceGetAttribute x2");
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  lap("cudaStreamCreate (context)");
  if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->ev_cams, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaMalloc(&ctx->counters, 32 * sizeof(unsigned long long))) != cudaSuccess) return bail("cudaMalloc", e);
  if ((e = cudaMemset(ctx->counters, 0, 32 * sizeof(unsigned long long))) != cudaSuccess) return bail("cudaMemset", e);
  lap("events + counters");
  {
    std::lock_guard<std::mutex> g(g_err_mutex);
    g_contexts.push_back(ctx);
  }
  *out = ctx;
  return RT_OK;
}

void rt_shutdown(rt_ctx* ctx) {
  if (!ctx) return;
  DebugScope dbg("rt_shutdown");
  {
    std::lock_guard<std::mutex> g(g_err_mutex);
    for (size_t i = 0; i < g_contexts.size(); i++)
      if (g_contexts[i] == ctx) g_contexts.erase(g_contexts.begin() + long(i)), i = g_contexts.size();
  }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  free_scene(ctx);
  cudaFree(ctx->arena);
  cudaFreeHost(ctx->staging);
  cudaFree(ctx->accum);
  cudaFree(ctx->reduce_buf);
  cudaFree(ctx->scratch);
  cudaFree(ctx->counters);
  cudaFree(ctx->cams_dev);
  cudaFreeHost(ctx->cams_host);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaEventDestroy(ctx->ev_cams);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* rt_last_error(rt_ctx* ctx) {
  if (ctx) return ctx->error.c_str();
  std::lock_guard<std::mutex> g(g_err_mutex);
  return g_init_error.c_str();
}

int rt_upload_scene(rt_ctx* ctx, const rt_scene_desc* scene) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_upload_scene");
  if (!scene) return fail(ctx, RT_ERR_INVALID, "null scene");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  free_scene(ctx);
  ctx->host = HostScene();
  if (!build_host_scene(scene, ctx->host)) {
    bool unsupported = ctx->host.error.find("unknown") != std::string::npos || ctx->host.error.find("not supported") != std::string::npos;
    return fail(ctx, unsupported ? RT_ERR_UNSUPPORTED : RT_ERR_INVALID, ctx->host.error);
  }
  const HostScene& h = ctx->host;
  if (h.bvh_depth > kStackDepth) return fail(ctx, RT_ERR_UNSUPPORTED, "BVH deeper than the traversal stack");
  if (h.leaf_refs.size() >= (size_t(1) << 27)) return fail(ctx, RT_ERR_UNSUPPORTED, "too many leaf references for the 32-bit leaf code");
  DeviceScene& s = ctx->sc;
  std::vector<ScenePiece> pieces;
#define UP(field, vec) pieces.push_back(ScenePiece{vec.data(), vec.size() * sizeof(vec[0]), &s.field, 0});
  UP(nodes, h.nodes)
  UP(leaf_refs, h.leaf_refs)
  UP(spheres, h.spheres)
  UP(sph_meta, h.sph_meta)
  UP(quads, h.quads)
  UP(quad_mat, h.quad_mat)
  UP(boxes, h.boxes)
  UP(box_meta, h.box_meta)
  UP(media, h.media)
  UP(medium_brefs, h.medium_brefs)
  UP(materials, h.materials)
  UP(textures, h.textures)
  UP(texels, h.texels)
  UP(images, h.images)
  UP(perlin_vec, h.perlin_vec)
  UP(perlin_perm, h.perlin_perm)
  UP(rotations, h.rotations)
  UP(xspheres, h.xspheres)
  UP(xquads, h.xquads)
  UP(xops, h.xops)
  UP(xchains, h.xchains)
#undef UP
  int rc = upload_pieces(ctx, pieces);
  if (rc != RT_OK) return rc;
  s.n_nodes = int(h.nodes.size() / 4);
  s.n_spheres = int(h.spheres.size() / 2);
  s.n_quads = int(h.quads.size() / 3);
  s.n_boxes = int(h.boxes.size() / 3);
  s.n_leaf_refs = int(h.leaf_refs.size());
  s.n_media = int(h.media.size());
  s.n_materials = int(h.materials.size() / 2);
  s.n_textures = int(h.textures.size() / 2);
  s.scene_abs_max = h.scene_abs_max;
  for (int a = 0; a < 3; a++) s.bounds_lo[a] = h.bounds_lo[a], s.bounds_hi[a] = h.bounds_hi[a];
  s.n_global_media = int(h.global_media.size());
  s.n_noise = int(h.perlin_vec.size() / 256);
  {  // how much of the scene is marble?  (decides the render kernel instantiation, plan_megakernel)
    auto may_noise = [&](int material) {
      if (material < 0 || size_t(2 * material + 1) >= h.materials.size()) return false;
      std::vector<int> todo{__builtin_bit_cast(int, h.materials[size_t(2 * material + 1)].y)};
      for (int guard = 0; guard < 64 && !todo.empty(); guard++) {
        const int tex = todo.back();
        todo.pop_back();
        if (tex < 0 || size_t(2 * tex + 1) >= h.textures.size()) continue;
        const float4 t1 = h.textures[size_t(2 * tex + 1)];
        const int kind = __builtin_bit_cast(int, t1.x);
        if (kind == TEX_NOISE) return true;
        if (kind == TEX_CHECKER) todo.push_back(__builtin_bit_cast(int, t1.y)), todo.push_back(__builtin_bit_cast(int, t1.z));
      }
      return false;
    };
    size_t prims = 0, marble = 0;
    for (size_t i = 0; i < h.sph_meta.size(); i++) prims++, marble += may_noise(h.sph_meta[i].x);
    for (size_t i = 0; i < h.quad_mat.size(); i++) prims++, marble += may_noise(h.quad_mat[i]);
    ctx->noise_share = s.n_noise > 0 && prims > 0 ? float(marble) / float(prims) : 0.0f;
  }
  for (int i = 0; i < 4; i++) s.global_media[i] = i < s.n_global_media ? h.global_media[size_t(i)] : -1;
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
#if RT_CHECKS
  // Self-test of the checks build (tools/sanitize.sh): RT_B200_CHECK_SELFTEST=1 plants ONE out-of-range reference — the first
  // sphere reference of the leaf list is pointed one past the end of the sphere array — which the device-side checks must
  // report (site CHK_SPHERE) at the next rt_synchronize.  The read it causes lands in the array staged next to the spheres:
  // garbage in the image, no fault.
  if (std::getenv("RT_B200_CHECK_SELFTEST") && s.n_spheres > 0) {
    for (size_t i = 0; i < h.leaf_refs.size(); i++)
      if (h.leaf_refs[i] != REF_NONE && (h.leaf_refs[i] >> 30) == REF_SPHERE) {
        const uint32_t bad = make_ref(REF_SPHERE, uint32_t(s.n_spheres));
        RT_CUDA(ctx, cudaMemcpy(const_cast<uint32_t*>(s.leaf_refs) + i, &bad, sizeof bad, cudaMemcpyHostToDevice));
        break;
      }
  }
#endif
  // top of the BVH in shared memory: as many breadth-first nodes as fit beside the static needs
  size_t budget = ctx->smem_optin > 8192 ? ctx->smem_optin - 4096 : 0;
  ctx->smem_nodes = int(std::min<size_t>(size_t(s.n_nodes), budget / 64));
  ctx->has_scene = true;
  return RT_OK;
}

// The megakernel's shared-memory plan for the uploaded scene: what is staged, where the per-thread records and the
// traversal stacks go.  Fills P.smem_nodes / P.state_off / P.stack_off.
struct MegaPlan {
  size_t smem;
  bool all_smem, sstack;
  bool coop_noise;  // the scene is largely noise-textured: the render kernel instantiation with cooperative turbulence
};
static MegaPlan plan_megakernel(const rt_ctx* ctx, RenderParams& P) {
  // the kernel is specialised for "the whole BVH — nodes, leaf references, spheres, boxes — is staged in shared
  // memory" (all BASELINE scenes): its node step then has neither the bounds test nor the global-memory path, and a
  // leaf visit makes no global load
  const size_t staged = size_t(ctx->sc.n_nodes) * 64 + size_t(ctx->sc.n_spheres) * 32 + size_t(ctx->sc.n_boxes) * 48 + size_t(ctx->sc.n_leaf_refs) * 4;
  constexpr size_t kStateBytes = size_t(32) * kRenderThreads;  // per-thread shade state (render_kernel)
  MegaPlan mp;
  mp.all_smem = staged + kStateBytes + 4096 <= ctx->smem_optin && !ctx->knobs.no_staging;
  size_t smem;
  if (mp.all_smem) {
    P.smem_nodes = ctx->sc.n_nodes, smem = staged;
  } else {  // the top of the BVH only, as much as fits beside the state records
    P.smem_nodes = int(std::min<size_t>(size_t(ctx->smem_nodes), (ctx->smem_optin - 4096 - kStateBytes) / 64));
    smem = size_t(P.smem_nodes) * 64;
  }
  P.state_off = unsigned((smem + 15) & ~size_t(15));
  smem = P.state_off + kStateBytes;
  // The traversal stacks go to shared memory too (one 32-bit entry per tree level and thread) when the child codes fit
  // their 16 bits and shared memory then still leaves L1 at least 64 KB for the spills and the global-memory scene
  // data: +2..3 % on bouncing_spheres / book1_final (40 KB staged), but -1.4..-7 % on book2_final, whose 127 KB staged
  // BVH + 50 KB of stacks would leave L1 23 KB (gpurun_out/ab_ss1.log).
  const size_t stack_bytes = size_t(std::max(1, ctx->host.bvh_depth)) * 4 * kRenderThreads;
  mp.sstack = mp.all_smem && RT_SMEM_STACK && !ctx->knobs.no_smem_stack && ctx->sc.n_nodes <= kSmemStackMaxCode && ((ctx->sc.n_leaf_refs << 3) | 7) <= kSmemStackMaxCode &&
              smem + stack_bytes <= kSmemStackBudget && smem + stack_bytes + 4096 <= ctx->smem_optin;
  if (mp.sstack) P.stack_off = unsigned(smem), P.stack_levels = unsigned(std::max(1, ctx->host.bvh_depth)), smem += stack_bytes;
  mp.smem = smem;
  // (a "lazy" form for scenes with a LITTLE marble — only lanes whose hit material is flagged build a hit record ahead of the
  //  shade — was measured on book2_final: bit-identical, -7 %; anything added to that scene's main loop costs more than the
  //  6 % its one marble sphere does: gpurun_out/ab_lazy.log)
  mp.coop_noise = RT_COOP_NOISE && ctx->noise_share >= 0.125f;
  return mp;
}

static cudaError_t launch_render(void (*kern)(RenderParams), int grid, size_t smem, cudaStream_t stream, RenderParams& P) {
  kern<<<grid, kRenderThreads, smem, stream>>>(P);
  return cudaGetLastError();
}

static void fill_camera(const rt_camera_desc* cam, const rt_camera_frame& f, CameraDev& c) {
  auto v3 = [](const double* p) { return make_float3(float(p[0]), float(p[1]), float(p[2])); };
  c.center = v3(f.center);
  // direction base relative to the centre, subtracted in double: |p00 - center| ~ focus_dist,
  // so fp32 keeps sub-pixel precision even when the camera sits at |x| ~ 1e3
  c.p00c = make_float3(float(f.pixel00_loc[0] - f.center[0]), float(f.pixel00_loc[1] - f.center[1]), float(f.pixel00_loc[2] - f.center[2]));
  c.du = v3(f.pixel_delta_u);
  c.dv = v3(f.pixel_delta_v);
  c.ddu = v3(f.defocus_disk_u);
  c.ddv = v3(f.defocus_disk_v);
  c.bg = v3(cam->background);
  c.W = f.image_width;
  c.H = f.image_height;
  c.max_depth = cam->max_depth;
  c.defocus = cam->defocus_angle > 0.0f ? 1 : 0;  // camera.hpp:155
}

// The streaming kernel's shared-memory plan for the uploaded scene; false when the scene does not fit it (the whole BVH
// must be staged, child codes must fit 16 bits) — the megakernel then renders.
static bool stream_layout(const rt_ctx* ctx, int bvh_depth, StreamLayout& L) {
  const DeviceScene& sc = ctx->sc;
  const int max_leaf_code = (sc.n_leaf_refs << 3) | 7;
  if (sc.n_nodes > kStreamMaxCode || max_leaf_code > kStreamMaxCode) return false;
  auto up16 = [](size_t v) { return (v + 15) & ~size_t(15); };
  size_t off = 0;
  L.node_plane = uint32_t(16u * size_t(sc.n_nodes));
  off = up16(3 * size_t(L.node_plane) + 8 * size_t(sc.n_nodes));
  L.off_sph = uint32_t(off), off = up16(off + 16 * size_t(sc.n_spheres));
  L.off_box = uint32_t(off), off = up16(off + 48 * size_t(sc.n_boxes));
  L.off_refs = uint32_t(off), off = up16(off + 4 * size_t(sc.n_leaf_refs));
  L.n_slots = RT_STREAM_SLOTS;
  L.slot_plane = 16u * L.n_slots;
  L.off_slots = uint32_t(off), off += 4 * size_t(L.slot_plane);
  const int levels = std::max(1, bvh_depth);  // a traversal never holds more postponed children than the tree has levels
  L.off_stack = uint32_t(off), off += size_t(levels) * kStackStride;
  uint32_t cap = 64;
  while (cap < 2 * L.n_slots) cap *= 2;  // ring capacity >= 2 x slots: a position is never reused while its last reader still holds it
  L.ring_mask = cap - 1;
  L.off_tq = uint32_t(off), off += 2 * size_t(cap);
  L.off_sq = uint32_t(off), off += 2 * size_t(cap);
  L.off_ctl = uint32_t(off), off += SC_BYTES;
  L.total = uint32_t(off);
  return off + sizeof(RenderParams) + 2048 <= ctx->smem_optin;
}

// The accumulator for `views` images of W x H (view-major); any change of shape reallocates it and clears it.
static int ensure_accum(rt_ctx* ctx, int W, int H, bool clear, int views = 1) {
  size_t values = size_t(W) * H * 3 * size_t(views);
  if (values != ctx->accum_values || ctx->acc_w != W || ctx->acc_views != views) {
    cudaFree(ctx->accum);
    ctx->accum = nullptr, ctx->accum_values = 0, ctx->acc_w = ctx->acc_h = ctx->acc_views = 0;  // a failed cudaMalloc below must not leave the old size behind
    RT_CUDA(ctx, cudaMalloc(&ctx->accum, values * 8));
    ctx->accum_values = values;
    ctx->acc_w = W, ctx->acc_h = H, ctx->acc_views = views;
    clear = true;
  }
  if (clear) {
    RT_CUDA(ctx, cudaMemsetAsync(ctx->accum, 0, values * 8, ctx->stream));
    RT_CUDA(ctx, cudaMemsetAsync(ctx->counters, 0, 32 * sizeof(unsigned long long), ctx->stream));
    ctx->rays_total = ctx->samples_total = 0;
  }
  return RT_OK;
}

static int render_range(rt_ctx* ctx, const rt_camera_desc* cam, const rt_render_opts* opts, bool first_piece, bool last_piece);

// One kernel launch addresses < 2^32 work items (pixel tile x chunk of 32 samples).  A request beyond that — e.g.
// 4096 x 4096 at 10,000 spp — is rendered as several stream-ordered launches over consecutive sample ranges; the
// fixed-point sums make the split invisible in the image.
int rt_render(rt_ctx* ctx, const rt_camera_desc* cam, const rt_render_opts* opts) {
  if (!ctx) return RT_ERR_INVALID;
  if (!cam || !opts) return fail(ctx, RT_ERR_INVALID, "null camera / options");
  if (cam->image_width <= 0 || cam->samples_per_pixel <= 0 || !(cam->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera");
  rt_camera_frame f;
  rt_camera_initialize(cam, &f);
  const long long count = opts->sample_count > 0 ? opts->sample_count : (long long)cam->samples_per_pixel - opts->sample_begin;
  const unsigned long long per_chunk = (unsigned long long)((f.image_width + 7) / 8) * (unsigned long long)((f.image_height + 3) / 4) * 32ull;
  unsigned long long max_chunks = (0xFFFFFFFFull - (unsigned long long)ctx->sm_count * kRenderThreads - 1ull) / per_chunk;
  if (ctx->knobs.max_chunks > 0) max_chunks = std::min<unsigned long long>(max_chunks, (unsigned long long)ctx->knobs.max_chunks);  // test hook
  if (max_chunks == 0) return fail(ctx, RT_ERR_INVALID, "image too large (more than 2^32 pixels per launch)");
  const long long cap = (long long)std::min<unsigned long long>(max_chunks * 32ull, 1ull << 30);
  if (count <= cap) return render_range(ctx, cam, opts, true, true);
  rt_render_opts piece = *opts;
  for (long long done = 0; done < count; done += cap) {
    piece.sample_begin = int32_t(opts->sample_begin + done);
    piece.sample_count = int32_t(std::min(cap, count - done));
    piece.clear = done == 0 ? opts->clear : 0;
    const bool last = done + cap >= count;
    piece.push_accum = last ? opts->push_accum : nullptr;
    int rc = render_range(ctx, cam, &piece, done == 0, last);
    if (rc != RT_OK) return rc;
  }
  return RT_OK;
}

static int render_range(rt_ctx* ctx, const rt_camera_desc* cam, const rt_render_opts* opts, bool first_piece, bool last_piece) {
  DebugScope dbg("rt_render");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_render before rt_upload_scene");
  if (cam->image_width <= 0 || cam->samples_per_pixel <= 0 || !(cam->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  rt_camera_frame f;
  rt_camera_initialize(cam, &f);
  int rc = ensure_accum(ctx, f.image_width, f.image_height, opts->clear != 0);
  if (rc != RT_OK) return rc;

  RenderParams P;
  std::memset(&P, 0, sizeof P);
  P.sc = ctx->sc;
  fill_camera(cam, f, P.cam);
  P.key = make_uint2((unsigned)opts->seed, (unsigned)(opts->seed >> 32));
  P.sample_begin = opts->sample_begin;
  P.sample_count = opts->sample_count > 0 ? opts->sample_count : cam->samples_per_pixel - opts->sample_begin;
  if (P.sample_begin < 0 || P.sample_count <= 0) return fail(ctx, RT_ERR_INVALID, "empty sample range");
  P.tiles_x = (f.image_width + 7) / 8;
  P.tiles_y = (f.image_height + 3) / 4;
  const int grid = ctx->sm_count;
  const long long threads = (long long)grid * kRenderThreads;
  // samples per work item: enough items (>= 8 per thread) for the dynamic balance, at most 32
  long long total = (long long)f.image_width * f.image_height * P.sample_count;
  long long chunk = total / (threads * 8);
  long long chunk_max = 32;
  if (ctx->knobs.chunk_max > 0) chunk_max = ctx->knobs.chunk_max;  // A/B knob (tools/ab_env.py)
  P.chunk = int(std::max<long long>(1, std::min<long long>({chunk, chunk_max, (long long)P.sample_count})));
  while (P.chunk & (P.chunk - 1)) P.chunk &= P.chunk - 1;  // largest power of two below: the megakernel finds the end of an item with a mask
  P.n_chunks = (P.sample_count + P.chunk - 1) / P.chunk;
  const unsigned long long n_items = (unsigned long long)P.tiles_x * P.tiles_y * 32ull * (unsigned long long)P.n_chunks;
  if (n_items >= 0xFFFFFFFFull - (unsigned long long)threads) return fail(ctx, RT_ERR_INVALID, "image x samples too large for one launch: shard the samples");
  P.per_chunk = unsigned(P.tiles_x) * unsigned(P.tiles_y) * 32u;
  P.n_items = unsigned(n_items);
  P.accum = opts->peer_accum ? static_cast<unsigned long long*>(opts->peer_accum) : ctx->accum;
  P.push = static_cast<unsigned long long*>(opts->push_accum);
  P.n_values = (unsigned long long)f.image_width * f.image_height * 3ull;
  if (P.push && opts->peer_accum) return fail(ctx, RT_ERR_INVALID, "peer_accum and push_accum are mutually exclusive");
  if (opts->peer_accum && opts->peer_accum != ctx->accum) {
    // The render kernel's per-sample adds are DEVICE-scope atomics (system scope in the hot loop costs every render):
    // they are only atomic among kernels of one GPU, and nothing in the call says how large the target is.  So the target
    // must be the accumulator of a live context of this process, on this context's device, of this camera's size;
    // across GPUs the exchange step is push_accum (system-scope red.add behind the render).
    const rt_ctx* owner = nullptr;
    {
      std::lock_guard<std::mutex> g(g_err_mutex);
      for (const rt_ctx* c : g_contexts)
        if (c->accum && c->accum == opts->peer_accum) owner = c;
    }
    if (!owner) return fail(ctx, RT_ERR_INVALID, "peer_accum is not the accumulator (rt_accum_device_ptr) of a live context of this process");
    if (owner->device != ctx->device)
      return fail(ctx, RT_ERR_UNSUPPORTED, "peer_accum lives on another GPU: the render kernel's adds are device-scope atomics; use push_accum across GPUs");
    if (owner->accum_values != size_t(P.n_values)) return fail(ctx, RT_ERR_INVALID, "peer_accum belongs to an image of another size");
  }

  P.counters = ctx->counters;
  P.smem_nodes = ctx->smem_nodes;
  size_t smem = size_t(P.smem_nodes) * 64;
  const bool count = (opts->flags & RT_RENDER_COUNTERS) != 0;
  // kernel choice: the megakernel unless another scheduling variant is asked for (rt_render_opts.flags; the library-wide
  // default can be moved with RT_B200_KERNEL, read once at rt_init) — all of them produce the same accumulator bits
  if (opts->flags & RT_RENDER_POOL_REMOVED)
    return fail(ctx, RT_ERR_UNSUPPORTED, "the per-warp path-pool kernel was removed (0.55-0.65x the megakernel); its queue-fed successor is RT_RENDER_STREAM");
  int kernel = ctx->knobs.kernel;
  if (opts->flags & RT_RENDER_MEGAKERNEL) kernel = KERNEL_MEGA;
  if (opts->flags & RT_RENDER_STREAM) kernel = KERNEL_STREAM;
  if (opts->flags & RT_RENDER_REFILL) kernel = KERNEL_REFILL;
  bool stream = kernel == KERNEL_STREAM;
  const bool refill = kernel == KERNEL_REFILL;
  StreamLayout SL;
  std::memset(&SL, 0, sizeof SL);
  if (stream && !stream_layout(ctx, ctx->host.bvh_depth, SL)) {
    if (opts->flags & RT_RENDER_STREAM) return fail(ctx, RT_ERR_UNSUPPORTED, "the scene does not fit the streaming kernel's shared-memory plan");
    stream = false;
  }
  if (first_piece) RT_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  if (P.cam.max_depth <= 0) {
    // ray_color returns black at once (camera.hpp:183-186): nothing to trace, the sums stay as they are
  } else if (stream) {
    P.sl = SL;
    P.smem_nodes = ctx->sc.n_nodes;
    smem = SL.total;
    void (*kern)(RenderParams) = count ? stream_kernel<true> : stream_kernel<false>;
    RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    const unsigned long long first = 0ull;
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->counters, &first, sizeof first, cudaMemcpyHostToDevice, ctx->stream));
    kern<<<grid, kStreamThreads, smem, ctx->stream>>>(P);
    RT_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
  } else if (refill) {
    const size_t staged = size_t(ctx->sc.n_nodes) * 64 + size_t(ctx->sc.n_spheres) * 32 + size_t(ctx->sc.n_boxes) * 48 + size_t(ctx->sc.n_leaf_refs) * 4;
    const bool all_smem = staged + kRefillStateBytes + 4096 <= ctx->smem_optin && !ctx->knobs.no_staging;
    if (all_smem) {
      P.smem_nodes = ctx->sc.n_nodes, smem = staged;
    } else {
      P.smem_nodes = int(std::min<size_t>(size_t(P.smem_nodes), (ctx->smem_optin - 4096 - kRefillStateBytes) / 64));
      smem = size_t(P.smem_nodes) * 64;
    }
    P.state_off = unsigned((smem + 15) & ~size_t(15));
    smem = P.state_off + kRefillStateBytes;
    void (*kern)(RenderParams) = count ? (all_smem ? refill_kernel<true, true> : refill_kernel<true, false>)
                                       : (all_smem ? refill_kernel<false, true> : refill_kernel<false, false>);
    RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    unsigned long long first = 0ull;
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->counters, &first, sizeof first, cudaMemcpyHostToDevice, ctx->stream));
    kern<<<grid, kRefillThreads, smem, ctx->stream>>>(P);
    RT_CUDA(ctx, cudaGetLastError());
    ctx->launches++;
  } else {
    // the kernel is specialised for "the whole BVH — nodes, leaf references, spheres, boxes — is staged in shared
    // memory" (all BASELINE scenes): its node step then has neither the bounds test nor the global-memory path, and a
    // leaf visit makes no global load
    const MegaPlan mp = plan_megakernel(ctx, P);
    smem = mp.smem;
    void (*kern)(RenderParams) = mp.sstack ? (count ? render_kernel<true, true, true> : render_kernel<false, true, true>)
                                           : count ? (mp.all_smem ? render_kernel<true, true> : render_kernel<true, false>)
                                                   : (mp.all_smem ? render_kernel<false, true> : render_kernel<false, false>);
    if (mp.coop_noise && !count)  // scenes made of marble (perlin_sphere, simple_light): +8..13 %, gpurun_out/ab_coop.log
      kern = mp.sstack ? render_kernel<false, true, true, false, true> : (mp.all_smem ? render_kernel<false, true, false, false, true> : render_kernel<false, false, false, false, true>);
    RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    // counters[0] = next work item: lanes take items with atomicAdd when they need one
    unsigned long long first = 0ull;
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->counters, &first, sizeof first, cudaMemcpyHostToDevice, ctx->stream));
    RT_CUDA(ctx, launch_render(kern, grid, smem, ctx->stream, P));
    ctx->launches++;
  }
  ctx->samples_total += (unsigned long long)f.image_width * f.image_height * P.sample_count;
  RT_CUDA(ctx, cudaGetLastError());
  if (P.push) {  // the exchange step, stream-ordered behind the render (inside the timed region)
    push_kernel<<<2 * grid, 512, 0, ctx->stream>>>(ctx->accum, P.push, P.n_values);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
  }
  if (last_piece) {
    RT_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->timed = true;
  }
  return RT_OK;
}

// One launch of render_kernel<.., VIEWS> over the sample range of `opts` for all views; the camera table is filled by the
// first piece of a request.  The views were checked by rt_render_views: same W x H (f) and spp.
static int views_range(rt_ctx* ctx, int32_t n_views, const rt_camera_desc* cams, const rt_camera_frame& f, const rt_render_opts* opts, bool first_piece,
                       bool last_piece) {
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  const int W = f.image_width, H = f.image_height;
  int rc = ensure_accum(ctx, W, H, opts->clear != 0, n_views);
  if (rc != RT_OK) return rc;
  if (first_piece) RT_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  if (first_piece) {
    if (n_views > ctx->cams_cap) {
      RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // a launch in flight may still read the old table
      cudaFree(ctx->cams_dev);
      cudaFreeHost(ctx->cams_host);
      ctx->cams_dev = nullptr, ctx->cams_host = nullptr, ctx->cams_cap = 0;
      RT_CUDA(ctx, cudaMalloc(&ctx->cams_dev, size_t(n_views) * sizeof(CameraDev)));
      RT_CUDA(ctx, cudaHostAlloc(&ctx->cams_host, size_t(n_views) * sizeof(CameraDev), cudaHostAllocDefault));
      ctx->cams_cap = n_views;
    } else {
      RT_CUDA(ctx, cudaEventSynchronize(ctx->ev_cams));  // the previous batch's copy has read the pinned buffer
    }
    for (int v = 0; v < n_views; v++) {
      rt_camera_frame fv;
      rt_camera_initialize(cams + v, &fv);
      fill_camera(cams + v, fv, ctx->cams_host[v]);
    }
    RT_CUDA(ctx, cudaMemcpyAsync(ctx->cams_dev, ctx->cams_host, size_t(n_views) * sizeof(CameraDev), cudaMemcpyHostToDevice, ctx->stream));
    RT_CUDA(ctx, cudaEventRecord(ctx->ev_cams, ctx->stream));
  }

  RenderParams P;
  std::memset(&P, 0, sizeof P);
  P.sc = ctx->sc;
  fill_camera(cams, f, P.cam);  // the size every view shares; the kernel reads each view's camera from P.cams
  P.key = make_uint2((unsigned)opts->seed, (unsigned)(opts->seed >> 32));
  P.sample_begin = opts->sample_begin;
  P.sample_count = opts->sample_count;
  P.tiles_x = (W + 7) / 8;
  P.tiles_y = (H + 3) / 4;
  const int grid = ctx->sm_count;
  const long long threads = (long long)grid * kRenderThreads;
  // samples per work item as rt_render chooses them, over the whole batch (the sums do not depend on the choice)
  const long long total = (long long)n_views * W * H * P.sample_count;
  long long chunk = total / (threads * 8);
  const long long chunk_max = ctx->knobs.chunk_max > 0 ? ctx->knobs.chunk_max : 32;
  P.chunk = int(std::max<long long>(1, std::min<long long>({chunk, chunk_max, (long long)P.sample_count})));
  while (P.chunk & (P.chunk - 1)) P.chunk &= P.chunk - 1;
  P.n_chunks = (P.sample_count + P.chunk - 1) / P.chunk;
  P.view_items = unsigned(P.tiles_x) * unsigned(P.tiles_y) * 32u;
  const unsigned long long per_chunk = (unsigned long long)P.view_items * (unsigned long long)n_views;
  const unsigned long long n_items = per_chunk * (unsigned long long)P.n_chunks;
  if (n_items >= 0xFFFFFFFFull - (unsigned long long)threads) return fail(ctx, RT_ERR_INVALID, "views x image x samples too large for one launch: shard the samples");
  P.per_chunk = unsigned(per_chunk);
  P.n_items = unsigned(n_items);
  P.accum = ctx->accum;
  P.n_values = (unsigned long long)n_views * W * H * 3ull;
  P.counters = ctx->counters;
  P.cams = ctx->cams_dev;
  P.n_views = n_views;
  P.view_pixels = unsigned(W) * unsigned(H);
  // the plan rt_render picks for this scene: the views of a batch take the same staging, stack and turbulence form
  const MegaPlan mp = plan_megakernel(ctx, P);
  void (*kern)(RenderParams) = mp.coop_noise ? (mp.sstack ? render_kernel<false, true, true, false, true, true>
                                                          : (mp.all_smem ? render_kernel<false, true, false, false, true, true> : render_kernel<false, false, false, false, true, true>))
                                             : (mp.sstack ? render_kernel<false, true, true, false, false, true>
                                                          : (mp.all_smem ? render_kernel<false, true, false, false, false, true> : render_kernel<false, false, false, false, false, true>));
  RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(mp.smem)));
  RT_CUDA(ctx, cudaMemsetAsync(ctx->counters, 0, sizeof(unsigned long long), ctx->stream));  // counters[0] = next work item
  RT_CUDA(ctx, launch_render(kern, grid, mp.smem, ctx->stream, P));
  ctx->launches++;
  // every view's samples count, also those of a view with max_depth <= 0 (as rt_render counts them)
  ctx->samples_total += (unsigned long long)n_views * W * H * P.sample_count;
  if (last_piece) {
    RT_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->timed = true;
  }
  return RT_OK;
}

int rt_render_views(rt_ctx* ctx, int32_t n_views, const rt_camera_desc* cams, const rt_render_opts* opts) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_render_views");
  if (n_views < 1 || !cams || !opts) return fail(ctx, RT_ERR_INVALID, "rt_render_views: n_views < 1, or null cameras / options");
  rt_camera_frame f;
  for (int32_t v = 0; v < n_views; v++) {
    const rt_camera_desc* c = cams + v;
    if (c->image_width <= 0 || c->samples_per_pixel <= 0 || !(c->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera (view " + std::to_string(v) + ")");
    rt_camera_frame fv;
    rt_camera_initialize(c, &fv);
    if (v == 0) {
      f = fv;
    } else if (fv.image_width != f.image_width || fv.image_height != f.image_height || c->samples_per_pixel != cams[0].samples_per_pixel) {
      return fail(ctx, RT_ERR_INVALID, "view " + std::to_string(v) + " differs from view 0 in image size or samples_per_pixel: the views of a batch share both");
    }
  }
  if ((long long)n_views * f.image_width * f.image_height > 0x7FFFFFFFll)
    return fail(ctx, RT_ERR_INVALID, "n_views x image_width x image_height exceeds 2^31 - 1 (the global pixel index is 32-bit)");
  if (opts->peer_accum || opts->push_accum) return fail(ctx, RT_ERR_UNSUPPORTED, "rt_render_views has no peer_accum / push_accum: shard a batch by views");
  if (opts->flags & (RT_RENDER_COUNTERS | RT_RENDER_STREAM | RT_RENDER_REFILL | RT_RENDER_POOL_REMOVED))
    return fail(ctx, RT_ERR_UNSUPPORTED, "rt_render_views renders with the megakernel only (no RT_RENDER_COUNTERS / STREAM / REFILL)");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_render_views before rt_upload_scene");
  const long long count = opts->sample_count > 0 ? opts->sample_count : (long long)cams[0].samples_per_pixel - opts->sample_begin;
  if (opts->sample_begin < 0 || count <= 0) return fail(ctx, RT_ERR_INVALID, "empty sample range");
  // more than 2^32 work items: consecutive sample ranges in stream-ordered launches, as rt_render splits
  const unsigned long long per_chunk = (unsigned long long)n_views * (unsigned long long)((f.image_width + 7) / 8) * (unsigned long long)((f.image_height + 3) / 4) * 32ull;
  unsigned long long max_chunks = (0xFFFFFFFFull - (unsigned long long)ctx->sm_count * kRenderThreads - 1ull) / per_chunk;
  if (ctx->knobs.max_chunks > 0) max_chunks = std::min<unsigned long long>(max_chunks, (unsigned long long)ctx->knobs.max_chunks);  // test hook
  if (max_chunks == 0) return fail(ctx, RT_ERR_INVALID, "batch too large (more than 2^32 work items per sample)");
  const long long cap = (long long)std::min<unsigned long long>(max_chunks * 32ull, 1ull << 30);
  rt_render_opts piece = *opts;
  for (long long done = 0; done < count; done += cap) {
    piece.sample_begin = int32_t(opts->sample_begin + done);
    piece.sample_count = int32_t(std::min(cap, count - done));
    piece.clear = done == 0 ? opts->clear : 0;
    int rc = views_range(ctx, n_views, cams, f, &piece, done == 0, done + cap >= count);
    if (rc != RT_OK) return rc;
  }
  return RT_OK;
}

int rt_synchronize(rt_ctx* ctx) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_synchronize");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
#if RT_CHECKS
  {  // checks build: a failed device-side bounds check turns into an error here
    unsigned int bad = 0, zero = 0, count = 0;
    RT_CUDA(ctx, cudaMemcpyFromSymbol(&bad, g_rt_check_fail, sizeof bad));
    RT_CUDA(ctx, cudaMemcpyFromSymbol(&count, g_rt_check_count, sizeof count));
    if (std::getenv("RT_B200_DEBUG")) std::fprintf(stderr, "[rt_b200 checks] %u device-side checks evaluated (mod 2^32), worst failing site %u\n", count, bad);
    if (bad) {
      RT_CUDA(ctx, cudaMemcpyToSymbol(g_rt_check_fail, &zero, sizeof zero));
      return fail(ctx, RT_ERR_CUDA, "device-side bounds check failed at site " + std::to_string(bad) + " (rt_device.cuh, CHK_*)");
    }
  }
#endif
  return RT_OK;
}

int rt_accum_device_ptr(rt_ctx* ctx, void** dev_ptr, size_t* bytes) {
  if (!ctx || !dev_ptr || !bytes) return RT_ERR_INVALID;
  if (!ctx->accum) return fail(ctx, RT_ERR_INVALID, "no accumulator yet (call rt_render first)");
  *dev_ptr = ctx->accum;
  *bytes = ctx->accum_values * 8;
  return RT_OK;
}

// ---- fused multi-GPU reduce: a reduce buffer other ranks' render kernels add their accumulators into ----------
int rt_reduce_buffer(rt_ctx* ctx, const rt_camera_desc* cam, void** dev_ptr, rt_ipc_handle* handle) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_reduce_buffer");
  if (!cam || !dev_ptr || cam->image_width <= 0 || !(cam->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera / null output");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  rt_camera_frame f;
  rt_camera_initialize(cam, &f);
  const size_t values = size_t(f.image_width) * f.image_height * 3;
  if (values != ctx->reduce_values) {
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaFree(ctx->reduce_buf);
    ctx->reduce_buf = nullptr, ctx->reduce_values = 0;
    RT_CUDA(ctx, cudaMalloc(&ctx->reduce_buf, values * 8));
    ctx->reduce_values = values;
  }
  RT_CUDA(ctx, cudaMemsetAsync(ctx->reduce_buf, 0, values * 8, ctx->stream));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // zeroed before any peer may add into it
  *dev_ptr = ctx->reduce_buf;
  if (handle) {
    static_assert(sizeof(cudaIpcMemHandle_t) == sizeof(rt_ipc_handle), "rt_ipc_handle must hold a cudaIpcMemHandle_t");
    cudaIpcMemHandle_t h;
    RT_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->reduce_buf));
    std::memcpy(handle->bytes, &h, sizeof h);
  }
  return RT_OK;
}

int rt_peer_open(rt_ctx* ctx, const rt_ipc_handle* handle, void** dev_ptr) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_peer_open");
  if (!handle || !dev_ptr) return fail(ctx, RT_ERR_INVALID, "null handle / output");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle->bytes, sizeof h);
  RT_CUDA(ctx, cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return RT_OK;
}

int rt_peer_enable(rt_ctx* ctx, rt_ctx* owner) {
  if (!ctx || !owner) return RT_ERR_INVALID;
  DebugScope dbg("rt_peer_enable");
  if (ctx->device == owner->device) return RT_OK;
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  int can = 0;
  RT_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, owner->device));
  if (!can) return fail(ctx, RT_ERR_UNSUPPORTED, "no peer access between devices " + std::to_string(ctx->device) + " and " + std::to_string(owner->device));
  cudaError_t e = cudaDeviceEnablePeerAccess(owner->device, 0);
  if (e == cudaErrorPeerAccessAlreadyEnabled) {
    cudaGetLastError();
    e = cudaSuccess;
  }
  RT_CUDA(ctx, e);
  return RT_OK;
}

int rt_peer_close(rt_ctx* ctx, void* dev_ptr) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_peer_close");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  RT_CUDA(ctx, cudaIpcCloseMemHandle(dev_ptr));
  return RT_OK;
}

int rt_adopt_reduce_buffer(rt_ctx* ctx) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_adopt_reduce_buffer");
  if (!ctx->reduce_buf) return fail(ctx, RT_ERR_INVALID, "no reduce buffer (call rt_reduce_buffer first)");
  if (ctx->reduce_values != ctx->accum_values || !ctx->accum) return fail(ctx, RT_ERR_INVALID, "reduce buffer and accumulator differ in size");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  // a copy, not a pointer swap: the reduce buffer (and its IPC handle, which peers keep open) stays where it is
  RT_CUDA(ctx, cudaMemcpyAsync(ctx->accum, ctx->reduce_buf, ctx->accum_values * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return RT_OK;
}

int rt_upload_accum(rt_ctx* ctx, const rt_camera_desc* cam, const void* src, size_t bytes) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_upload_accum");
  if (!cam || !src || cam->image_width <= 0 || !(cam->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera / null source");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  rt_camera_frame f;
  rt_camera_initialize(cam, &f);
  const size_t values = size_t(f.image_width) * f.image_height * 3;
  if (bytes != values * 8) return fail(ctx, RT_ERR_INVALID, "source is not image_width x image_height x 3 int64 sums");
  int rc = ensure_accum(ctx, f.image_width, f.image_height, true);  // also resets the ray / sample counters
  if (rc != RT_OK) return rc;
  RT_CUDA(ctx, cudaMemcpyAsync(ctx->accum, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // src may be pageable and may be freed by the caller right away
  return RT_OK;
}

int rt_download(rt_ctx* ctx, rt_buffer_kind kind, int32_t spp, void* dst, size_t bytes) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_download");
  if (!dst) return fail(ctx, RT_ERR_INVALID, "null destination");
  if (!ctx->accum) return fail(ctx, RT_ERR_INVALID, "nothing rendered yet");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  const size_t n = ctx->accum_values;
  if (kind == RT_BUF_ACCUM_I64) {
    if (bytes < n * 8) return fail(ctx, RT_ERR_INVALID, "destination too small");
    RT_CUDA(ctx, cudaMemcpyAsync(dst, ctx->accum, n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RT_OK;
  }
  if (spp <= 0) return fail(ctx, RT_ERR_INVALID, "samples_per_pixel must be positive");
  const bool f32 = kind == RT_BUF_RADIANCE_F32;
  if (!f32 && kind != RT_BUF_RGB8) return fail(ctx, RT_ERR_INVALID, "unknown buffer kind");
  const size_t need = f32 ? n * 4 : n;
  if (bytes < need) return fail(ctx, RT_ERR_INVALID, "destination too small");
  // persistent scratch: with peer access enabled (NCCL, CUDA IPC) every cudaMalloc / cudaFree also updates the peers'
  // mappings and costs tens of milliseconds
  if (need > ctx->scratch_bytes) {
    cudaFree(ctx->scratch);
    ctx->scratch = nullptr, ctx->scratch_bytes = 0;
    RT_CUDA(ctx, cudaMalloc(&ctx->scratch, need));
    ctx->scratch_bytes = need;
  }
  void* tmp = ctx->scratch;
  const double scale = double(1.0f / float(spp));  // pixel_samples_scale, camera.hpp:83
  finalize_kernel<<<unsigned((n + 255) / 256), 256, 0, ctx->stream>>>(reinterpret_cast<const long long*>(ctx->accum), (long long)n, scale,
                                                                      f32 ? static_cast<float*>(tmp) : nullptr,
                                                                      f32 ? nullptr : static_cast<unsigned char*>(tmp));
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(dst, tmp, need, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e != cudaSuccess) return fail(ctx, RT_ERR_CUDA, std::string("rt_download: ") + cudaGetErrorString(e));
  return RT_OK;
}

int rt_get_stats(rt_ctx* ctx, rt_stats* out) {
  if (!ctx || !out) return RT_ERR_INVALID;
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  std::memset(out, 0, sizeof *out);
  unsigned long long c[32];
  RT_CUDA(ctx, cudaMemcpy(c, ctx->counters, sizeof c, cudaMemcpyDeviceToHost));
  out->rays = c[1];
  if (c[19] && std::getenv("RT_B200_DEBUG")) {  // the streaming kernel's watchdog records (debug builds)
    std::fprintf(stderr, "[rt_b200] stream watchdog: %llu reports\n", c[19]);
    for (int k = 0; k < 3 && k < int(c[19]); k++) {
      const unsigned long long* o = c + 20 + 4 * k;
      std::fprintf(stderr, "  where %llu thread %llu cta %llu a %d b %d | tq_avail %d sq_avail %d | tq head %llu tail %llu sq head %llu tail %llu | dead %d\n", o[0] & 0xFF,
                   (o[0] >> 8) & 0xFFFF, (o[0] >> 24) & 0xFFFF, int(o[0] >> 40), int(o[3] >> 32), int(unsigned(o[1])), int(unsigned(o[1] >> 32)), o[2] & 0xFFFF,
                   (o[2] >> 16) & 0xFFFF, (o[2] >> 32) & 0xFFFF, (o[2] >> 48) & 0xFFFF, int(unsigned(o[3])));
    }
  }
  out->samples = ctx->samples_total;  // every sample of the requested range is rendered: W*H*count per launch
  for (int i = 0; i < CN_COUNT; i++) out->census[i] = c[4 + i];
  if (ctx->timed) {
    float ms = 0;
    RT_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    out->last_render_ms = ms;
  }
  out->image_width = ctx->acc_w;
  out->image_height = ctx->acc_h;
  out->n_views = ctx->acc_views;
  out->n_nodes = ctx->sc.n_nodes;
  out->n_spheres = ctx->sc.n_spheres;
  out->n_quads = ctx->sc.n_quads;
  out->n_boxes = ctx->sc.n_boxes;
  out->n_media = ctx->sc.n_media;
  out->bvh_nodes_in_smem = ctx->smem_nodes;
  out->kernel_launches = ctx->launches;
  return RT_OK;
}

int rt_trace_rays(rt_ctx* ctx, int64_t n, const double* origin, const double* direction, const double* time, double tmin, double tmax, int32_t flags,
                  int32_t* prim_id, double* t, double* normal, uint8_t* front_face) {
  return rt_trace_rays_from(ctx, n, origin, direction, time, nullptr, tmin, tmax, flags, prim_id, t, normal, front_face);
}

int rt_trace_rays_from(rt_ctx* ctx, int64_t n, const double* origin, const double* direction, const double* time, const int32_t* start_prim, double tmin,
                       double tmax, int32_t flags, int32_t* prim_id, double* t, double* normal, uint8_t* front_face) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_trace_rays");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_trace_rays before rt_upload_scene");
  if (n < 0 || (n > 0 && (!origin || !direction))) return fail(ctx, RT_ERR_INVALID, "bad ray arrays");
  if (start_prim && (flags & RT_TRACE_EXACT))
    return fail(ctx, RT_ERR_INVALID, "RT_TRACE_EXACT follows the reference, which has no start primitive: start_prim is for the fp32 traversal");
  std::vector<uint32_t> skip;
  if (start_prim) {
    int rc = start_refs(ctx, n, start_prim, skip);
    if (rc != RT_OK) return rc;
  }
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  Scratch sx;
  const double* d_o = sx.to_device(origin, size_t(3 * n));
  const double* d_d = sx.to_device(direction, size_t(3 * n));
  const double* d_t = sx.to_device(time, size_t(n));
  const uint32_t* d_s = start_prim ? sx.to_device(skip.data(), size_t(n)) : nullptr;
  if (n > 0 && (!d_o || !d_d || (time && !d_t) || (start_prim && !d_s))) return fail(ctx, RT_ERR_CUDA, "cudaMalloc / copy of the rays failed");
  return run_trace(ctx, n, d_o, d_d, d_t, d_s, tmin, tmax, flags, prim_id, t, normal, front_face, sx);
}

// The pixel-centre rays through render_kernel itself (its AOV instantiation), planned exactly as rt_render plans it for
// this scene: same staging, same node form, same stack.  `bounce`: also the second segment (P.aov_b).  Host outputs:
// prim_id, t (n), normal (3n), rec (kAovBounce n); prim_id and rec may be NULL.
static int render_aov(rt_ctx* ctx, const rt_camera_desc* cam, const rt_camera_frame& f, uint64_t seed, bool bounce, int32_t* prim_id, float* t, float* normal,
                      float* rec) {
  const long long n = (long long)f.image_width * f.image_height;
  Scratch sx;
  RenderParams P;
  std::memset(&P, 0, sizeof P);
  P.sc = ctx->sc;
  fill_camera(cam, f, P.cam);
  P.cam.max_depth = bounce ? 2 : 1;
  P.key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
  P.sample_begin = 0, P.sample_count = 1, P.chunk = 1, P.n_chunks = 1;
  P.tiles_x = (f.image_width + 7) / 8, P.tiles_y = (f.image_height + 3) / 4;
  const unsigned long long n_items = (unsigned long long)P.tiles_x * P.tiles_y * 32ull;
  if (n_items >= 0xFFFFFFFFull - (unsigned long long)ctx->sm_count * kRenderThreads) return fail(ctx, RT_ERR_INVALID, "image too large");
  P.per_chunk = unsigned(n_items), P.n_items = unsigned(n_items);
  P.counters = sx.alloc<unsigned long long>(32);
  P.aov_id = sx.alloc<int>(size_t(n));
  P.aov_t = sx.alloc<float>(size_t(n));
  P.aov_n = sx.alloc<float>(size_t(3 * n));
  P.aov_b = bounce ? sx.alloc<float>(size_t(kAovBounce * n)) : nullptr;
  if (!P.counters || !P.aov_id || !P.aov_t || !P.aov_n || (bounce && !P.aov_b)) return fail(ctx, RT_ERR_CUDA, "cudaMalloc failed");
  RT_CUDA(ctx, cudaMemsetAsync(P.counters, 0, 32 * sizeof(unsigned long long), ctx->stream));
  const MegaPlan mp = plan_megakernel(ctx, P);
  void (*kern)(RenderParams) = mp.sstack ? render_kernel<false, true, true, true> : (mp.all_smem ? render_kernel<false, true, false, true> : render_kernel<false, false, false, true>);
  RT_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(mp.smem)));
  RT_CUDA(ctx, launch_render(kern, ctx->sm_count, mp.smem, ctx->stream, P));
  ctx->launches++;
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (prim_id) RT_CUDA(ctx, cudaMemcpy(prim_id, P.aov_id, size_t(n) * 4, cudaMemcpyDeviceToHost));
  RT_CUDA(ctx, cudaMemcpy(t, P.aov_t, size_t(n) * 4, cudaMemcpyDeviceToHost));
  RT_CUDA(ctx, cudaMemcpy(normal, P.aov_n, size_t(3 * n) * 4, cudaMemcpyDeviceToHost));
  if (rec) RT_CUDA(ctx, cudaMemcpy(rec, P.aov_b, size_t(kAovBounce * n) * 4, cudaMemcpyDeviceToHost));
  return RT_OK;
}

int rt_bounce_visibility(rt_ctx* ctx, const rt_camera_desc* cam, uint64_t seed, int32_t* prim_id, double* t, float* origin1, float* dir1, int32_t* bounce_id,
                         double* bounce_t, double* bounce_normal, uint8_t* bounce_front) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_bounce_visibility");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_bounce_visibility before rt_upload_scene");
  if (!cam || cam->image_width <= 0 || !(cam->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  rt_camera_frame f;
  rt_camera_initialize(cam, &f);
  const size_t n = size_t(f.image_width) * size_t(f.image_height);
  std::vector<float> ht(n), hn(3 * n), rec(kAovBounce * n);
  int rc = render_aov(ctx, cam, f, seed, true, prim_id, ht.data(), hn.data(), rec.data());
  if (rc != RT_OK) return rc;
  for (size_t i = 0; i < n; i++) {
    const float* r = rec.data() + kAovBounce * i;
    if (t) t[i] = double(ht[i]);
    for (int k = 0; k < 3; k++) {
      if (origin1) origin1[3 * i + k] = r[k];
      if (dir1) dir1[3 * i + k] = r[3 + k];
      if (bounce_normal) bounce_normal[3 * i + k] = double(r[6 + k]);
    }
    if (bounce_t) bounce_t[i] = double(r[9]);
    if (bounce_id) bounce_id[i] = __builtin_bit_cast(int32_t, r[10]);
    if (bounce_front) bounce_front[i] = r[11] != 0.0f;
  }
  return RT_OK;
}

int rt_primary_visibility(rt_ctx* ctx, const rt_camera_desc* cam, int32_t flags, int32_t* prim_id, double* t, double* normal) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_primary_visibility");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_primary_visibility before rt_upload_scene");
  if (!cam || cam->image_width <= 0 || !(cam->aspect_ratio > 0)) return fail(ctx, RT_ERR_INVALID, "bad camera");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  rt_camera_frame f;
  rt_camera_initialize(cam, &f);
  const long long n = (long long)f.image_width * f.image_height;
  Scratch sx;
  if (flags & RT_TRACE_RENDER_KERNEL) {
    if (flags & RT_TRACE_EXACT) return fail(ctx, RT_ERR_INVALID, "RT_TRACE_RENDER_KERNEL is the fp32 production traversal: not with RT_TRACE_EXACT");
    std::vector<float> ht(static_cast<size_t>(n)), hn(static_cast<size_t>(3 * n));
    int rc = render_aov(ctx, cam, f, 0, false, prim_id, ht.data(), hn.data(), nullptr);
    if (rc != RT_OK) return rc;
    if (t)
      for (long long i = 0; i < n; i++) t[i] = double(ht[size_t(i)]);
    if (normal)
      for (long long i = 0; i < 3 * n; i++) normal[i] = double(hn[size_t(i)]);
    return RT_OK;
  }
  double* d_o = sx.alloc<double>(size_t(3 * n));
  double* d_d = sx.alloc<double>(size_t(3 * n));
  if (!d_o || !d_d) return fail(ctx, RT_ERR_CUDA, "cudaMalloc failed");
  dim3 grid((f.image_width + 127) / 128, f.image_height);
  center_rays_kernel<<<grid, 128, 0, ctx->stream>>>(f, d_o, d_d);
  ctx->launches++;
  RT_CUDA(ctx, cudaGetLastError());
  return run_trace(ctx, n, d_o, d_d, nullptr, nullptr, 0.001, INFINITY, flags, prim_id, t, normal, nullptr, sx);
}

int rt_medium_spans(rt_ctx* ctx, int32_t medium_index, int64_t n, const double* origin, const double* direction, const double* time, double* t1,
                    double* t2) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_medium_spans");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_medium_spans before rt_upload_scene");
  if (medium_index < 0 || medium_index >= ctx->sc.n_media) return fail(ctx, RT_ERR_INVALID, "medium index out of range");
  if (n < 0 || !origin || !direction || !t1 || !t2) return fail(ctx, RT_ERR_INVALID, "bad arrays");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  Scratch sx;
  const double* d_o = sx.to_device(origin, size_t(3 * n));
  const double* d_d = sx.to_device(direction, size_t(3 * n));
  const double* d_t = sx.to_device(time, size_t(n));
  double* d_1 = sx.alloc<double>(size_t(n));
  double* d_2 = sx.alloc<double>(size_t(n));
  if (!d_o || !d_d || !d_1 || !d_2) return fail(ctx, RT_ERR_CUDA, "cudaMalloc failed");
  if (n > 0) {
    medium_spans_kernel<<<unsigned((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->sc, medium_index, n, d_o, d_d, d_t, d_1, d_2);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
  }
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  RT_CUDA(ctx, cudaMemcpy(t1, d_1, size_t(n) * 8, cudaMemcpyDeviceToHost));
  RT_CUDA(ctx, cudaMemcpy(t2, d_2, size_t(n) * 8, cudaMemcpyDeviceToHost));
  return RT_OK;
}

int rt_eval_texture(rt_ctx* ctx, int32_t texture, int64_t n, const double* uvp, float* rgb) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_eval_texture");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_eval_texture before rt_upload_scene");
  if (texture < 0 || texture >= ctx->sc.n_textures) return fail(ctx, RT_ERR_INVALID, "texture index out of range");
  if (n < 0 || !uvp || !rgb) return fail(ctx, RT_ERR_INVALID, "bad arrays");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  Scratch sx;
  const double* d_in = sx.to_device(uvp, size_t(5 * n));
  float* d_out = sx.alloc<float>(size_t(3 * n));
  if (!d_in || !d_out) return fail(ctx, RT_ERR_CUDA, "cudaMalloc failed");
  if (n > 0) {
    eval_texture_kernel<<<unsigned((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->sc, texture, n, d_in, d_out);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
  }
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  RT_CUDA(ctx, cudaMemcpy(rgb, d_out, size_t(n) * 12, cudaMemcpyDeviceToHost));
  return RT_OK;
}

int rt_eval_scatter(rt_ctx* ctx, int32_t material, int64_t n, uint64_t seed, const double* dir_in, const double* normal, const uint8_t* front_face,
                    float* dir_out, float* attenuation, uint8_t* scattered) {
  if (!ctx) return RT_ERR_INVALID;
  DebugScope dbg("rt_eval_scatter");
  if (!ctx->has_scene) return fail(ctx, RT_ERR_NO_SCENE, "rt_eval_scatter before rt_upload_scene");
  if (material < 0 || material >= ctx->sc.n_materials) return fail(ctx, RT_ERR_INVALID, "material index out of range");
  if (n < 0 || !dir_in || !normal || !front_face || !dir_out || !attenuation || !scattered) return fail(ctx, RT_ERR_INVALID, "bad arrays");
  RT_CUDA(ctx, cudaSetDevice(ctx->device));
  Scratch sx;
  const double* d_di = sx.to_device(dir_in, size_t(3 * n));
  const double* d_n = sx.to_device(normal, size_t(3 * n));
  const unsigned char* d_f = sx.to_device(front_face, size_t(n));
  float* d_do = sx.alloc<float>(size_t(3 * n));
  float* d_a = sx.alloc<float>(size_t(3 * n));
  unsigned char* d_s = sx.alloc<unsigned char>(size_t(n));
  if (!d_di || !d_n || !d_f || !d_do || !d_a || !d_s) return fail(ctx, RT_ERR_CUDA, "cudaMalloc failed");
  if (n > 0) {
    eval_scatter_kernel<<<unsigned((n + 255) / 256), 256, 0, ctx->stream>>>(ctx->sc, material, n, seed, d_di, d_n, d_f, d_do, d_a, d_s);
    ctx->launches++;
    RT_CUDA(ctx, cudaGetLastError());
  }
  RT_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  RT_CUDA(ctx, cudaMemcpy(dir_out, d_do, size_t(n) * 12, cudaMemcpyDeviceToHost));
  RT_CUDA(ctx, cudaMemcpy(attenuation, d_a, size_t(n) * 12, cudaMemcpyDeviceToHost));
  RT_CUDA(ctx, cudaMemcpy(scattered, d_s, size_t(n), cudaMemcpyDeviceToHost));
  return RT_OK;
}

// Host-only view of the scene converter, for CPU tests of the host logic (no GPU needed):
// fills counts[0..8] = nodes, spheres, quads, media, leaf refs, bvh depth, chains, materials, boxes.
int rt_debug_build_stats(const rt_scene_desc* scene, int32_t* counts, double* sah_cost) {
  HostScene h;
  if (!build_host_scene(scene, h)) return RT_ERR_INVALID;
  if (counts) {
    counts[0] = int(h.nodes.size() / 4), counts[1] = int(h.spheres.size() / 2), counts[2] = int(h.quads.size() / 3);
    counts[3] = int(h.media.size()), counts[4] = int(h.leaf_refs.size()), counts[5] = h.bvh_depth;
    counts[6] = int(h.xchains.size()), counts[7] = int(h.materials.size() / 2);
    counts[8] = int(h.boxes.size() / 3);
  }
  if (sah_cost) *sah_cost = h.sah_cost;
  return RT_OK;
}

}  // extern "C"
