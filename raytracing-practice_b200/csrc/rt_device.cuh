// rt_device.cuh — device-side building blocks of the B200 path tracer (sm_100a).
//
// What each block replaces in the reference (file:line under src/):
//   philox4x32 / Rng         std::rand via random_double           common/rtweekend.hpp:23-39
//   closest_hit              hittable_list::hit + bvh_node::hit    hittable/hittable_list.hpp:40-64,
//                            + aabb::hit                           accelerator/bvh_node.hpp:80-94, aabb.hpp:61-112
//   hit_sphere / hit_quad    sphere::hit / quad::hit               hittable/sphere.hpp:47-93, quad.hpp:44-114
//   medium_sample            constant_medium::hit                  SURVEY.md Appendix B.2
//   texture_value            texture::value (4 kinds) + perlin     core/texture.hpp:34-151, core/perlin.hpp:95-255
//   scatter_ray              material::scatter / emitted (5 kinds) core/material.hpp:29-236, SURVEY B.3
//   exact_*                  the same hit() routines in fp64 with the reference's operation order
//                            (no FMA contraction), used only by the parity harness.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

#include "device_scene.h"

namespace rtb200 {

// ---- checks build (-DRT_CHECKS=1; tools/sanitize.sh) ---------------------------------------------------------------------
// compute-sanitizer is closed on this GPU pool, so the library carries its own bounds checks: in a checks build every
// dynamically indexed access of the kernels (BVH nodes, leaf references, primitive / material / texture / texel arrays,
// both traversal stacks, the accumulator) is tested against its array's size; a failure records its site code in
// g_rt_check_fail (largest code wins) and the next rt_synchronize returns RT_ERR_CUDA naming the site (the access itself
// still happens: the check reports, it does not repair).  RT_B200_CHECK_SELFTEST=1 plants one bad reference at upload so
// that the mechanism itself can be seen to fire.  Product builds compile none of it.
#ifndef RT_CHECKS
#define RT_CHECKS 0
#endif
#if RT_CHECKS
__device__ unsigned int g_rt_check_fail = 0u;
__device__ unsigned int g_rt_check_count = 0u;  // checks evaluated (a checks build that evaluates none proves nothing)
#define RT_CHECK(cond, code) \
  do { \
    atomicAdd(&g_rt_check_count, 1u); \
    if (!(cond)) atomicMax(&g_rt_check_fail, (unsigned int)(code)); \
  } while (0)
#else
#define RT_CHECK(cond, code) \
  do { \
  } while (0)
#endif
// site codes
enum : int { CHK_NODE = 1, CHK_STACK_LOCAL = 2, CHK_STACK_SMEM = 3, CHK_LEAF_REF = 4, CHK_SPHERE = 5, CHK_QUAD = 6, CHK_BOX = 7, CHK_MEDIUM = 8, CHK_MATERIAL = 9,
             CHK_TEXTURE = 10, CHK_TEXEL = 11, CHK_PIXEL = 12, CHK_BREF = 13, CHK_STATE = 14, CHK_VIEW = 15 };

// Big, rarely executed helpers are kept OUT of line (RT_OUTLINE): the fully inlined megakernel was
// 4,096 SASS instructions = 64 KB, and with 32 resident warps at scattered PCs the top stall was
// 'no instruction' (instruction-cache misses), profiles/r04_render_t1024.md.
#ifndef RT_OUTLINE
#define RT_OUTLINE __noinline__
#endif

// ---------------------------------------------------------------------------------------
// small float3 algebra
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(s * a.x, s * a.y, s * a.z); }
__device__ __forceinline__ float dot(float3 a, float3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
__device__ __forceinline__ float3 fma3(float s, float3 a, float3 b) { return f3(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z)); }
__device__ __forceinline__ float3 xyz(float4 v) { return f3(v.x, v.y, v.z); }
__device__ __forceinline__ float3 normalize3(float3 a) { return rsqrtf(dot(a, a)) * a; }
// 1/x as ONE MUFU.RCP (1 ulp): the IEEE __frcp_rn is a Newton step plus a denormal slow-path call, ~10 instructions
// at every use, and the production fp32 path has no use for the last bit (the exact predicate is fp64)
__device__ __forceinline__ float rcp_fast(float x) { return __fdividef(1.0f, x); }

// ---------------------------------------------------------------------------------------
// Philox-4x32 (Salmon et al. 2011; RT_PHILOX_ROUNDS rounds), counter-based: the sample set of a (pixel, sample,
// bounce) is a pure function of the key, so images do not depend on how samples are sharded
// over threads, launches or GPUs.
#ifndef RT_PHILOX_ROUNDS
#define RT_PHILOX_ROUNDS 7  // Philox4x32-7: the fewest rounds that pass BigCrush (Salmon et al. 2011, table 2); 10 is their
                            // conservative default and costs +2.5..5 % of the whole render (gpurun_out/ab_philox.log)
#endif
#ifndef RT_OUTLINE_PHILOX
#define RT_OUTLINE_PHILOX __forceinline__  // 4 call sites of ~45 instructions: inlined since the state diet (+1.3..2.2 %, gpurun_out/ab_phinl.log)
#endif
__device__ __forceinline__ uint4 philox4x32_10_inl(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < RT_PHILOX_ROUNDS; r++) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ RT_OUTLINE_PHILOX uint4 philox4x32_10(uint4 ctr, uint2 key) { return philox4x32_10_inl(ctr, key); }
// 24-bit uniform in [0,1): same granularity as the reference's int/float random_double
// (rtweekend.hpp:26) but never exactly 1.0 (SURVEY A.11 / §8 a22).
__device__ __forceinline__ float u01(uint32_t x) { return float(x >> 8) * 5.9604644775390625e-8f; }

struct PathKey {
  uint2 key;       // seed
  uint32_t pixel;  // counter.x
  uint32_t sample; // counter.y
};
__device__ __forceinline__ uint4 rng_block(const PathKey& k, uint32_t bounce, uint32_t stream) {
  return philox4x32_10(make_uint4(k.pixel, k.sample, bounce, stream), k.key);
}
// the same block with the generator inlined: for code that must stay CALL-FREE (see closest_hit_outlined)
__device__ __forceinline__ uint4 rng_block_inl(const PathKey& k, uint32_t bounce, uint32_t stream) {
  return philox4x32_10_inl(make_uint4(k.pixel, k.sample, bounce, stream), k.key);
}

// sin / cos of 2 pi u for u in [0, 1): two MUFU ops after an exact range reduction to [-pi, pi) (|error| ~ 5e-7, far
// below what a sampled direction can show), instead of sincospif's ~40-instruction polynomial path
__device__ __forceinline__ void sincos_2pi(float u, float& s, float& c) {
  const float x = 6.283185307179586f * (u - (u >= 0.5f ? 1.0f : 0.0f));
  s = __sinf(x);
  c = __cosf(x);
}

// uniform direction on the unit sphere from two uniforms: distribution-identical to the
// reference's rejection sampler random_unit_vector (common/vec3.hpp:172-184).
__device__ __forceinline__ float3 unit_vector_from(float u0, float u1) {
  float z = 1.0f - 2.0f * u0;
  float r = sqrtf(fmaxf(0.0f, 1.0f - z * z));
  float s, c;
  sincos_2pi(u1, s, c);
  return f3(r * c, r * s, z);
}

// ---------------------------------------------------------------------------------------
struct Hit {
  float t;
  uint32_t ref;  // REF_NONE = miss
};

// sphere::hit (sphere.hpp:47-93) in a cancellation-free fp32 form: with l = oc - (b/a) d the
// discriminant is a (r^2 - |l|^2) instead of b^2 - a c (both ~1e6 for the r=1000 ground).
// `self`: the ray starts ON this sphere (it scattered there); the roots are then exactly 0
// and -2b/a, which removes fp32 self-intersection without an epsilon.
__device__ __forceinline__ float hit_sphere(float4 g0, float4 g1, float3 o, float3 d, float time, float tmin, float tmax, bool self) {
  float3 c = fma3(time, xyz(g1), xyz(g0));
  float3 oc = o - c;
  float a = dot(d, d);
  float b = dot(oc, d);
  float inv_a = rcp_fast(a);
  if (self) {
    float t = -2.0f * b * inv_a;
    return (t > tmin && t < tmax) ? t : -1.0f;
  }
  float3 l = fma3(-b * inv_a, d, oc);
  float disc = fmaf(g0.w, g0.w, -dot(l, l));
  if (disc < 0.0f) return -1.0f;
  float s = sqrtf(a * disc);
  float t = (-b - s) * inv_a;
  if (!(t > tmin && t < tmax)) {  // interval::surrounds
    t = (-b + s) * inv_a;
    if (!(t > tmin && t < tmax)) return -1.0f;
  }
  return t;
}

// both roots (for medium boundaries); returns false when the line misses the sphere
__device__ __forceinline__ bool sphere_roots(float4 g0, float4 g1, float3 o, float3 d, float time, float& r0, float& r1) {
  float3 c = fma3(time, xyz(g1), xyz(g0));
  float3 oc = o - c;
  float a = dot(d, d);
  float b = dot(oc, d);
  float inv_a = rcp_fast(a);
  float3 l = fma3(-b * inv_a, d, oc);
  float disc = fmaf(g0.w, g0.w, -dot(l, l));
  if (disc < 0.0f) return false;
  float s = sqrtf(a * disc);
  r0 = (-b - s) * inv_a;
  r1 = (-b + s) * inv_a;
  return true;
}

// quad::hit (quad.hpp:44-94) with the interior test (:97-114) folded into two plane
// equations: alpha = A.p + a0, beta = B.p + b0 (A = v x w, B = w x u precomputed on the host).
__device__ __forceinline__ float hit_quad(float4 nD, float4 A, float4 B, float3 o, float3 d, float tmin, float tmax) {
  float denom = dot(xyz(nD), d);
  if (fabsf(denom) < 1e-8f) return -1.0f;
  float t = __fdividef(nD.w - dot(xyz(nD), o), denom);
  if (!(t >= tmin && t <= tmax)) return -1.0f;  // interval::contains
  float3 p = fma3(t, d, o);
  float alpha = dot(xyz(A), p) + A.w;
  float beta = dot(xyz(B), p) + B.w;
  if (!(alpha >= 0.0f && alpha <= 1.0f && beta >= 0.0f && beta <= 1.0f)) return -1.0f;
  return t;
}

// box(a, b, mat) (quad.hpp:129-159: six quads) as one slab test in the box's frame.  A translate / rotate_y
// instance of the box is the 2x2 rotation of (o - t, d) — the per-ray transform of translate::hit / rotate_y::hit
// (hittable.hpp:86-104, SURVEY B.1), paid only by rays that reach this leaf.  The two roots are where the line
// crosses the box surface: the smaller one is the closest of the (up to two) quads quad::hit would report.
struct BoxSlabs {
  float nx, ny, nz, fx, fy, fz;  // per-axis entry / exit parameters
  float3 d;                      // direction in the box frame (its signs name the faces)
  float tn, tf;
};
// `inv`, `ood` = 1/d and o/d of the WORLD ray: an unrotated box (translation folded into its bounds) reuses them
__device__ __forceinline__ bool box_slabs(float4 b0, float4 b1, float4 b2, float3 o, float3 d, float3 inv, float3 ood, int self_face, BoxSlabs& r) {
  float x0, x1, y0, y1, z0, z1;
  if (b2.w != 0.0f) {
    const float3 q = o - xyz(b2);
    const float c = b0.w, s = b1.w;
    o = f3(c * q.x - s * q.z, q.y, s * q.x + c * q.z);
    d = f3(c * d.x - s * d.z, d.y, s * d.x + c * d.z);
    const float ix = fabsf(d.x) > 1e-30f ? rcp_fast(d.x) : copysignf(1e30f, d.x);
    const float iz = fabsf(d.z) > 1e-30f ? rcp_fast(d.z) : copysignf(1e30f, d.z);
    x0 = (b0.x - o.x) * ix, x1 = (b1.x - o.x) * ix;
    y0 = (b0.y - o.y) * inv.y, y1 = (b1.y - o.y) * inv.y;  // rotate_y leaves d.y alone: the world 1/d.y serves
    z0 = (b0.z - o.z) * iz, z1 = (b1.z - o.z) * iz;
  } else {
    x0 = fmaf(b0.x, inv.x, -ood.x), x1 = fmaf(b1.x, inv.x, -ood.x);
    y0 = fmaf(b0.y, inv.y, -ood.y), y1 = fmaf(b1.y, inv.y, -ood.y);
    z0 = fmaf(b0.z, inv.z, -ood.z), z1 = fmaf(b1.z, inv.z, -ood.z);
  }
  if (self_face >= 0) {  // a ray that starts ON that face of this box crosses its plane at exactly 0: no fp32 epsilon
    x0 = self_face == 0 ? 0.0f : x0, x1 = self_face == 1 ? 0.0f : x1;  // selects, not a jump table
    y0 = self_face == 2 ? 0.0f : y0, y1 = self_face == 3 ? 0.0f : y1;
    z0 = self_face == 4 ? 0.0f : z0, z1 = self_face == 5 ? 0.0f : z1;
  }
  r.nx = fminf(x0, x1), r.ny = fminf(y0, y1), r.nz = fminf(z0, z1);
  r.fx = fmaxf(x0, x1), r.fy = fmaxf(y0, y1), r.fz = fmaxf(z0, z1);
  r.d = d;
  r.tn = fmaxf(fmaxf(r.nx, r.ny), r.nz);
  r.tf = fminf(fminf(r.fx, r.fy), r.fz);
  return r.tn <= r.tf;
}
// quad::hit over the six faces with interval::contains on (tmin, tmax): the entry point if it is inside the
// interval, else the exit point; returns -1 or t, and the face hit (axis * 2 + hi side)
__device__ __forceinline__ float hit_box(float4 b0, float4 b1, float4 b2, float3 o, float3 d, float3 inv, float3 ood, float tmin, float tmax, int self_face,
                                         int& face) {
  BoxSlabs r;
  if (!box_slabs(b0, b1, b2, o, d, inv, ood, self_face, r)) return -1.0f;
  if (r.tn >= tmin && r.tn <= tmax) {  // entry: the axis whose near plane is crossed last, on the side the ray comes from
    const int a = (r.nx >= r.ny && r.nx >= r.nz) ? 0 : (r.ny >= r.nz ? 1 : 2);
    const float da = a == 0 ? r.d.x : (a == 1 ? r.d.y : r.d.z);
    face = a * 2 + (da > 0.0f ? 0 : 1);
    return r.tn;
  }
  if (r.tf >= tmin && r.tf <= tmax) {
    const int a = (r.fx <= r.fy && r.fx <= r.fz) ? 0 : (r.fy <= r.fz ? 1 : 2);
    const float da = a == 0 ? r.d.x : (a == 1 ? r.d.y : r.d.z);
    face = a * 2 + (da > 0.0f ? 1 : 0);
    return r.tf;
  }
  return -1.0f;
}
// both surface crossings of the LINE (for medium boundaries)
__device__ __forceinline__ bool box_roots(float4 b0, float4 b1, float4 b2, float3 o, float3 d, float& r0, float& r1) {
  const float3 inv = f3(fabsf(d.x) > 1e-30f ? rcp_fast(d.x) : copysignf(1e30f, d.x), fabsf(d.y) > 1e-30f ? rcp_fast(d.y) : copysignf(1e30f, d.y),
                        fabsf(d.z) > 1e-30f ? rcp_fast(d.z) : copysignf(1e30f, d.z));
  BoxSlabs r;
  const bool ok = box_slabs(b0, b1, b2, o, d, inv, o * inv, -1, r);
  r0 = r.tn, r1 = r.tf;
  return ok;
}

// ---------------------------------------------------------------------------------------
// BVH node access: the first `smem_nodes` nodes (breadth-first = top levels) live in shared
// memory, the rest is read through the read-only path (L1/L2 resident: the arrays are tiny).
#ifndef RT_NODE_CH
#define RT_NODE_CH 2  // staged BVH nodes as (centre, half extent), node_step without per-axis min / max: +4..5.5 % on the BVH-heavy scenes, same accumulators (gpurun_out/ab_ch1.log, ab_ss1.log); 0 = the (lo, hi) form
#endif
#ifndef RT_NODE_PLANAR
#define RT_NODE_PLANAR 0  // 1: fully staged BVHs keep the four quarters of the node records in four planes (bank spreading)
#endif
static_assert(!RT_NODE_PLANAR || RT_NODE_CH, "planar staging is implemented on the (centre, half extent) staging path");
struct NodeSource {
  const float4* smem;
  const float4* gmem;
  int smem_nodes;
  uint32_t smem_addr;  // 32-bit shared-window address of `smem`, see node_source()
  uint32_t plane;      // RT_NODE_PLANAR: bytes per plane = 16 x staged nodes
#if RT_CHECKS
  int n_nodes;
#endif
};
// The shared address is laundered through an opaque mov so that it LIVES IN A REGISTER: left to itself the compiler
// rebuilds it (S2R CgaCtaId, MOV, LEA, IMAD) at every node step.
__device__ __forceinline__ NodeSource node_source(const float4* smem, const float4* gmem, int smem_nodes, int n_nodes = 0x7fffffff) {
  uint32_t a = uint32_t(__cvta_generic_to_shared(smem));
  asm volatile("mov.u32 %0, %0;" : "+r"(a));
#if RT_CHECKS
  return NodeSource{smem, gmem, smem_nodes, a, 16u * uint32_t(smem_nodes), n_nodes};
#else
  return NodeSource{smem, gmem, smem_nodes, a, 16u * uint32_t(smem_nodes)};
#endif
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
// Leaf data staged in shared memory next to the nodes (kernels specialised with ALL_SMEM): 32-bit shared-window
// addresses of copies of leaf_refs / spheres / boxes.  A leaf visit then makes no global load at all (quads and media,
// rare as leaf items, still go to global memory), and the reference -> primitive chain is two LDS, not two LDG.
struct LeafSource {
  uint32_t refs, spheres, boxes;
};
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t opaque_u32(uint32_t a) {  // keeps a shared address in a register (see node_source)
  asm volatile("mov.u32 %0, %0;" : "+r"(a));
  return a;
}

template <bool ALL_SMEM = false>
__device__ __forceinline__ void load_node(const NodeSource& ns, int idx, float4& a, float4& b, float4& c, int& c0, int& c1) {
  float4 dd;
  RT_CHECK(idx >= 0 && idx < ns.n_nodes, CHK_NODE);
  if (RT_NODE_PLANAR && ALL_SMEM) {
    // planar staging (stage_nodes): quarter q of every record in its own plane, so the 16-byte reads a warp makes of 32
    // random nodes spread over all eight 16-byte bank groups (idx & 7) instead of the two a 64-byte record allows
    const uint32_t p = ns.smem_addr + 16u * uint32_t(idx);
    a = lds_f4(p), b = lds_f4(p + ns.plane), c = lds_f4(p + 2u * ns.plane);
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(dd.x), "=f"(dd.y) : "r"(ns.smem_addr + 3u * ns.plane + 8u * uint32_t(idx)));
  } else if (ALL_SMEM || idx < ns.smem_nodes) {
    // 32-bit shared-window address: through the generic pointer the compiler rebuilt the window base
    // (S2R CgaCtaId, MOV, LEA, LEA) at every node step
    const uint32_t p = ns.smem_addr + 64u * uint32_t(idx);
    a = lds_f4(p), b = lds_f4(p + 16u), c = lds_f4(p + 32u);
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(dd.x), "=f"(dd.y) : "r"(p + 48u));
  } else {
    const float4* p = ns.gmem + 4 * idx;
    a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), dd = __ldg(p + 3);
  }
  c0 = __float_as_int(dd.x);
  c1 = __float_as_int(dd.y);
}

// Copies the first `n` BVH node records into shared memory.  With RT_NODE_CH and a fully staged BVH every (lo, hi) pair
// becomes (centre, half extent) on the way, rounded so that [c - h, c + h] contains [lo, hi]: the box the traversal sees
// never shrinks.  The staged record is child-interleaved, {c0x c1x c0y c1y} {c0z c1z h0x h1x} {h0y h1y h0z h1z}
// {child0 child1 - -}, so that each (child 0, child 1) pair of a value sits in two adjacent registers: the operand of
// one packed FFMA2 in node_step.
template <bool ALL_SMEM>
__device__ __forceinline__ void stage_nodes(float4* s_nodes, const float4* __restrict__ g_nodes, int n) {
  if (RT_NODE_CH && ALL_SMEM) {
    auto ch = [](float& lo, float& hi) {
      const float c = 0.5f * (lo + hi);
      const float h = fmaxf(__fsub_ru(hi, c), __fsub_ru(c, lo));
      lo = c, hi = h;
    };
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      float4 a = g_nodes[4 * i], b = g_nodes[4 * i + 1], c = g_nodes[4 * i + 2];
      ch(a.x, a.w), ch(a.y, b.x), ch(a.z, b.y);  // child 0: x, y, z
      ch(b.z, c.y), ch(b.w, c.z), ch(c.x, c.w);  // child 1
      const float4 q0 = make_float4(a.x, b.z, a.y, b.w), q1 = make_float4(a.z, c.x, a.w, c.y), q2 = make_float4(b.x, c.z, b.y, c.w);
      a = q0, b = q1, c = q2;
      if (RT_NODE_PLANAR) {
        const float4 dd = g_nodes[4 * i + 3];
        s_nodes[i] = a, s_nodes[n + i] = b, s_nodes[2 * n + i] = c;
        reinterpret_cast<float2*>(s_nodes + 3 * n)[i] = make_float2(dd.x, dd.y);
      } else {
        s_nodes[4 * i] = a, s_nodes[4 * i + 1] = b, s_nodes[4 * i + 2] = c, s_nodes[4 * i + 3] = g_nodes[4 * i + 3];
      }
    }
  } else {
    for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) s_nodes[i] = g_nodes[i];
  }
}

// constant_medium::hit (SURVEY B.2) for one medium: entry/exit over the boundary primitives,
// then an exponential free-flight sample.  `u` is the uniform this medium owns for this ray.
__device__ __forceinline__ bool medium_span(const DeviceScene& sc, const DMedium& m, float3 o, float3 d, float time, float& t1, float& t2) {
  const float INF = __int_as_float(0x7f800000);
  if (m.n_bref == 1) {  // a single sphere (the usual boundary): both passes below come from ONE pair of roots
    const uint32_t ref = __ldg(sc.medium_brefs + m.first_bref);
    RT_CHECK((ref >> 30) != REF_SPHERE || (ref & 0x3FFFFFFFu) < uint32_t(sc.n_spheres), CHK_BREF);
    if ((ref >> 30) == REF_SPHERE) {
      const uint32_t idx = ref & 0x3FFFFFFFu;
      float r0, r1;
      t1 = INF;
      if (!sphere_roots(__ldg(sc.spheres + 2 * idx), __ldg(sc.spheres + 2 * idx + 1), o, d, time, r0, r1)) return false;
      t1 = r0;                                // pass 1: the smallest crossing
      t2 = r1 > t1 + 0.0001f ? r1 : INF;      // pass 2: the next crossing beyond t1 + 0.0001 (r0 itself never is)
      return t2 != INF;
    }
    if ((ref >> 30) == REF_BOX) {  // a single box() (the Cornell smoke volumes): likewise ONE pair of roots instead of two
      const uint32_t b = (ref & 0x3FFFFFFFu) >> 3;  // slab evaluations — the general passes below would compute the same r0, r1 twice
      float r0, r1;
      t1 = INF;
      if (!box_roots(__ldg(sc.boxes + 3 * b), __ldg(sc.boxes + 3 * b + 1), __ldg(sc.boxes + 3 * b + 2), o, d, r0, r1)) return false;
      t1 = r0;                                // pass 1
      t2 = r1 >= t1 + 0.0001f ? r1 : INF;     // pass 2 (quads: interval::contains); r0 >= r0 + 0.0001 never holds
      return t2 != INF;
    }
  }
  t1 = INF;
  // pass 1: boundary->hit(r, universe): the smallest crossing
  for (int k = 0; k < m.n_bref; k++) {
    uint32_t ref = __ldg(sc.medium_brefs + m.first_bref + k);
    uint32_t idx = ref & 0x3FFFFFFFu;
    if ((ref >> 30) == REF_SPHERE) {
      float r0, r1;
      if (sphere_roots(__ldg(sc.spheres + 2 * idx), __ldg(sc.spheres + 2 * idx + 1), o, d, time, r0, r1)) t1 = fminf(t1, r0);
    } else if ((ref >> 30) == REF_BOX) {
      float r0, r1;
      const uint32_t b = idx >> 3;
      if (box_roots(__ldg(sc.boxes + 3 * b), __ldg(sc.boxes + 3 * b + 1), __ldg(sc.boxes + 3 * b + 2), o, d, r0, r1)) t1 = fminf(t1, r0);
    } else {
      float t = hit_quad(__ldg(sc.quads + 3 * idx), __ldg(sc.quads + 3 * idx + 1), __ldg(sc.quads + 3 * idx + 2), o, d, -INF, INF);
      if (t != -1.0f) t1 = fminf(t1, t);
    }
  }
  if (t1 == INF) return false;
  // pass 2: boundary->hit(r, interval(t1 + 0.0001, inf)): the next crossing
  const float lo = t1 + 0.0001f;
  t2 = INF;
  for (int k = 0; k < m.n_bref; k++) {
    uint32_t ref = __ldg(sc.medium_brefs + m.first_bref + k);
    uint32_t idx = ref & 0x3FFFFFFFu;
    if ((ref >> 30) == REF_SPHERE) {
      float r0, r1;
      if (sphere_roots(__ldg(sc.spheres + 2 * idx), __ldg(sc.spheres + 2 * idx + 1), o, d, time, r0, r1)) {
        float t = r0 > lo ? r0 : (r1 > lo ? r1 : INF);
        t2 = fminf(t2, t);
      }
    } else if ((ref >> 30) == REF_BOX) {
      float r0, r1;
      const uint32_t b = idx >> 3;
      if (box_roots(__ldg(sc.boxes + 3 * b), __ldg(sc.boxes + 3 * b + 1), __ldg(sc.boxes + 3 * b + 2), o, d, r0, r1)) {
        float t = r0 >= lo ? r0 : (r1 >= lo ? r1 : INF);  // quads: interval::contains
        t2 = fminf(t2, t);
      }
    } else {
      float t = hit_quad(__ldg(sc.quads + 3 * idx), __ldg(sc.quads + 3 * idx + 1), __ldg(sc.quads + 3 * idx + 2), o, d, lo, INF);
      if (t != -1.0f) t2 = fminf(t2, t);
    }
  }
  return t2 != INF;
}

// Per-ray uniforms for media: medium k owns component (k & 3) of Philox block stream 1 + (k >> 2)
// of the ray's (pixel, sample, bounce) counter.
template <bool CALLFREE = false>
__device__ __forceinline__ float medium_uniform(const PathKey& key, uint32_t bounce, int medium) {
  uint4 r = CALLFREE ? rng_block_inl(key, bounce, 1u + (uint32_t(medium) >> 2)) : rng_block(key, bounce, 1u + (uint32_t(medium) >> 2));
  uint32_t c = uint32_t(medium) & 3u;
  return u01(c == 0 ? r.x : (c == 1 ? r.y : (c == 2 ? r.z : r.w)));
}

// The free-flight uniform is drawn LAZILY, only once the ray is known to cross the medium inside
// [tmin, tmax]: most BVH-leaf visits of a medium's bounding box miss the boundary itself, and the
// Philox block was 2/3 of this function's instructions (profiles/r06_pool_kernel.md).
template <bool CALLFREE>
__device__ __forceinline__ float medium_sample_impl(const DeviceScene& sc, const DMedium& m, int mi, float3 o, float3 d, float time, float tmin, float tmax,
                                                    const PathKey& key, uint32_t bounce) {
  float t1, t2;
  if (!medium_span(sc, m, o, d, time, t1, t2)) return -1.0f;
  t1 = fmaxf(t1, tmin);
  t2 = fminf(t2, tmax);
  if (t1 >= t2) return -1.0f;
  t1 = fmaxf(t1, 0.0f);
  float len = sqrtf(dot(d, d));
  float inside = (t2 - t1) * len;
  const float u = medium_uniform<CALLFREE>(key, bounce, mi);
  float hit_distance = m.neg_inv_density * __logf(u);  // u == 0 -> +inf -> miss, as log(0) in the reference
  if (!(hit_distance <= inside)) return -1.0f;
  return t1 + hit_distance / len;
}
__device__ RT_OUTLINE float medium_sample(const DeviceScene& sc, const DMedium& m, int mi, float3 o, float3 d, float time, float tmin, float tmax,
                                          const PathKey& key, uint32_t bounce) {
  return medium_sample_impl<false>(sc, m, mi, o, d, time, tmin, tmax, key, bounce);
}

constexpr int kStackDepth = 32;
// TravState::cur of a finished (or idle) traversal: negative like a leaf code, but no leaf code can have this value
// (it would need 2^28 leaf references).  Lets a loop read the lane's mode off `cur` alone: >= 0 node, else leaf / done.
constexpr int kTravDone = int(0x80000000u);
#ifndef RT_GM_INLINE
#define RT_GM_INLINE 0
#endif
#ifndef RT_GM_NOUNROLL
#define RT_GM_NOUNROLL 1  // one medium_sample call site for the scene-enclosing media: +0.4..1.2 % (gpurun_out/ab_lean2.log)
#endif
#ifndef RT_NODE_THR
#define RT_NODE_THR 1
#endif
#ifndef RT_POP_BOTH
#define RT_POP_BOTH 1  // +1.3..3 % on book2_final over five A/B runs, other scenes unchanged (gpurun_out/ab_pop.log, ab_pair.log, ab_pair2.log) — see trav_pop
#endif
// (Also measured on the stack: 64-bit {node, distance} entries, one LDL.64 per pop: +-0 %; the newest entry cached in two
//  registers until the next push — most pops then touch no memory —: -7 % on book2_final, the two registers cost more than
//  the latency, gpurun_out/ab_tc.log.  All bit-identical.)
#ifndef RT_KEYFN_NODE_THR
#define RT_KEYFN_NODE_THR 1  // > 1: the render kernel's traversal prefers leaf steps while fewer lanes than this want a node step
#endif
#ifndef RT_SPECULATIVE
#define RT_SPECULATIVE 0  // 1: speculative while-while (node_step_spec); measured 0.88x on book2_final, 0.96-1.00x elsewhere (gpurun_out/ab_spec.log)
#endif
#ifndef RT_NODE_UNROLL
#define RT_NODE_UNROLL 2  // node steps per warp vote: +3..5 % on the BVH-heavy scenes, -4 % on 2-node Cornell trees (gpurun_out/ab_unroll.log)
#endif

// Census slots of the instrumented build (RT_RENDER_COUNTERS): the N_* of SURVEY.md §8(d).
enum : int { CN_NODE = 0, CN_SPH = 1, CN_SPH_HIT = 2, CN_QUAD = 3, CN_QUAD_FULL = 4, CN_MEDIUM = 5, CN_LAMB = 6, CN_METAL = 7,
             CN_DIEL = 8, CN_LIGHT = 9, CN_ISO = 10, CN_TEX_CHECKER = 11, CN_TEX_IMAGE = 12, CN_TEX_NOISE = 13, CN_BOX = 14, CN_COUNT = 15 };

// ---------------------------------------------------------------------------------------
// world.hit(r, interval(tmin, tmax), rec) as a per-lane state machine.
//   bvh_node::hit + aabb::hit  -> node_step  (one BVH2 node: both children's slab tests)
//   hittable_list::hit over leaves, sphere::hit / quad::hit / constant_medium::hit -> leaf_step
// A lane is in one of these modes; the CALLER decides which step the warp executes next
// (closest_hit: while-while; render_kernel: the most populated mode wins), so the same
// traversal code serves the parity queries and the production megakernel.
enum : int { MODE_SHADE = 0, MODE_NODE = 1, MODE_LEAF = 2, MODE_DONE = 3 };

struct TravState {
  float3 o, d, inv, nood;  // nood = -o/d: the addend of the slab FFMA2 in node_step, which has no negation modifier
  float time, tmin;
  Hit best;
  uint32_t skip;  // the primitive the ray starts on (REF_NONE for camera rays / medium scatters)
  int cur, sp;
};
// The traversal stack is kept OUT of TravState (two plain local arrays) so that the scalars above
// are promoted to registers; only the dynamically indexed stack lives in local memory (L1).
struct TravStack {
  int node[kStackDepth];
  float t[kStackDepth];
};

// pop, skipping subtrees that start beyond the current closest hit
__device__ __forceinline__ int trav_pop(TravState& ts, TravStack& st) {
  while (ts.sp > 0) {
    ts.sp--;
#if RT_POP_BOTH
    // Written to request both words of the entry together (the pop loop is 12 % of the PC samples for 7 % of the
    // instructions, profiles/r22_render_final.md).  It does not: NVVM still sinks this load below the distance test — the
    // pop loop's SASS is unchanged — and a real pairing (LDL.64 entries) measures +-0.  What the edit does change is the
    // register allocation of the surrounding loop, and THAT build is reproducibly 1.3-3 % faster on book2_final: kept as a
    // measured code-generation effect, not as a mechanism.
    const int node = *reinterpret_cast<const volatile int*>(&st.node[ts.sp]);
    if (st.t[ts.sp] <= ts.best.t) {
      ts.cur = node;
      return ts.cur >= 0 ? MODE_NODE : MODE_LEAF;
    }
#else
    if (st.t[ts.sp] <= ts.best.t) {
      ts.cur = st.node[ts.sp];
      return ts.cur >= 0 ? MODE_NODE : MODE_LEAF;
    }
#endif
  }
  ts.cur = kTravDone;
  return MODE_SHADE;  // traversal finished: ts.best is the answer
}
__device__ __forceinline__ void trav_push(TravState& ts, TravStack& st, int node, float t) {
  // no overflow guard: rt_upload_scene rejects a BVH deeper than kStackDepth, and the stack never holds more
  // entries than the tree has levels
  RT_CHECK(ts.sp >= 0 && ts.sp < kStackDepth, CHK_STACK_LOCAL);
  st.node[ts.sp] = node;
  st.t[ts.sp] = t;
  ts.sp++;
}

// The same stack in SHARED memory, for kernels whose launch has the room (render_range decides): one 32-bit entry per
// level, (entry distance rounded DOWN to bf16) << 16 | 16-bit child code, laid out [level][thread] so that a warp's
// accesses to one level hit 32 different banks.  One STS per push and one LDS per pop instead of two local-memory
// accesses each, no L1 misses (the local stack's lines compete with the spills for what shared memory leaves of L1:
// 71 % hit rate, profiles/r15_render_lean.md), and the rounded distance is a lower bound of the real one, so a pop
// never culls a subtree the local stack would keep: the closest hit is the same.  Needs child codes that fit 16 bits
// (< 32768 nodes, < 4096 leaf references) and a tree no deeper than the levels the launch reserved; ts.sp is the
// shared-window byte address of the next free entry.
struct TravStackS {
  uint32_t base;    // address of this thread's level-0 entry
  uint32_t stride;  // bytes between levels = 4 x threads per CTA
#if RT_CHECKS
  uint32_t levels;
#endif
};
constexpr int kSmemStackMaxCode = 32767;
__device__ __forceinline__ int trav_pop(TravState& ts, TravStackS& st) {
  while (uint32_t(ts.sp) != st.base) {
    ts.sp -= int(st.stride);
    uint32_t e;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(e) : "r"(uint32_t(ts.sp)) : "memory");
    if (__uint_as_float(e & 0xFFFF0000u) <= ts.best.t) {
      ts.cur = int(e << 16) >> 16;
      return ts.cur >= 0 ? MODE_NODE : MODE_LEAF;
    }
  }
  ts.cur = kTravDone;
  return MODE_SHADE;
}
__device__ __forceinline__ void trav_push(TravState& ts, TravStackS& st, int node, float t) {
  // entry distances are >= tmin > 0: truncating the mantissa rounds down
#if RT_CHECKS
  RT_CHECK(uint32_t(ts.sp) >= st.base && uint32_t(ts.sp) < st.base + st.levels * st.stride, CHK_STACK_SMEM);
  RT_CHECK(node >= -kSmemStackMaxCode - 1 && node <= kSmemStackMaxCode, CHK_STACK_SMEM);
#endif
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(uint32_t(ts.sp)), "r"((__float_as_uint(t) & 0xFFFF0000u) | (uint32_t(node) & 0xFFFFu)) : "memory");
  ts.sp += int(st.stride);
}
__device__ __forceinline__ void trav_reset(TravState& ts, TravStack&) { ts.sp = 0; }
__device__ __forceinline__ void trav_reset(TravState& ts, TravStackS& st) { ts.sp = int(st.base); }

// 1/d with +-huge instead of +-inf so that 0 * inf never produces NaN in the slab test
__device__ __forceinline__ void trav_set_ray(TravState& ts, float3 o, float3 d, float time, float tmin, uint32_t skip) {
  ts.o = o, ts.d = d, ts.time = time, ts.tmin = tmin, ts.skip = skip;
  ts.inv = f3(fabsf(d.x) > 1e-30f ? rcp_fast(d.x) : copysignf(1e30f, d.x), fabsf(d.y) > 1e-30f ? rcp_fast(d.y) : copysignf(1e30f, d.y),
              fabsf(d.z) > 1e-30f ? rcp_fast(d.z) : copysignf(1e30f, d.z));
  ts.nood = -(o * ts.inv);
}

// The scene-enclosing media (met by every ray — the r=5000 fog of the Book-2 final scene) are not BVH leaves:
// they are sampled once per ray, where the caller's lanes are converged; the result seeds the closest hit.
template <bool COUNT>
__device__ __forceinline__ Hit sample_global_media(const DeviceScene& sc, float3 o, float3 d, float time, float tmin, float tmax, const PathKey& key,
                                                   uint32_t bounce, unsigned int* cn) {
  Hit best{tmax, REF_NONE};
#if RT_GM_NOUNROLL
#pragma unroll 1  // one medium_sample call site instead of seven (the compiler unrolls and peels the <= 4 iterations)
#endif
  for (int g = 0; g < sc.n_global_media; g++) {
    const int mi = sc.global_media[g];
    const DMedium m = sc.media[mi];
#if RT_GM_INLINE
    float t = medium_sample_impl<true>(sc, m, mi, o, d, time, tmin, best.t, key, bounce);
#else
    float t = medium_sample(sc, m, mi, o, d, time, tmin, best.t, key, bounce);
#endif
    if (COUNT) cn[CN_MEDIUM]++;
    if (t != -1.0f) best = Hit{t, make_ref(REF_MEDIUM, uint32_t(mi))};
  }
  return best;
}

// Does the ray cross the box of everything the BVH holds inside (tmin, tmax)?  Same arithmetic as node_step on
// boxes that are subsets of this one, and fma / min / max are monotone, so a miss here implies a miss at every
// node: skipping the traversal for such rays cannot change any result.
__device__ __forceinline__ bool ray_meets_scene(const DeviceScene& sc, const TravState& ts, float tmax) {
  const float x0 = fmaf(sc.bounds_lo[0], ts.inv.x, ts.nood.x), x1 = fmaf(sc.bounds_hi[0], ts.inv.x, ts.nood.x);
  const float y0 = fmaf(sc.bounds_lo[1], ts.inv.y, ts.nood.y), y1 = fmaf(sc.bounds_hi[1], ts.inv.y, ts.nood.y);
  const float z0 = fmaf(sc.bounds_lo[2], ts.inv.z, ts.nood.z), z1 = fmaf(sc.bounds_hi[2], ts.inv.z, ts.nood.z);
  const float n = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), ts.tmin));
  const float f = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), tmax));
  return n <= f;
}

// Start a query.  `media`: sample the scene-enclosing media right here.
template <bool COUNT>
__device__ __forceinline__ int trav_begin(TravState& ts, const DeviceScene& sc, float3 o, float3 d, float time, float tmin, float tmax, uint32_t skip,
                                          bool media, const PathKey& key, uint32_t bounce, unsigned int* cn) {
  trav_set_ray(ts, o, d, time, tmin, skip);
  ts.best = Hit{tmax, REF_NONE};
  if (media) ts.best = sample_global_media<COUNT>(sc, o, d, time, tmin, tmax, key, bounce, cn);
  ts.sp = 0;
  ts.cur = 0;
  return MODE_NODE;
}

template <bool COUNT, bool ALL_SMEM = false, typename Stack = TravStack>
__device__ __forceinline__ int node_step(TravState& ts, Stack& st, const NodeSource& ns, unsigned int* cn) {
  float4 a, b, c;
  int c0, c1;
  load_node<ALL_SMEM>(ns, ts.cur, a, b, c, c0, c1);
  if (COUNT) cn[CN_NODE]++;
  const float3 inv = ts.inv, ood = -ts.nood;
  float n0, f0, n1, f1;
  if (RT_NODE_CH && ALL_SMEM) {
    // Staged nodes hold (centre, half extent) per axis, child-interleaved — see stage_nodes(): the slab's two plane
    // distances are tc -+ h |1/d| with tc = (c - o)/d, so near and far need no per-axis min / max.  Each (child 0,
    // child 1) pair of an axis is one packed FFMA2 with the per-lane 1/d, -o/d or |1/d| broadcast to both halves; per
    // component it is the scalar FFMA(.FTZ) of the unpaired form, same operands, same rounding, so the bits are those of
    // three scalar FFMA per axis and child.  FFMA2 has no negation modifier, so packed near planes need -|1/d| in three
    // registers of their own.  That pays in the local-stack plan (the large BVHs: +5 % on C5) and loses 3-5 % in the
    // shared-memory-stack plan of the small scenes (C3a, C3b), which already spills more: there the near planes stay
    // scalar FFMA with the -|.| operand modifier (profiles/r5_ffma2.md).
    constexpr bool kPackNear = !std::is_same<Stack, TravStackS>::value;
    const float2 tx = __ffma2_rn(make_float2(a.x, a.y), make_float2(inv.x, inv.x), make_float2(ts.nood.x, ts.nood.x));
    const float2 ty = __ffma2_rn(make_float2(a.z, a.w), make_float2(inv.y, inv.y), make_float2(ts.nood.y, ts.nood.y));
    const float2 tz = __ffma2_rn(make_float2(b.x, b.y), make_float2(inv.z, inv.z), make_float2(ts.nood.z, ts.nood.z));
    const float2 hx = make_float2(b.z, b.w), hy = make_float2(c.x, c.y), hz = make_float2(c.z, c.w);
    const float3 ai = f3(fabsf(inv.x), fabsf(inv.y), fabsf(inv.z));
    const float2 fx = __ffma2_rn(hx, make_float2(ai.x, ai.x), tx), fy = __ffma2_rn(hy, make_float2(ai.y, ai.y), ty),
                 fz = __ffma2_rn(hz, make_float2(ai.z, ai.z), tz);
    float2 nx, ny, nz;
    if constexpr (kPackNear) {
      const float3 nai = f3(-fabsf(inv.x), -fabsf(inv.y), -fabsf(inv.z));
      nx = __ffma2_rn(hx, make_float2(nai.x, nai.x), tx), ny = __ffma2_rn(hy, make_float2(nai.y, nai.y), ty);
      nz = __ffma2_rn(hz, make_float2(nai.z, nai.z), tz);
    } else {
      nx = make_float2(fmaf(hx.x, -fabsf(inv.x), tx.x), fmaf(hx.y, -fabsf(inv.x), tx.y));
      ny = make_float2(fmaf(hy.x, -fabsf(inv.y), ty.x), fmaf(hy.y, -fabsf(inv.y), ty.y));
      nz = make_float2(fmaf(hz.x, -fabsf(inv.z), tz.x), fmaf(hz.y, -fabsf(inv.z), tz.y));
    }
    n0 = fmaxf(fmaxf(nx.x, ny.x), fmaxf(nz.x, ts.tmin));
    f0 = fminf(fminf(fx.x, fy.x), fminf(fz.x, ts.best.t));
    n1 = fmaxf(fmaxf(nx.y, ny.y), fmaxf(nz.y, ts.tmin));
    f1 = fminf(fminf(fx.y, fy.y), fminf(fz.y, ts.best.t));
  } else {
    // slab test of both children (aabb.hpp:61-112), conservative: keep when tnear <= tfar
    float x0 = fmaf(a.x, inv.x, -ood.x), x1 = fmaf(a.w, inv.x, -ood.x);
    float y0 = fmaf(a.y, inv.y, -ood.y), y1 = fmaf(b.x, inv.y, -ood.y);
    float z0 = fmaf(a.z, inv.z, -ood.z), z1 = fmaf(b.y, inv.z, -ood.z);
    n0 = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), ts.tmin));
    f0 = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), ts.best.t));
    x0 = fmaf(b.z, inv.x, -ood.x), x1 = fmaf(c.y, inv.x, -ood.x);
    y0 = fmaf(b.w, inv.y, -ood.y), y1 = fmaf(c.z, inv.y, -ood.y);
    z0 = fmaf(c.x, inv.z, -ood.z), z1 = fmaf(c.w, inv.z, -ood.z);
    n1 = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), ts.tmin));
    f1 = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), ts.best.t));
  }
  const bool h0 = n0 <= f0, h1 = n1 <= f1;
  if (h0 && h1) {  // near child first, far child on the stack with its entry distance
    const bool first0 = n0 <= n1;
    trav_push(ts, st, first0 ? c1 : c0, first0 ? n1 : n0);
    ts.cur = first0 ? c0 : c1;
    return ts.cur >= 0 ? MODE_NODE : MODE_LEAF;
  }
  if (h0 || h1) {
    ts.cur = h0 ? c0 : c1;
    return ts.cur >= 0 ? MODE_NODE : MODE_LEAF;
  }
  return trav_pop(ts, st);
}

// Speculative variant (Aila & Laine's "speculative while-while"): a lane that reaches a leaf while its postponed-leaf
// slot `pend` is free parks the leaf there and keeps walking, so it stays useful in the node loop instead of idling
// until the slowest lane finds a leaf.  The nodes it visits meanwhile are culled against the closest hit BEFORE the
// parked leaf is intersected — extra visits, never a different answer (a subtree culled later starts beyond best.t).
template <bool COUNT, bool ALL_SMEM = false>
__device__ __forceinline__ void node_step_spec(TravState& ts, TravStack& st, const NodeSource& ns, int& pend, unsigned int* cn) {
  float4 a, b, c;
  int c0, c1;
  load_node<ALL_SMEM>(ns, ts.cur, a, b, c, c0, c1);
  if (COUNT) cn[CN_NODE]++;
  const float3 inv = ts.inv, ood = -ts.nood;
  float x0 = fmaf(a.x, inv.x, -ood.x), x1 = fmaf(a.w, inv.x, -ood.x);
  float y0 = fmaf(a.y, inv.y, -ood.y), y1 = fmaf(b.x, inv.y, -ood.y);
  float z0 = fmaf(a.z, inv.z, -ood.z), z1 = fmaf(b.y, inv.z, -ood.z);
  float n0 = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), ts.tmin));
  float f0 = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), ts.best.t));
  x0 = fmaf(b.z, inv.x, -ood.x), x1 = fmaf(c.y, inv.x, -ood.x);
  y0 = fmaf(b.w, inv.y, -ood.y), y1 = fmaf(c.z, inv.y, -ood.y);
  z0 = fmaf(c.x, inv.z, -ood.z), z1 = fmaf(c.w, inv.z, -ood.z);
  float n1 = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), ts.tmin));
  float f1 = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), ts.best.t));
  const bool h0 = n0 <= f0, h1 = n1 <= f1;
  // (written branch by branch like node_step: folding both cases into one `first0 = h0 && (!h1 || n0 <= n1)` made
  //  nvcc 12.9 push the SAME child it descends into — st.local of c1 unconditionally in the PTX)
  int next = kTravDone;
  if (h0 && h1) {
    const bool first0 = n0 <= n1;
    st.node[ts.sp] = first0 ? c1 : c0;
    st.t[ts.sp] = first0 ? n1 : n0;
    ts.sp++;
    next = first0 ? c0 : c1;
  } else if (h0 || h1) {
    next = h0 ? c0 : c1;
  }
  if (next >= 0 || (next != kTravDone && pend != kTravDone)) {  // a node, or a leaf while the parking slot is taken
    ts.cur = next;
    return;
  }
  if (next != kTravDone) pend = next;  // park the leaf, carry on with the stack
  trav_pop(ts, st);
}

// leaf: ~cur = (first << 3) | (count - 1)
// `key_of(key, bounce)` yields the ray's Philox counter; it is only called when a medium is actually sampled
template <bool COUNT, bool CALLFREE = false, bool STAGED = false, typename KeyFn>
__device__ __forceinline__ void leaf_body(TravState& ts, int leaf, const DeviceScene& sc, bool media, KeyFn key_of, unsigned int* cn, const LeafSource& ls) {
  const int code = ~leaf;
  const int first = code >> 3, count = (code & 7) + 1;
  const float3 o = ts.o, d = ts.d;
  for (int k = 0; k < count; k++) {
    RT_CHECK(first + k >= 0 && first + k < sc.n_leaf_refs, CHK_LEAF_REF);
    uint32_t ref = STAGED ? lds_u32(ls.refs + 4u * uint32_t(first + k)) : __ldg(sc.leaf_refs + first + k);
    uint32_t type = ref >> 30, idx = ref & 0x3FFFFFFFu;
    float t = -1.0f;
    if (ref != REF_NONE) {
      RT_CHECK(type != REF_SPHERE || idx < uint32_t(sc.n_spheres), CHK_SPHERE);
      RT_CHECK(type != REF_QUAD || idx < uint32_t(sc.n_quads), CHK_QUAD);
      RT_CHECK(type != REF_BOX || (idx >> 3) < uint32_t(sc.n_boxes), CHK_BOX);
      RT_CHECK(type != REF_MEDIUM || idx < uint32_t(sc.n_media), CHK_MEDIUM);
    }
    if (type == REF_SPHERE) {
      const float4 g0 = STAGED ? lds_f4(ls.spheres + 32u * idx) : __ldg(sc.spheres + 2 * idx);
      const float4 g1 = STAGED ? lds_f4(ls.spheres + 32u * idx + 16u) : __ldg(sc.spheres + 2 * idx + 1);
      t = hit_sphere(g0, g1, o, d, ts.time, ts.tmin, ts.best.t, ref == ts.skip);
      if (COUNT) cn[CN_SPH]++, cn[CN_SPH_HIT] += t != -1.0f;
    } else if (type == REF_QUAD) {
      if (ref != ts.skip) {
        t = hit_quad(__ldg(sc.quads + 3 * idx), __ldg(sc.quads + 3 * idx + 1), __ldg(sc.quads + 3 * idx + 2), o, d, ts.tmin, ts.best.t);
        if (COUNT) {
          float4 nD = __ldg(sc.quads + 3 * idx);  // "full" = got past the plane / t-range early-outs
          float den = dot(xyz(nD), d), tq = (nD.w - dot(xyz(nD), o)) / den;
          cn[CN_QUAD]++, cn[CN_QUAD_FULL] += (fabsf(den) >= 1e-8f && tq >= ts.tmin && tq <= ts.best.t) || t != -1.0f;
        }
      }
    } else if (type == REF_BOX) {
      if (ref != REF_NONE) {
        const uint32_t b = idx >> 3;
        const int self_face = ((ts.skip >> 30) == REF_BOX && ts.skip != REF_NONE && ((ts.skip & 0x3FFFFFFFu) >> 3) == b) ? int(ts.skip & 7u) : -1;
        int face = 0;
        const float4 b0 = STAGED ? lds_f4(ls.boxes + 48u * b) : __ldg(sc.boxes + 3 * b);
        const float4 b1 = STAGED ? lds_f4(ls.boxes + 48u * b + 16u) : __ldg(sc.boxes + 3 * b + 1);
        const float4 b2 = STAGED ? lds_f4(ls.boxes + 48u * b + 32u) : __ldg(sc.boxes + 3 * b + 2);
        t = hit_box(b0, b1, b2, o, d, ts.inv, -ts.nood, ts.tmin, ts.best.t, self_face, face);
        if (COUNT) cn[CN_BOX]++;
        ref = make_ref(REF_BOX, (b << 3) | uint32_t(face));
      }
    } else if (media) {
      const DMedium m = sc.media[idx];
      PathKey key;
      uint32_t bounce;
      key_of(key, bounce);
      t = CALLFREE ? medium_sample_impl<true>(sc, m, int(idx), o, d, ts.time, ts.tmin, ts.best.t, key, bounce)
                   : medium_sample(sc, m, int(idx), o, d, ts.time, ts.tmin, ts.best.t, key, bounce);
      if (COUNT) cn[CN_MEDIUM]++;
    }
    if (t != -1.0f) ts.best = Hit{t, ref};
  }
}
template <bool COUNT, bool CALLFREE = false, bool STAGED = false, typename KeyFn, typename Stack = TravStack>
__device__ __forceinline__ int leaf_step(TravState& ts, Stack& st, const DeviceScene& sc, bool media, KeyFn key_of, unsigned int* cn,
                                         const LeafSource& ls = LeafSource{0u, 0u, 0u}) {
  leaf_body<COUNT, CALLFREE, STAGED>(ts, ts.cur, sc, media, key_of, cn, ls);
  return trav_pop(ts, st);
}

// Closest hit for one ray per lane, "while-while" (Aila & Laine): all lanes walk internal nodes
// until every lane sits on a leaf, then the leaves are intersected together.  Loop boundaries are
// warp votes with the full mask, which force reconvergence every iteration; MUST be called with
// the warp converged (exited lanes excepted).  With plain per-lane `continue`s the compiler never
// re-merged the lanes: ncu showed 4.75 of 32 active per instruction (profiles/r01_*.md).
// `ts` holds a ray (trav_set_ray) and its closest hit so far (ts.best); lanes with active == false only vote
template <bool COUNT, bool CALLFREE = false>
__device__ __forceinline__ Hit closest_hit_prepared(const DeviceScene& sc, const NodeSource& ns, TravState& ts, bool media, const PathKey& key,
                                                    uint32_t bounce, unsigned int* cn, bool active) {
  const unsigned FULL = 0xFFFFFFFFu;
  TravStack st;
  int mode = MODE_DONE;
  trav_reset(ts, st);
  if (active) ts.cur = 0, mode = MODE_NODE;
#if RT_NODE_THR == 1
  for (;;) {  // while-while: node steps while ANY lane wants one (one vote per step), then one leaf step for the rest
    while (__any_sync(FULL, mode == MODE_NODE))
      if (mode == MODE_NODE) mode = node_step<COUNT>(ts, st, ns, cn);
    if (!__any_sync(FULL, mode == MODE_LEAF)) break;
    if (mode == MODE_LEAF) mode = leaf_step<COUNT, CALLFREE>(ts, st, sc, media, [&](PathKey& k, uint32_t& b) { k = key, b = bounce; }, cn);
  }
#else
  for (;;) {
    const unsigned bN = __ballot_sync(FULL, mode == MODE_NODE), bL = __ballot_sync(FULL, mode == MODE_LEAF);
    if ((bN | bL) == 0u) break;
    if (__popc(bN) >= RT_NODE_THR || bL == 0u) {
      if (mode == MODE_NODE) mode = node_step<COUNT>(ts, st, ns, cn);
    } else {
      if (mode == MODE_LEAF) mode = leaf_step<COUNT, CALLFREE>(ts, st, sc, media, [&](PathKey& k, uint32_t& b) { k = key, b = bounce; }, cn);
    }
  }
#endif
  return ts.best;
}

// The production traversal as an OUTLINED, CALL-FREE function.  Inlined into a kernel that also calls other
// outlined helpers (Philox, perlin, media), ptxas homes every value that lives across those calls in local memory
// — the node index, 1/d, o/d — and each node step paid 6 LDL + 2 STL for it (profiles/r06_pool_kernel.md).  With its own
// register allocation and no call inside, the node loop touches local memory only for the traversal stack.
// `sc`, `ns` must be addressable from a function: the kernel passes its shared-memory copy of the parameters.
template <bool COUNT>
__device__ __noinline__ Hit closest_hit_outlined(const DeviceScene* __restrict__ sc, const float4* s_nodes, int smem_nodes, float3 o, float3 d, float time,
                                                 uint32_t skip, Hit best, uint2 seed, uint32_t pixel, uint32_t sample, uint32_t bounce, bool active,
                                                 unsigned int* cn) {
  TravState ts;
  trav_set_ray(ts, o, d, time, 0.001f, skip);
  ts.best = best;
  const NodeSource ns = node_source(s_nodes, sc->nodes, smem_nodes);
  const PathKey key{seed, pixel, sample};
  return closest_hit_prepared<COUNT, true>(*sc, ns, ts, sc->n_media != 0, key, bounce, cn, active);
}

// ALL_SMEM: every BVH node is staged in shared memory (true for all the BASELINE scenes): no bounds test, no global path
template <bool COUNT, bool ALL_SMEM = false>
__device__ __forceinline__ Hit closest_hit(const DeviceScene& sc, const NodeSource& ns, float3 o, float3 d, float time, float tmin, float tmax,
                                           uint32_t skip_ref, bool media, const PathKey& key, uint32_t bounce, unsigned int* cn, bool active = true,
                                           const LeafSource& ls = LeafSource{0u, 0u, 0u}) {
  const unsigned FULL = 0xFFFFFFFFu;
  TravState ts;
  TravStack st;
  ts.best = Hit{tmax, REF_NONE};
  ts.cur = kTravDone;
  if (active) trav_begin<COUNT>(ts, sc, o, d, time, tmin, tmax, skip_ref, media, key, bounce, cn);
  trav_reset(ts, st);
#if RT_SPECULATIVE
  int pend = kTravDone;  // the parked leaf, kTravDone = none
  for (;;) {
    while (__any_sync(FULL, ts.cur >= 0)) {
#pragma unroll
      for (int u = 0; u < RT_NODE_UNROLL; u++)
        if (ts.cur >= 0) node_step_spec<COUNT, ALL_SMEM>(ts, st, ns, pend, cn);
    }
    // every lane: cur is a leaf or finished, pend a parked (nearer) leaf or none
    const bool parked = pend != kTravDone;
    const int leaf = parked ? pend : ts.cur;
    if (!__any_sync(FULL, leaf != kTravDone)) break;
    if (leaf != kTravDone) {
      leaf_body<COUNT, false, ALL_SMEM>(ts, leaf, sc, media, [&](PathKey& k, uint32_t& b) { k = key, b = bounce; }, cn, ls);
      const int second = ts.cur;
      pend = kTravDone;
      if (second != kTravDone) {  // a second leaf moves up to the parking slot; the lane walks on from the stack
        if (parked) pend = second;
        trav_pop(ts, st);
      }
    }
  }
#elif RT_NODE_THR == 1
  // classic while-while with the lane's mode read off ts.cur (>= 0: node, kTravDone: finished, else a leaf): the
  // node loop drains to the last lane — one vote per step —, then the leaves are intersected together
  for (;;) {
    while (__any_sync(FULL, ts.cur >= 0)) {
#pragma unroll
      for (int u = 0; u < RT_NODE_UNROLL; u++)  // RT_NODE_UNROLL node steps per vote
        if (ts.cur >= 0) node_step<COUNT, ALL_SMEM>(ts, st, ns, cn);
    }
    if (!__any_sync(FULL, ts.cur != kTravDone)) break;
    if (ts.cur != kTravDone) leaf_step<COUNT, false, ALL_SMEM>(ts, st, sc, media, [&](PathKey& k, uint32_t& b) { k = key, b = bounce; }, cn, ls);
  }
#else
  int mode = active ? MODE_NODE : MODE_DONE;
  for (;;) {
    const unsigned bN = __ballot_sync(FULL, mode == MODE_NODE), bL = __ballot_sync(FULL, mode == MODE_LEAF);
    if ((bN | bL) == 0u) break;
    // node steps while at least RT_NODE_THR lanes want one; below the threshold the lanes waiting on leaves go first
    if (__popc(bN) >= RT_NODE_THR || bL == 0u) {
      if (mode == MODE_NODE) mode = node_step<COUNT, ALL_SMEM>(ts, st, ns, cn);
    } else {
      if (mode == MODE_LEAF) mode = leaf_step<COUNT, false, ALL_SMEM>(ts, st, sc, media, [&](PathKey& k, uint32_t& b) { k = key, b = bounce; }, cn, ls);
    }
  }
#endif
  return ts.best;
}

// closest_hit for a caller that keeps as little as possible in registers across the traversal: `key_of(key, bounce)`
// fetches the ray's Philox counter where a medium needs it — for the scene-enclosing media at the start (every ray of
// such a scene, warp converged), and lazily for a medium leaf — and `aux_of(time, skip)` fetches the ray's time and the
// primitive it starts on, which only the leaves (and the media) look at: the node loop carries neither.
template <bool COUNT, bool ALL_SMEM, typename Stack, typename KeyFn, typename AuxFn>
__device__ __forceinline__ Hit closest_hit_keyfn(const DeviceScene& sc, const NodeSource& ns, float3 o, float3 d, float tmin, float tmax, bool media,
                                                 KeyFn key_of, AuxFn aux_of, unsigned int* cn, bool active, const LeafSource& ls, Stack& st) {
  const unsigned FULL = 0xFFFFFFFFu;
  TravState ts;
  ts.best = Hit{tmax, REF_NONE};
  ts.cur = kTravDone;
  if (active) {
    trav_set_ray(ts, o, d, 0.0f, tmin, REF_NONE);
    if (media && sc.n_global_media) {
      PathKey k;
      uint32_t b, skip;
      float time;
      key_of(k, b);
      aux_of(time, skip);
      ts.best = sample_global_media<COUNT>(sc, o, d, time, tmin, tmax, k, b, cn);
    }
    trav_reset(ts, st);
    ts.cur = 0;
  }
#if RT_KEYFN_NODE_THR > 1
  // node steps while at least RT_KEYFN_NODE_THR lanes want one; below that the lanes waiting on a leaf go first (they
  // come back with fresh node work), and only when no lane sits on a leaf do the stragglers step alone
  for (;;) {
    const unsigned bn = __ballot_sync(FULL, ts.cur >= 0);
    if (__popc(bn) >= RT_KEYFN_NODE_THR) {
#pragma unroll
      for (int u = 0; u < RT_NODE_UNROLL; u++)
        if (ts.cur >= 0) node_step<COUNT, ALL_SMEM>(ts, st, ns, cn);
      continue;
    }
    const unsigned busy = __ballot_sync(FULL, ts.cur != kTravDone);
    if (busy == 0u) break;
    if (busy & ~bn) {
      if (ts.cur < 0 && ts.cur != kTravDone) {
        aux_of(ts.time, ts.skip);
        leaf_step<COUNT, false, ALL_SMEM>(ts, st, sc, media, key_of, cn, ls);
      }
    } else {
      if (ts.cur >= 0) node_step<COUNT, ALL_SMEM>(ts, st, ns, cn);
    }
  }
#else
  for (;;) {
    while (__any_sync(FULL, ts.cur >= 0)) {
#pragma unroll
      for (int u = 0; u < RT_NODE_UNROLL; u++)
        if (ts.cur >= 0) node_step<COUNT, ALL_SMEM>(ts, st, ns, cn);
    }
    if (!__any_sync(FULL, ts.cur != kTravDone)) break;
    if (ts.cur != kTravDone) {
      aux_of(ts.time, ts.skip);
      leaf_step<COUNT, false, ALL_SMEM>(ts, st, sc, media, key_of, cn, ls);
    }
  }
#endif
  return ts.best;
}

// ---------------------------------------------------------------------------------------
// textures (core/texture.hpp, core/perlin.hpp)
__device__ __forceinline__ float perlin_noise(const float4* __restrict__ vec, const uint8_t* __restrict__ perm, float3 p) {
  float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
  float u = p.x - fx, v = p.y - fy, w = p.z - fz;
  int i = int(fx), j = int(fy), k = int(fz);
  float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);
  int px[2] = {perm[i & 255], perm[(i + 1) & 255]};
  int py[2] = {perm[256 + (j & 255)], perm[256 + ((j + 1) & 255)]};
  int pz[2] = {perm[512 + (k & 255)], perm[512 + ((k + 1) & 255)]};
  float accum = 0.0f;
#pragma unroll
  for (int di = 0; di < 2; di++)
#pragma unroll
    for (int dj = 0; dj < 2; dj++)
#pragma unroll
      for (int dk = 0; dk < 2; dk++) {
        float4 g = __ldg(vec + (px[di] ^ py[dj] ^ pz[dk]));
        float wgt = (di ? uu : 1.0f - uu) * (dj ? vv : 1.0f - vv) * (dk ? ww : 1.0f - ww);
        accum = fmaf(wgt, g.x * (u - di) + g.y * (v - dj) + g.z * (w - dk), accum);
      }
  return accum;
}

__device__ RT_OUTLINE float perlin_turb(const float4* __restrict__ vec, const uint8_t* __restrict__ perm, float3 p) {
  float accum = 0.0f, weight = 1.0f;
#pragma unroll 1
  for (int i = 0; i < 7; i++) {  // noise.turb(p, 7), texture.hpp:150
    accum = fmaf(weight, perlin_noise(vec, perm, p), accum);
    weight *= 0.5f;
    p = 2.0f * p;
  }
  return fabsf(accum);
}

#ifndef RT_COOP_NOISE
#define RT_COOP_NOISE 1
#endif
// Will the texture of `material` end in a noise texture at point p?  Returns its table index, or -1.  (The walk of
// texture_value down a checker nesting, without evaluating anything.)
__device__ __forceinline__ int noise_request(const DeviceScene& sc, int material, float3 p) {
  int tex = __float_as_int(__ldg(sc.materials + 2 * material + 1).y);
#pragma unroll 1
  for (int guard = 0; guard < 16 && tex >= 0; guard++) {
    const float4 t0 = __ldg(sc.textures + 2 * tex), t1 = __ldg(sc.textures + 2 * tex + 1);
    const int kind = __float_as_int(t1.x);
    if (kind == TEX_NOISE) return __float_as_int(t1.y);
    if (kind != TEX_CHECKER) return -1;
    const int s = int(floorf(t0.w * p.x)) + int(floorf(t0.w * p.y)) + int(floorf(t0.w * p.z));
    tex = (s & 1) ? __float_as_int(t1.z) : __float_as_int(t1.y);
  }
  return -1;
}
// noise.turb(p, 7) (texture.hpp:150, perlin.hpp) for the lanes with want >= 0, computed by the WHOLE converged warp: up to
// four requesting lanes at a time get eight lanes each, lane k of a group evaluates octave k — perlin_noise(2^k p), the very
// call the serial loop of perlin_turb makes in its k-th iteration (doubling is exact, so 2^k p has the bits of k doublings)
// — and every requester then folds its seven octaves with the serial loop's own fmaf chain: bit-identical to perlin_turb,
// whichever lanes ask together, so the image stays independent of the schedule.  More than four requesters (a scene made of
// marble): every lane evaluates its own point, as before.  Returns the turbulence for requesters, -1 for the others.
__device__ __forceinline__ float coop_noise_turb(const DeviceScene& sc, int want, float3 p, unsigned lane) {
  const unsigned FULL = 0xFFFFFFFFu;
  const unsigned m = __ballot_sync(FULL, want >= 0);
  if (m == 0u) return -1.0f;
  if (__popc(m) > 4) return want >= 0 ? perlin_turb(sc.perlin_vec + 256 * want, sc.perlin_perm + 768 * want, p) : -1.0f;
  const unsigned grp = lane >> 3, k = lane & 7u;
  unsigned mm = m;  // the grp-th requester = the grp-th set bit of m
#pragma unroll
  for (unsigned i = 0; i < 3; i++)
    if (i < grp) mm &= mm - 1u;
  const int src = mm ? __ffs(int(mm)) - 1 : 0;
  const float px = __shfl_sync(FULL, p.x, src), py = __shfl_sync(FULL, p.y, src), pz = __shfl_sync(FULL, p.z, src);
  const int idx = __shfl_sync(FULL, want, src);
  float n = 0.0f;
  if (mm != 0u && k < 7u) {
    const float f = float(1u << k);
    n = perlin_noise(sc.perlin_vec + 256 * idx, sc.perlin_perm + 768 * idx, f3(f * px, f * py, f * pz));
  }
  const unsigned rank = __popc(m & ((1u << lane) - 1u));  // a requester's group = its rank among the requesters
  float accum = 0.0f, weight = 1.0f;
#pragma unroll
  for (int kk = 0; kk < 7; kk++) {
    const float nk = __shfl_sync(FULL, n, int(((rank & 3u) << 3) + unsigned(kk)));
    accum = fmaf(weight, nk, accum);
    weight *= 0.5f;
  }
  return want >= 0 ? fabsf(accum) : -1.0f;
}

// get_sphere_uv (sphere.hpp:100-111) from the OBJECT-space outward normal
__device__ __forceinline__ float2 sphere_uv(float3 n) {
  const float PI = 3.14159265358979323846f;
  float theta = acosf(fminf(fmaxf(-n.y, -1.0f), 1.0f));
  float phi = atan2f(-n.z, n.x) + PI;
  return make_float2(phi * (0.5f / PI), theta * (1.0f / PI));
}

template <bool COUNT>
__device__ __forceinline__ float3 texture_value(const DeviceScene& sc, int tex, float u, float v, float3 p, unsigned int* cn, float turb_pre = -1.0f) {
#pragma unroll 1
  for (int guard = 0; guard < 16; guard++) {
    RT_CHECK(tex >= 0 && tex < sc.n_textures, CHK_TEXTURE);
    float4 t0 = __ldg(sc.textures + 2 * tex), t1 = __ldg(sc.textures + 2 * tex + 1);
    int kind = __float_as_int(t1.x), a = __float_as_int(t1.y), b = __float_as_int(t1.z);
    if (kind == TEX_SOLID) return xyz(t0);
    if (kind == TEX_CHECKER) {  // texture.hpp:57-79 ; (sum % 2 == 0) == ((sum & 1) == 0) for negatives too
      int s = int(floorf(t0.w * p.x)) + int(floorf(t0.w * p.y)) + int(floorf(t0.w * p.z));
      tex = (s & 1) ? b : a;
      if (COUNT) cn[CN_TEX_CHECKER]++;
      continue;
    }
    if (kind == TEX_IMAGE) {  // texture.hpp:97-118 + rtw_stb_image.hpp:104-134
      int4 im = __ldg(sc.images + a);
      if (COUNT) cn[CN_TEX_IMAGE]++;
      if (im.z <= 0) return f3(0.0f, 1.0f, 1.0f);
      u = fminf(fmaxf(u, 0.0f), 1.0f);
      v = 1.0f - fminf(fmaxf(v, 0.0f), 1.0f);
      int i = min(int(u * im.y), im.y - 1);
      int j = min(int(v * im.z), im.z - 1);
      RT_CHECK(i >= 0 && j >= 0 && i < im.y && j < im.z, CHK_TEXEL);
      uchar4 px = __ldg(sc.texels + im.x + j * im.y + i);
      const float s = 1.0f / 255.0f;
      return f3(s * px.x, s * px.y, s * px.z);
    }
    // TEX_NOISE: marble, texture.hpp:150
    if (COUNT) cn[CN_TEX_NOISE]++;
    // (turb_pre >= 0: this lane's turbulence was already evaluated by coop_noise_turb — same point, same bits)
    float turb = turb_pre >= 0.0f ? turb_pre : perlin_turb(sc.perlin_vec + 256 * a, sc.perlin_perm + 768 * a, p);
    float g = 0.5f * (1.0f + sinf(fmaf(t0.w, p.z, 10.0f * turb)));
    return f3(g, g, g);
  }
  return f3(0.0f, 0.0f, 0.0f);
}

// ---------------------------------------------------------------------------------------
// surface reconstruction at the hit + material::emitted / material::scatter
struct Surface {
  float3 p, n;  // n already flipped against the ray (hit_record::set_face_normal)
  float u, v;
  float t;      // the hit's ray parameter; with RT_SPHERE_REFINE a sphere root re-solved in fp64
  bool front;
  int material;
};

#ifndef RT_SPHERE_REFINE
#define RT_SPHERE_REFINE 2  // 0: fp32 roots as found; 1: fp64 quadratic; 2: one fp64-residual Newton step (default: t within 1e-5 of the
                            // reference on all but <= 3 pixels per scene instead of on 87-99 % of them, for -1 % on book2_final,
                            // gpurun_out/ab_refine3.log, profiles/r2_primary_parity.md)
#endif
// The root of |o + t d - c|^2 = r^2 nearest to the fp32 root `t32`, solved in fp64 from the same fp32 ray and sphere.
// fp32 cannot resolve the root on a radius-1000 sphere better than ~5e-5 relative (6e-5 of absolute resolution on a
// coordinate of 1000, amplified by the cancellation in tca - sqrt(r^2 - l^2)); profiles/r2_primary_parity.md.  Once per
// SHADED sphere hit (not per candidate): ~45 fp64 instructions.
// RT_SPHERE_REFINE == 2: one Newton step on f(t) = a t^2 + 2 b t + cc from the fp32 root, with f evaluated in fp64 (the
// residual is what fp32 cannot see) and the division in fp32 (the correction is ~1e-5 t: seven digits of it are plenty).
// No fp64 square root or division: ~25 fp64 instructions.  A correction beyond 1e-3 |t| (grazing hit, f' ~ 0) is dropped.
// Also returns p - c = (o - c) + t d evaluated in fp64: its magnitude is r, not |p|, so the normal (p - c) / r keeps seven
// digits even for a small sphere far from the origin.
__device__ __forceinline__ float sphere_root_newton(float3 c32, float r32, float3 o, float3 d, float t32, float3& p_minus_c) {
  const double ocx = double(o.x) - double(c32.x), ocy = double(o.y) - double(c32.y), ocz = double(o.z) - double(c32.z);
  const double dx = d.x, dy = d.y, dz = d.z, r = r32, t = t32;
  const double a = dx * dx + dy * dy + dz * dz, b = ocx * dx + ocy * dy + ocz * dz, cc = ocx * ocx + ocy * ocy + ocz * ocz - r * r;
  const double at_b = a * t + b;
  const float f = float((at_b + b) * t + cc), fp = float(2.0 * at_b);
  const float delta = f * rcp_fast(fp);
  const float t_new = fabsf(delta) <= 1e-3f * fabsf(t32) ? t32 - delta : t32;
  const double tn = t_new;
  p_minus_c = f3(float(ocx + tn * dx), float(ocy + tn * dy), float(ocz + tn * dz));
  return t_new;
}
__device__ __forceinline__ float sphere_root_fp64(float3 c32, float r32, float3 o, float3 d, float t32) {
  const double cx = c32.x, cy = c32.y, cz = c32.z, r = r32;
  const double ocx = double(o.x) - cx, ocy = double(o.y) - cy, ocz = double(o.z) - cz;
  const double dx = d.x, dy = d.y, dz = d.z;
  const double a = dx * dx + dy * dy + dz * dz, b = ocx * dx + ocy * dy + ocz * dz, cc = ocx * ocx + ocy * ocy + ocz * ocz - r * r;
  const double disc = b * b - a * cc;
  if (!(disc >= 0.0)) return t32;  // fp32 saw a grazing hit that fp64 does not: keep it
  const double sq = sqrt(disc);
  // both roots without cancellation: q = -(b + sign(b) sqrt(disc)), roots q / a and cc / q
  const double q = -(b + (b < 0.0 ? -sq : sq));
  const double r0 = q / a, r1 = q != 0.0 ? cc / q : r0;
  return float(fabs(r0 - double(t32)) <= fabs(r1 - double(t32)) ? r0 : r1);
}

__device__ __forceinline__ Surface surface_at(const DeviceScene& sc, Hit h, float3 o, float3 d, float time) {
  Surface s;
  uint32_t type = h.ref >> 30, idx = h.ref & 0x3FFFFFFFu;
  s.p = fma3(h.t, d, o);
  s.t = h.t;
  s.u = s.v = 0.0f;
  RT_CHECK(type != REF_SPHERE || idx < uint32_t(sc.n_spheres), CHK_SPHERE);
  RT_CHECK(type != REF_QUAD || idx < uint32_t(sc.n_quads), CHK_QUAD);
  RT_CHECK(type != REF_BOX || (idx >> 3) < uint32_t(sc.n_boxes), CHK_BOX);
  RT_CHECK(type != REF_MEDIUM || idx < uint32_t(sc.n_media), CHK_MEDIUM);
  if (type == REF_SPHERE) {
    float4 g0 = __ldg(sc.spheres + 2 * idx), g1 = __ldg(sc.spheres + 2 * idx + 1);
    int2 meta = __ldg(sc.sph_meta + idx);
    float3 c = fma3(time, xyz(g1), xyz(g0));
#if RT_SPHERE_REFINE == 2
    float3 pc;
    s.t = sphere_root_newton(c, g0.w, o, d, h.t, pc);
    float3 outward = rcp_fast(g0.w) * pc;
#elif RT_SPHERE_REFINE
    s.t = sphere_root_fp64(c, g0.w, o, d, h.t);
    s.p = fma3(s.t, d, o);
    float3 outward = rcp_fast(g0.w) * (s.p - c);
#else
    float3 outward = rcp_fast(g0.w) * (s.p - c);
#endif
    s.p = fma3(g0.w, outward, c);  // re-project onto the sphere: removes the O(t*eps) drift of o + t d
    s.material = meta.x;
    float4 m1 = __ldg(sc.materials + 2 * meta.x + 1);
    if (__float_as_int(m1.z) & MATF_NEEDS_UV) {
      float3 no = outward;
      if (meta.y >= 0) {  // back to the instance's object space (inverse y-rotation)
        float2 r = __ldg(sc.rotations + meta.y);
        no = f3(r.y * outward.x - r.x * outward.z, outward.y, r.x * outward.x + r.y * outward.z);
      }
      float2 uv = sphere_uv(no);
      s.u = uv.x, s.v = uv.y;
    }
    s.front = dot(d, outward) < 0.0f;
    s.n = s.front ? outward : -outward;
  } else if (type == REF_QUAD) {
    float4 nD = __ldg(sc.quads + 3 * idx);
    s.material = __ldg(sc.quad_mat + idx);
    float4 m1 = __ldg(sc.materials + 2 * s.material + 1);
    if (__float_as_int(m1.z) & MATF_NEEDS_UV) {
      float4 A = __ldg(sc.quads + 3 * idx + 1), B = __ldg(sc.quads + 3 * idx + 2);
      s.u = dot(xyz(A), s.p) + A.w;
      s.v = dot(xyz(B), s.p) + B.w;
    }
    s.front = dot(d, xyz(nD)) < 0.0f;
    s.n = s.front ? xyz(nD) : -xyz(nD);
  } else if (type == REF_BOX) {
    const uint32_t b = idx >> 3, face = idx & 7u;
    const float4 b0 = __ldg(sc.boxes + 3 * b), b1 = __ldg(sc.boxes + 3 * b + 1), b2 = __ldg(sc.boxes + 3 * b + 2);
    const int4 meta = __ldg(sc.box_meta + b);
    const uint32_t fm = (uint32_t(meta.z) >> (4u * face)) & 15u;
    const float sgn = ((face & 1u) != 0u) != ((fm & 8u) != 0u) ? 1.0f : -1.0f;  // the QUAD's normal: outward unless flagged
    float3 n = f3((face >> 1) == 0u ? sgn : 0.0f, (face >> 1) == 1u ? sgn : 0.0f, (face >> 1) == 2u ? sgn : 0.0f);
    if (b2.w != 0.0f) n = f3(b0.w * n.x + b1.w * n.z, n.y, -b1.w * n.x + b0.w * n.z);  // back to world (rotate_y)
    s.material = meta.x;
    float4 m1 = __ldg(sc.materials + 2 * s.material + 1);
    if (__float_as_int(m1.z) & MATF_NEEDS_UV) {
      const int qi = meta.y + int(fm & 7u);
      float4 A = __ldg(sc.quads + 3 * qi + 1), B = __ldg(sc.quads + 3 * qi + 2);
      s.u = dot(xyz(A), s.p) + A.w;
      s.v = dot(xyz(B), s.p) + B.w;
    }
    s.front = dot(d, n) < 0.0f;
    s.n = s.front ? n : -n;
  } else {  // medium: arbitrary normal, front face (SURVEY B.2)
    s.material = sc.media[idx].material;
    s.n = f3(1.0f, 0.0f, 0.0f);
    s.front = true;
  }
  return s;
}

// returns true when the path continues along (o, d); `emit` is material::emitted.
template <bool COUNT>
__device__ __forceinline__ bool scatter_ray(const DeviceScene& sc, const Surface& s, float3 d_in, uint4 rnd, float3& emit, float3& atten, float3& d_out,
                                            unsigned int* cn, float turb_pre = -1.0f) {
  RT_CHECK(s.material >= 0 && s.material < sc.n_materials, CHK_MATERIAL);
  float4 m0 = __ldg(sc.materials + 2 * s.material), m1 = __ldg(sc.materials + 2 * s.material + 1);
  const int kind = __float_as_int(m1.x), tex = __float_as_int(m1.y);
  emit = f3(0.0f, 0.0f, 0.0f);
  if (COUNT) cn[CN_LAMB + (kind - MAT_LAMBERTIAN)]++;
  // one texture call site and one unit-vector site for all materials (code size: see RT_OUTLINE)
  float3 tv = f3(1.0f, 1.0f, 1.0f);
  if (tex >= 0) tv = texture_value<COUNT>(sc, tex, s.u, s.v, s.p, cn, turb_pre);
  const float3 rv = unit_vector_from(u01(rnd.x), u01(rnd.y));
  switch (kind) {
    case MAT_LAMBERTIAN: {  // material.hpp:51-71
      float3 dir = s.n + rv;
      if (fabsf(dir.x) < 1e-8f && fabsf(dir.y) < 1e-8f && fabsf(dir.z) < 1e-8f) dir = s.n;
      d_out = dir;
      atten = tv;
      return true;
    }
    case MAT_METAL: {  // material.hpp:86-106
      float3 refl = fma3(-2.0f * dot(d_in, s.n), s.n, d_in);
      d_out = fma3(m0.w, rv, normalize3(refl));
      atten = xyz(m0);
      return dot(d_out, s.n) > 0.0f;
    }
    case MAT_DIELECTRIC: {  // material.hpp:128-206
      atten = f3(1.0f, 1.0f, 1.0f);
      float ri = s.front ? rcp_fast(m0.w) : m0.w;
      float3 ud = normalize3(d_in);
      float cos_t = fminf(-dot(ud, s.n), 1.0f);
      float sin_t = sqrtf(fmaxf(0.0f, 1.0f - cos_t * cos_t));
      bool reflect = ri * sin_t > 1.0f;
      if (!reflect) {
        float r0 = (1.0f - ri) / (1.0f + ri);
        r0 *= r0;
        float x = 1.0f - cos_t, x2 = x * x;
        reflect = fmaf(1.0f - r0, x2 * x2 * x, r0) > u01(rnd.z);
      }
      if (reflect) {
        d_out = fma3(-2.0f * dot(ud, s.n), s.n, ud);
      } else {  // refract, vec3.hpp:216-226
        float3 perp = ri * fma3(cos_t, s.n, ud);
        float par = -sqrtf(fabsf(1.0f - dot(perp, perp)));
        d_out = fma3(par, s.n, perp);
      }
      return true;
    }
    case MAT_LIGHT:  // material.hpp:223-240: emits on both faces, never scatters
      emit = tv;
      return false;
    default:  // MAT_ISOTROPIC, SURVEY B.3
      d_out = rv;
      atten = tv;
      return true;
  }
}

// ---------------------------------------------------------------------------------------
// fp64 exact predicates: every operation is an explicit IEEE round-to-nearest intrinsic, so
// nvcc cannot contract a*b+c into an FMA and the results round exactly like the reference
// built by g++ for x86-64 (which has no FMA at the baseline ISA).
struct sd {
  double v;
};
__device__ __forceinline__ sd S(double v) { return sd{v}; }
__device__ __forceinline__ sd operator+(sd a, sd b) { return sd{__dadd_rn(a.v, b.v)}; }
__device__ __forceinline__ sd operator-(sd a, sd b) { return sd{__dsub_rn(a.v, b.v)}; }
__device__ __forceinline__ sd operator*(sd a, sd b) { return sd{__dmul_rn(a.v, b.v)}; }
__device__ __forceinline__ sd operator/(sd a, sd b) { return sd{__ddiv_rn(a.v, b.v)}; }
__device__ __forceinline__ sd operator-(sd a) { return sd{-a.v}; }
struct sv {
  sd x, y, z;
};
__device__ __forceinline__ sv SV(const double* p) { return sv{S(p[0]), S(p[1]), S(p[2])}; }
__device__ __forceinline__ sv operator+(sv a, sv b) { return sv{a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ sv operator-(sv a, sv b) { return sv{a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ sv operator-(sv a) { return sv{-a.x, -a.y, -a.z}; }
__device__ __forceinline__ sv operator*(sd t, sv v) { return sv{t * v.x, t * v.y, t * v.z}; }
__device__ __forceinline__ sd sdot(sv a, sv b) { return a.x * b.x + a.y * b.y + a.z * b.z; }  // vec3.hpp:138-141, left to right
__device__ __forceinline__ sv scross(sv a, sv b) { return sv{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

struct XRay {
  sv o, d;
  sd tm;
};
struct XRec {
  sd t;
  sv n;
  bool front;
};

// translate::hit / rotate_y::hit ray transforms, outermost wrapper first
__device__ __forceinline__ XRay exact_to_object(const DeviceScene& sc, int chain, XRay r) {
  int2 ch = sc.xchains[chain];
  for (int k = 0; k < ch.y; k++) {
    const XOp& op = sc.xops[ch.x + k];
    if (op.kind == 0) {  // hittable.hpp:89
      r.o = r.o - SV(op.a);
    } else {  // SURVEY B.1
      sd s = S(op.a[0]), c = S(op.a[1]);
      r.o = sv{(c * r.o.x) - (s * r.o.z), r.o.y, (s * r.o.x) + (c * r.o.z)};
      r.d = sv{(c * r.d.x) - (s * r.d.z), r.d.y, (s * r.d.x) + (c * r.d.z)};
    }
  }
  return r;
}
// ... and rec.normal back to world space, innermost wrapper first (translate leaves it alone)
__device__ __forceinline__ sv exact_normal_to_world(const DeviceScene& sc, int chain, sv n) {
  int2 ch = sc.xchains[chain];
  for (int k = ch.y - 1; k >= 0; k--) {
    const XOp& op = sc.xops[ch.x + k];
    if (op.kind == 1) {
      sd s = S(op.a[0]), c = S(op.a[1]);
      n = sv{(c * n.x) + (s * n.z), n.y, (-s * n.x) + (c * n.z)};
    }
  }
  return n;
}

// sphere::hit, sphere.hpp:47-93, operation for operation
__device__ __forceinline__ bool exact_sphere(const DeviceScene& sc, const XSphere& q, const XRay& rw, double tmin, double tmax, XRec& rec) {
  XRay r = exact_to_object(sc, q.chain, rw);
  sv cc = SV(q.c) + r.tm * SV(q.dc);  // center.at(r.time())
  sv oc = r.o - cc;
  sd a = sdot(r.d, r.d);
  sd half_b = sdot(oc, r.d);
  sd c = sdot(oc, oc) - S(q.r) * S(q.r);
  sd disc = half_b * half_b - a * c;
  if (disc.v < 0) return false;
  sd sq = S(__dsqrt_rn(disc.v));
  sd root = (-half_b - sq) / a;
  if (!(tmin < root.v && root.v < tmax)) {
    root = (-half_b + sq) / a;
    if (!(tmin < root.v && root.v < tmax)) return false;
  }
  rec.t = root;
  sv p = r.o + root * r.d;
  sv outward = (S(1.0) / S(q.r)) * (p - cc);
  rec.front = sdot(r.d, outward).v < 0;
  sv n = rec.front ? outward : -outward;
  rec.n = exact_normal_to_world(sc, q.chain, n);
  return true;
}

// quad::hit + is_interior, quad.hpp:44-114
__device__ __forceinline__ bool exact_quad(const DeviceScene& sc, const XQuad& q, const XRay& rw, double tmin, double tmax, XRec& rec) {
  XRay r = exact_to_object(sc, q.chain, rw);
  sv normal = SV(q.n);
  sd denom = sdot(normal, r.d);
  if (fabs(denom.v) < 1e-8) return false;
  sd t = (S(q.D) - sdot(normal, r.o)) / denom;
  if (!(tmin <= t.v && t.v <= tmax)) return false;
  sv ip = r.o + t * r.d;
  sv hp = ip - SV(q.Q);
  sd alpha = sdot(SV(q.w), scross(hp, SV(q.v)));
  sd beta = sdot(SV(q.w), scross(SV(q.u), hp));
  if (!(0.0 <= alpha.v && alpha.v <= 1.0) || !(0.0 <= beta.v && beta.v <= 1.0)) return false;
  rec.t = t;
  rec.front = sdot(r.d, normal).v < 0;
  sv n = rec.front ? normal : -normal;
  rec.n = exact_normal_to_world(sc, q.chain, n);
  return true;
}

}  // namespace rtb200
