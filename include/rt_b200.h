/*
 * rt_b200.h — the C-ABI drop-in boundary of the B200 path tracer.
 *
 * The reference (jooo0922/raytracing-practice) has no FFI: its "API" is the set of
 * C++ classes that src/main.cpp constructs and the single hot entry point
 *     void camera::render(std::ostream&, const hittable& world)   (src/core/camera.hpp:29-72)
 * Our host-side mirror of those classes (raytracing-practice_b200/host/) only records
 * parameters; camera::render flattens the shared_ptr graph into the POD arrays below
 * and drives the functions declared here.  Nothing in these signatures is a torch or a
 * C++ type: plain pointers, sizes and ints, so a cgo / JNI / ctypes binding is
 * mechanical (see INTEGRATION.md).
 *
 * Every struct mirrors a reference type; the reference file:line is cited next to it.
 * All scene parameters cross the boundary as DOUBLE (the reference's arithmetic type:
 * src/common/vec3.hpp:11); the library narrows to fp32 device layouts itself and keeps
 * the doubles for the exact (fp64) primary-visibility predicate.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 1

/* ---- error codes (the reference's render path returns void; we return 0 or <0) ---- */
enum {
  RT_OK = 0,
  RT_ERR_INVALID = -1,     /* bad argument / malformed scene description            */
  RT_ERR_CUDA = -2,        /* a CUDA runtime call failed (see rt_last_error)        */
  RT_ERR_NO_SCENE = -3,    /* rt_render / rt_trace_rays before rt_upload_scene      */
  RT_ERR_UNSUPPORTED = -4, /* unknown hittable / material / texture kind            */
  RT_ERR_NO_DEVICE = -5    /* no CUDA device: there is NO CPU fallback              */
};

/* ---- hittable graph -------------------------------------------------------------- */
/* One record per node of the reference's shared_ptr<hittable> graph, in the order the
 * flattener first reaches it (DFS, list order, BVH left before right; shared nodes are
 * emitted once).  Leaf primitives (sphere, quad) additionally get a dense "primitive
 * id" = their rank in that same DFS — the id the primary-visibility parity test uses
 * (SURVEY.md §8(c)).                                                                 */
enum rt_hittable_kind {
  RT_H_SPHERE = 1,    /* src/hittable/sphere.hpp:7-119                               */
  RT_H_QUAD = 2,      /* src/hittable/quad.hpp:8-126                                 */
  RT_H_LIST = 3,      /* src/hittable/hittable_list.hpp:21-76                        */
  RT_H_BVH = 4,       /* src/accelerator/bvh_node.hpp:16-134                         */
  RT_H_TRANSLATE = 5, /* src/hittable/hittable.hpp:74-117                            */
  RT_H_ROTATE_Y = 6,  /* not in the reference; book semantics, SURVEY.md App. B.1    */
  RT_H_MEDIUM = 7     /* constant_medium; not in the reference; SURVEY.md App. B.2   */
};

typedef struct rt_hittable {
  int32_t kind;     /* rt_hittable_kind                                               */
  int32_t material; /* SPHERE/QUAD: material index. MEDIUM: phase-function material   */
  int32_t child0;   /* BVH: left. TRANSLATE/ROTATE_Y: object. MEDIUM: boundary.
                       LIST: first slot in rt_scene_desc.child_index                  */
  int32_t child1;   /* BVH: right (== left for a span-1 node, bvh_node.hpp:57).
                       LIST: number of children                                       */
  int32_t prim_id;  /* SPHERE/QUAD: dense DFS leaf id; otherwise -1                   */
  int32_t reserved;
  /* SPHERE   : p[0..2] = center.origin (center1), p[3..5] = center.direction
   *            (center2-center1, zero when static), p[6] = radius   (sphere.hpp:16-44)
   * QUAD     : p[0..2] = Q, p[3..5] = u, p[6..8] = v                 (quad.hpp:12-27)
   * TRANSLATE: p[0..2] = offset                                  (hittable.hpp:77-84)
   * ROTATE_Y : p[0] = angle in degrees, p[1] = sin_theta, p[2] = cos_theta
   * MEDIUM   : p[0] = density, p[1] = neg_inv_density = -1/density                  */
  double p[9];
  /* bounding_box() exactly as the reference computes it (padding rules of
   * src/accelerator/aabb.hpp:22-48,135-154): x.min,x.max,y.min,y.max,z.min,z.max    */
  double bbox[6];
} rt_hittable;

/* ---- materials (src/core/material.hpp) -------------------------------------------- */
enum rt_material_kind {
  RT_M_LAMBERTIAN = 1,    /* material.hpp:42-75                                       */
  RT_M_METAL = 2,         /* material.hpp:80-111                                      */
  RT_M_DIELECTRIC = 3,    /* material.hpp:122-207                                     */
  RT_M_DIFFUSE_LIGHT = 4, /* material.hpp:223-240                                     */
  RT_M_ISOTROPIC = 5      /* not in the reference; SURVEY.md App. B.3                 */
};

typedef struct rt_material {
  int32_t kind;    /* rt_material_kind                                                */
  int32_t texture; /* LAMBERTIAN / DIFFUSE_LIGHT / ISOTROPIC: texture index; else -1  */
  double albedo[3]; /* METAL                                                          */
  double fuzz;      /* METAL, already clamped to <= 1 (material.hpp:83)               */
  double ior;       /* DIELECTRIC refraction_index                                    */
} rt_material;

/* ---- textures (src/core/texture.hpp) ----------------------------------------------- */
enum rt_texture_kind {
  RT_T_SOLID = 1,   /* texture.hpp:25-41                                              */
  RT_T_CHECKER = 2, /* texture.hpp:47-85                                              */
  RT_T_IMAGE = 3,   /* texture.hpp:91-122                                             */
  RT_T_NOISE = 4    /* texture.hpp:127-156                                            */
};

typedef struct rt_texture {
  int32_t kind;   /* rt_texture_kind                                                  */
  int32_t even;   /* CHECKER: texture index of the even cell                          */
  int32_t odd;    /* CHECKER: texture index of the odd cell                           */
  int32_t image;  /* IMAGE: index into images (its width may be 0 = failed load)      */
  int32_t perlin; /* NOISE: index into perlins                                        */
  int32_t reserved;
  double color[3]; /* SOLID albedo                                                    */
  double scale;    /* CHECKER: inv_scale (= 1.0f/scale, texture.hpp:51); NOISE: scale */
} rt_texture;

/* rtw_image after convert_to_bytes (src/core/rtw_stb_image.hpp:154-169): tightly packed
 * RGB8, row-major from the top.  width == 0 / rgb == NULL is a failed load (cyan in
 * image_texture::value, texture.hpp:100-103).                                         */
typedef struct rt_image {
  int32_t width;
  int32_t height;
  const uint8_t* rgb;
} rt_image;

/* perlin tables (src/core/perlin.hpp:257-265), one set per noise_texture instance.    */
typedef struct rt_perlin {
  double randvec[256][3];
  int32_t perm_x[256];
  int32_t perm_y[256];
  int32_t perm_z[256];
} rt_perlin;

typedef struct rt_scene_desc {
  int32_t abi_version; /* RT_B200_ABI_VERSION                                         */
  int32_t root;        /* index of the world hittable passed to camera::render        */
  int32_t n_hittables;
  int32_t n_child_index;
  int32_t n_materials;
  int32_t n_textures;
  int32_t n_images;
  int32_t n_perlins;
  int32_t n_prims; /* number of SPHERE/QUAD leaves = 1 + max prim_id                  */
  int32_t reserved;
  const rt_hittable* hittables;
  const int32_t* child_index; /* LIST children, hittable indices, in insertion order  */
  const rt_material* materials;
  const rt_texture* textures;
  const rt_image* images;
  const rt_perlin* perlins;
} rt_scene_desc;

/* ---- camera: the public fields of src/core/camera.hpp:13-25 ------------------------ */
typedef struct rt_camera_desc {
  double aspect_ratio;
  int32_t image_width;
  int32_t samples_per_pixel;
  int32_t max_depth;
  int32_t reserved;
  double background[3];
  double vfov;
  double lookfrom[3];
  double lookat[3];
  double vup[3];
  double defocus_angle;
  double focus_dist;
} rt_camera_desc;

/* What camera::initialize derives (src/core/camera.hpp:76-136), in double.            */
typedef struct rt_camera_frame {
  int32_t image_width;
  int32_t image_height;
  double pixel_samples_scale;
  double center[3];
  double pixel00_loc[3];
  double pixel_delta_u[3];
  double pixel_delta_v[3];
  double u[3], v[3], w[3];
  double defocus_disk_u[3];
  double defocus_disk_v[3];
} rt_camera_frame;

/* Pure host arithmetic, double, same operation order as camera::initialize.           */
int rt_camera_initialize(const rt_camera_desc* cam, rt_camera_frame* out);

/* ---- context ----------------------------------------------------------------------- */
typedef struct rt_ctx rt_ctx;

/* One context = one CUDA device = one rank.  Fails with RT_ERR_NO_DEVICE when there is
 * no GPU: there is no CPU fallback anywhere in this library.                           */
int rt_init(int device, rt_ctx** out);
void rt_shutdown(rt_ctx* ctx);
const char* rt_last_error(rt_ctx* ctx); /* ctx may be NULL: last error of rt_init      */

/* Copies everything it needs; the caller keeps ownership of the description.  Builds
 * the device scene: instance transforms baked into world-space primitives, SAH BVH,
 * material / texture tables, RGBA8 texels, perlin tables.                              */
int rt_upload_scene(rt_ctx* ctx, const rt_scene_desc* scene);

/* ---- render: the hot path (camera::render's pixel x sample loop) ------------------- */
typedef struct rt_render_opts {
  uint64_t seed;        /* Philox key                                                  */
  int32_t sample_begin; /* this rank renders sample indices [begin, begin+count) of    */
  int32_t sample_count; /*   every pixel; count <= 0 means all of samples_per_pixel    */
  int32_t clear;        /* non-zero: zero the accumulator before rendering             */
  int32_t flags;        /* RT_RENDER_* bits                                            */
  void* peer_accum;     /* optional: the accumulator (rt_accum_device_ptr) of ANOTHER LIVE CONTEXT OF
                           THIS PROCESS ON THE SAME DEVICE, for a camera of the same image size; when
                           non-NULL the kernel adds its samples THERE (device-scope red.add.u64)
                           instead of locally.  Anything else is refused: RT_ERR_INVALID for an
                           unknown pointer or another image size, RT_ERR_UNSUPPORTED for another
                           GPU's accumulator (device-scope adds are not atomic across GPUs — use
                           push_accum there)                                              */
  void* push_accum;     /* optional: a reduce buffer (rt_reduce_buffer of this or another
                           rank, peer-mapped over NVLink): the render accumulates
                           locally and a push kernel, stream-ordered right behind it,
                           ADDS the whole accumulator into that buffer (system-scope
                           red.add.u64) — the multi-GPU reduce without a collective    */
} rt_render_opts;

enum {
  RT_RENDER_DEFAULT = 0,
  RT_RENDER_COUNTERS = 1,  /* instrumented kernel: also fills rt_stats.census (slower; not for timing) */
  RT_RENDER_MEGAKERNEL = 2, /* force the one-path-per-lane megakernel (render_kernel)               */
  /* 4: was RT_RENDER_POOL, the per-warp path-pool kernel (removed: 0.55-0.65x the megakernel; rt_render answers
        RT_ERR_UNSUPPORTED to the bit).  With no kernel bit the library's default renders (the megakernel; the
        process environment RT_B200_KERNEL=mega|stream|refill, read once at rt_init, can move the default) */
  RT_RENDER_STREAM = 8,     /* force the streaming kernel (stream_kernel: CTA-wide ray queues, lanes refilled
                               mid-traversal); RT_ERR_UNSUPPORTED when the scene does not fit its
                               shared-memory plan                                                   */
  RT_RENDER_REFILL = 16     /* force the in-place-refill kernel (refill_kernel: a lane keeps its path, the warp
                               leaves the traversal to shade as soon as enough lanes have their answer)  */
};

/* Asynchronous on the context's stream.  Accumulates fixed-point (2^-32) int64 RGB
 * sums per pixel: integer addition is associative, so the image is bit-identical for
 * any sharding of the samples over ranks / GPUs / launches.                            */
int rt_render(rt_ctx* ctx, const rt_camera_desc* cam, const rt_render_opts* opts);

/* n_views camera views of the uploaded scene in ONE launch: a turntable, the frames of an
 * animation, a multi-view dataset.  View v of the accumulator gets exactly the bits
 * rt_render(&cams[v], opts) gives (same Philox stream: the counter is the in-view pixel,
 * sample and bounce).  The accumulator becomes n_views x H x W x 3 int64, view-major;
 * rt_download and rt_accum_device_ptr return the whole batch, and rt_stats.n_views says
 * how many images it holds.  A later rt_render / rt_upload_accum makes it one image again.
 *   - Every camera has the same image_width, image height (as rt_camera_initialize
 *     computes it) and samples_per_pixel; every other field (lookfrom / lookat / vup,
 *     vfov, defocus, max_depth, background) may differ per view.  A view with
 *     max_depth <= 0 traces nothing, as rt_render; its samples still count in stats.
 *   - opts: seed, sample_begin / sample_count and clear mean what they mean for rt_render;
 *     one seed serves all views.  Always the megakernel (RT_B200_KERNEL does not apply).
 *   - RT_ERR_INVALID: n_views < 1, NULL cams / opts, a camera rt_render refuses, views of
 *     different sizes or spp, an empty sample range, n_views x W x H > INT32_MAX.
 *     RT_ERR_UNSUPPORTED: peer_accum, push_accum, RT_RENDER_COUNTERS, RT_RENDER_STREAM,
 *     RT_RENDER_REFILL (across GPUs, shard a batch by views).  RT_ERR_NO_SCENE.
 * Asynchronous like rt_render; more than 2^32 work items are split over sample ranges. */
int rt_render_views(rt_ctx* ctx, int32_t n_views, const rt_camera_desc* cams, const rt_render_opts* opts);
int rt_synchronize(rt_ctx* ctx);

/* The accumulator (3 x int64 per pixel, row-major from the top-left, interleaved RGB;
 * after rt_render_views, one such image per view, view-major)
 * as a raw device pointer, for the multi-GPU reduce (NCCL ncclInt64 sum, or peer adds). */
int rt_accum_device_ptr(rt_ctx* ctx, void** dev_ptr, size_t* bytes);

/* ---- peer-memory multi-GPU reduce (the exchange step of camera.hpp:61,65 without a collective call) ----
 * Rank 0 allocates a zeroed reduce buffer (same layout as the accumulator) and exports it; the other
 * ranks (processes) open it through CUDA IPC / peer access; every rank renders its sample shard with
 * rt_render_opts.push_accum pointing at it; after a barrier rank 0 adopts the buffer as its image.   */
typedef struct rt_ipc_handle {
  unsigned char bytes[64]; /* cudaIpcMemHandle_t */
} rt_ipc_handle;
int rt_reduce_buffer(rt_ctx* ctx, const rt_camera_desc* cam, void** dev_ptr, rt_ipc_handle* handle /* may be NULL */);
int rt_peer_open(rt_ctx* ctx, const rt_ipc_handle* handle, void** dev_ptr);
/* Same process, several devices (the C++ host's RT_B200_DEVICES path): lets ctx's device address `owner`'s
 * memory directly (cudaDeviceEnablePeerAccess); a no-op when both contexts sit on the same device.      */
int rt_peer_enable(rt_ctx* ctx, rt_ctx* owner);
int rt_peer_close(rt_ctx* ctx, void* dev_ptr);
/* Copies the reduce buffer over the context's accumulator (rt_download / rt_accum_device_ptr then read the
 * reduced image).  The buffer and its handle stay valid: rt_reduce_buffer with the same camera re-zeroes it. */
int rt_adopt_reduce_buffer(rt_ctx* ctx);

typedef enum rt_buffer_kind {
  RT_BUF_ACCUM_I64 = 0,    /* raw fixed-point sums, 3 x int64 per pixel                */
  RT_BUF_RADIANCE_F32 = 1, /* sums * 2^-32 * pixel_samples_scale, 3 x float per pixel  */
  RT_BUF_RGB8 = 2          /* write_color's gamma/clamp/int(256x) (color.hpp:26-58),
                              3 x uint8 per pixel, computed on the device              */
} rt_buffer_kind;

/* Synchronises and copies the image to host memory.  samples_per_pixel is the total
 * number of samples accumulated (over all ranks) and only scales F32 / RGB8 output.
 * After rt_render_views every kind holds the whole batch, view-major (n_views images). */
int rt_download(rt_ctx* ctx, rt_buffer_kind kind, int32_t samples_per_pixel, void* dst,
                size_t bytes);

/* The inverse of rt_download(RT_BUF_ACCUM_I64): replaces the context's accumulator with image_width x image_height x 3
 * int64 sums from host memory (bytes must be exactly that), e.g. the sums a checkpoint saved.  A following
 * rt_render with clear == 0 and the next sample_begin continues the render; because the sums are integers the
 * finished image has the bits of an uninterrupted one (camera.hpp:55-61 is a plain sum over samples).            */
int rt_upload_accum(rt_ctx* ctx, const rt_camera_desc* cam, const void* src, size_t bytes);

typedef struct rt_stats {
  uint64_t rays;        /* closest-hit queries issued by the integrator since the last
                           clear (= world.hit calls at camera.hpp:192)                 */
  uint64_t samples;     /* camera paths started since the last clear                   */
  double last_render_ms; /* CUDA-event time of the last rt_render on its stream         */
  int32_t image_width;
  int32_t image_height;
  int32_t n_nodes; /* device BVH                                                       */
  int32_t n_spheres;
  int32_t n_quads; /* quad records, including the six behind every box                 */
  int32_t n_media;
  int32_t bvh_nodes_in_smem;
  int32_t kernel_launches; /* number of kernels this context has launched              */
  int32_t n_boxes;         /* box() lists turned into one slab-test primitive each     */
  int32_t n_views;         /* images the accumulator holds: 1 after rt_render / rt_upload_accum,
                              n_views after rt_render_views, 0 before anything was rendered */
  /* RT_RENDER_COUNTERS only, since the last clear — the N_* of the roofline model:
   * [0] BVH node visits (2 box tests each) [1] sphere tests [2] sphere hits [3] quad tests
   * [4] quad tests past the plane/t early-outs [5] medium tests [6..10] scatters by material
   * (lambertian, metal, dielectric, diffuse_light, isotropic) [11] checker [12] image
   * [13] noise texture evaluations [14] box tests                                       */
  uint64_t census[16];
} rt_stats;
int rt_get_stats(rt_ctx* ctx, rt_stats* out);

/* ---- closest-hit queries (parity harness; the same device traversal as rt_render) -- */
enum {
  RT_TRACE_FP32 = 0,  /* the production fp32 traversal + intersection                  */
  RT_TRACE_EXACT = 1, /* fp32 conservative traversal; every candidate re-evaluated in
                         fp64 with the reference's operation order (no FMA) so that the
                         winner is the one hittable::hit would report                  */
  RT_TRACE_SKIP_MEDIA = 2, /* constant_medium is transparent (SURVEY.md §8(c))         */
  RT_TRACE_RENDER_KERNEL = 4 /* rt_primary_visibility only: the rays are generated and traced by the
                         render kernel ITSELF (its AOV instantiation, planned for the scene as
                         rt_render plans it: same staging, node form, leaf steps and stack) in
                         fp32, media transparent — the traversal rt_render runs, under the
                         id / t / normal gate (camera.hpp:192, hittable_list.hpp:40-64)   */
};

/* n rays given as double origin[3n], direction[3n], time[n]; interval (tmin, tmax) as
 * in world.hit(r, interval(tmin, tmax), rec).  Outputs (any may be NULL): prim id or
 * -1; t in the reference's units (per un-normalised direction); normal = rec.normal
 * (already flipped against the ray); front_face.                                      */
int rt_trace_rays(rt_ctx* ctx, int64_t n, const double* origin, const double* direction,
                  const double* time, double tmin, double tmax, int32_t flags,
                  int32_t* prim_id, double* t, double* normal, uint8_t* front_face);

/* rt_trace_rays for rays that start ON a primitive, as every ray after the first of a path
 * does in rt_render: start_prim[i] is the reference primitive id (rt_hittable.prim_id) ray i
 * leaves from, or -1 for none, and the traversal applies rt_render's start-primitive rules
 * instead of an epsilon (a sphere gets the roots 0 and -2b/a, a quad is skipped, a box face's
 * slab plane is crossed at exactly 0).  start_prim == NULL is rt_trace_rays.  FP32 mode
 * only: RT_TRACE_EXACT with a start_prim is RT_ERR_INVALID (the reference has no start
 * primitive), and so is an id that is not a primitive of the device BVH (the boundary of a
 * medium, say) or that names more than one device primitive.                           */
int rt_trace_rays_from(rt_ctx* ctx, int64_t n, const double* origin, const double* direction,
                       const double* time, const int32_t* start_prim, double tmin, double tmax,
                       int32_t flags, int32_t* prim_id, double* t, double* normal,
                       uint8_t* front_face);

/* Pixel-centre primary rays (no jitter, no defocus, time 0, interval (0.001, inf)),
 * generated on the device from the camera frame: SURVEY.md §8(c) convention.  With
 * RT_TRACE_RENDER_KERNEL the rays are the fp32 rays the render kernel builds (get_ray
 * at zero jitter) and t / normal are its fp32 results widened to double.               */
int rt_primary_visibility(rt_ctx* ctx, const rt_camera_desc* cam, int32_t flags,
                          int32_t* prim_id, double* t, double* normal);

/* The render kernel's first TWO segments of the pixel-centre path, traced by render_kernel
 * itself (its AOV instantiation under the plan rt_render picks for the scene; media
 * transparent, time 0).  Where the pixel-centre ray hits, the kernel shades the hit as
 * rt_render does (surface_at + material scatter with the Philox stream of sample 0 of the
 * pixel under `seed`, bounce 1), starts the scattered ray on that primitive (rt_render's
 * start-primitive rule) and traces it with the same traversal.  Per pixel (row-major, any
 * output may be NULL): prim_id / t of the primary hit (-1 / inf on a miss); origin1 /
 * dir1 = the fp32 bounce ray (3 floats each, 0 without one); bounce_id / bounce_t /
 * bounce_normal / bounce_front = its closest hit as in rt_trace_rays, bounce_id =
 * RT_NO_BOUNCE when there is no bounce ray (primary miss, or the material absorbed or
 * emitted: a light, a metal ray scattered below the surface).                          */
enum { RT_NO_BOUNCE = -2147483647 - 1 };
int rt_bounce_visibility(rt_ctx* ctx, const rt_camera_desc* cam, uint64_t seed,
                         int32_t* prim_id, double* t, float* origin1, float* dir1,
                         int32_t* bounce_id, double* bounce_t, double* bounce_normal,
                         uint8_t* bounce_front);

/* Entry/exit parameters (rec1.t, rec2.t of SURVEY.md App. B.2, before clamping) of the
 * boundary of the medium_index-th RT_H_MEDIUM (DFS order) for n rays; NaN when missed. */
int rt_medium_spans(rt_ctx* ctx, int32_t medium_index, int64_t n, const double* origin,
                    const double* direction, const double* time, double* t1, double* t2);

/* texture::value(u, v, p) on the device for n points (fp32 arithmetic): uvp = n x
 * (u, v, px, py, pz) doubles in, rgb = n x 3 floats out.                               */
int rt_eval_texture(rt_ctx* ctx, int32_t texture, int64_t n, const double* uvp,
                    float* rgb);

/* material::scatter on the device for n hits, for distribution tests: inputs are the
 * incoming direction, the (flipped) normal, front_face; outputs scattered direction,
 * attenuation and the scatter flag.  Philox stream = (seed, i, 0).                    */
int rt_eval_scatter(rt_ctx* ctx, int32_t material, int64_t n, uint64_t seed,
                    const double* dir_in, const double* normal, const uint8_t* front_face,
                    float* dir_out, float* attenuation, uint8_t* scattered);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
