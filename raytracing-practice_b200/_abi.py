"""ctypes mirror of include/rt_b200.h (the C-ABI drop-in boundary).

Field order and types must match the header exactly; tests/test_abi.py checks sizeof()
against the values the C compiler reports (rt_abi_sizeof in the shared library).
"""
import ctypes as C

RT_B200_ABI_VERSION = 1

# error codes
RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_NO_SCENE, RT_ERR_UNSUPPORTED, RT_ERR_NO_DEVICE = 0, -1, -2, -3, -4, -5

# hittable kinds (reference file:line in the header)
RT_H_SPHERE, RT_H_QUAD, RT_H_LIST, RT_H_BVH, RT_H_TRANSLATE, RT_H_ROTATE_Y, RT_H_MEDIUM = 1, 2, 3, 4, 5, 6, 7
RT_M_LAMBERTIAN, RT_M_METAL, RT_M_DIELECTRIC, RT_M_DIFFUSE_LIGHT, RT_M_ISOTROPIC = 1, 2, 3, 4, 5
RT_T_SOLID, RT_T_CHECKER, RT_T_IMAGE, RT_T_NOISE = 1, 2, 3, 4

RT_BUF_ACCUM_I64, RT_BUF_RADIANCE_F32, RT_BUF_RGB8 = 0, 1, 2
RT_TRACE_FP32, RT_TRACE_EXACT, RT_TRACE_SKIP_MEDIA, RT_TRACE_RENDER_KERNEL = 0, 1, 2, 4
RT_NO_BOUNCE = -(2 ** 31)  # rt_bounce_visibility: no bounce ray
RT_RENDER_DEFAULT, RT_RENDER_COUNTERS, RT_RENDER_MEGAKERNEL, RT_RENDER_STREAM, RT_RENDER_REFILL = 0, 1, 2, 8, 16


class rt_hittable(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("material", C.c_int32),
        ("child0", C.c_int32),
        ("child1", C.c_int32),
        ("prim_id", C.c_int32),
        ("reserved", C.c_int32),
        ("p", C.c_double * 9),
        ("bbox", C.c_double * 6),
    ]


class rt_material(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("texture", C.c_int32),
        ("albedo", C.c_double * 3),
        ("fuzz", C.c_double),
        ("ior", C.c_double),
    ]


class rt_texture(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("even", C.c_int32),
        ("odd", C.c_int32),
        ("image", C.c_int32),
        ("perlin", C.c_int32),
        ("reserved", C.c_int32),
        ("color", C.c_double * 3),
        ("scale", C.c_double),
    ]


class rt_image(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgb", C.POINTER(C.c_uint8))]


class rt_perlin(C.Structure):
    _fields_ = [
        ("randvec", (C.c_double * 3) * 256),
        ("perm_x", C.c_int32 * 256),
        ("perm_y", C.c_int32 * 256),
        ("perm_z", C.c_int32 * 256),
    ]


class rt_scene_desc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("root", C.c_int32),
        ("n_hittables", C.c_int32),
        ("n_child_index", C.c_int32),
        ("n_materials", C.c_int32),
        ("n_textures", C.c_int32),
        ("n_images", C.c_int32),
        ("n_perlins", C.c_int32),
        ("n_prims", C.c_int32),
        ("reserved", C.c_int32),
        ("hittables", C.POINTER(rt_hittable)),
        ("child_index", C.POINTER(C.c_int32)),
        ("materials", C.POINTER(rt_material)),
        ("textures", C.POINTER(rt_texture)),
        ("images", C.POINTER(rt_image)),
        ("perlins", C.POINTER(rt_perlin)),
    ]


class rt_camera_desc(C.Structure):
    _fields_ = [
        ("aspect_ratio", C.c_double),
        ("image_width", C.c_int32),
        ("samples_per_pixel", C.c_int32),
        ("max_depth", C.c_int32),
        ("reserved", C.c_int32),
        ("background", C.c_double * 3),
        ("vfov", C.c_double),
        ("lookfrom", C.c_double * 3),
        ("lookat", C.c_double * 3),
        ("vup", C.c_double * 3),
        ("defocus_angle", C.c_double),
        ("focus_dist", C.c_double),
    ]


class rt_camera_frame(C.Structure):
    _fields_ = [
        ("image_width", C.c_int32),
        ("image_height", C.c_int32),
        ("pixel_samples_scale", C.c_double),
        ("center", C.c_double * 3),
        ("pixel00_loc", C.c_double * 3),
        ("pixel_delta_u", C.c_double * 3),
        ("pixel_delta_v", C.c_double * 3),
        ("u", C.c_double * 3),
        ("v", C.c_double * 3),
        ("w", C.c_double * 3),
        ("defocus_disk_u", C.c_double * 3),
        ("defocus_disk_v", C.c_double * 3),
    ]


class rt_render_opts(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("sample_begin", C.c_int32),
        ("sample_count", C.c_int32),
        ("clear", C.c_int32),
        ("flags", C.c_int32),
        ("peer_accum", C.c_void_p),
        ("push_accum", C.c_void_p),
    ]


class rt_ipc_handle(C.Structure):
    _fields_ = [("bytes", C.c_ubyte * 64)]


class rt_stats(C.Structure):
    _fields_ = [
        ("rays", C.c_uint64),
        ("samples", C.c_uint64),
        ("last_render_ms", C.c_double),
        ("image_width", C.c_int32),
        ("image_height", C.c_int32),
        ("n_nodes", C.c_int32),
        ("n_spheres", C.c_int32),
        ("n_quads", C.c_int32),
        ("n_media", C.c_int32),
        ("bvh_nodes_in_smem", C.c_int32),
        ("kernel_launches", C.c_int32),
        ("n_boxes", C.c_int32),
        ("n_views", C.c_int32),
        ("census", C.c_uint64 * 16),
    ]


# Every symbol include/rt_b200.h declares (tests check the library exports all of them).
C_ABI_SYMBOLS = [
    "rt_camera_initialize",
    "rt_init",
    "rt_shutdown",
    "rt_last_error",
    "rt_upload_scene",
    "rt_render",
    "rt_render_views",
    "rt_synchronize",
    "rt_accum_device_ptr",
    "rt_reduce_buffer",
    "rt_peer_open",
    "rt_peer_enable",
    "rt_peer_close",
    "rt_adopt_reduce_buffer",
    "rt_download",
    "rt_upload_accum",
    "rt_get_stats",
    "rt_trace_rays",
    "rt_trace_rays_from",
    "rt_primary_visibility",
    "rt_bounce_visibility",
    "rt_medium_spans",
    "rt_eval_texture",
    "rt_eval_scatter",
]
