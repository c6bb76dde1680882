"""ctypes mirror of include/rtfs_b200.h (types and constants only; no behaviour).

Field order and types must match the header exactly; tests/test_abi.py checks sizeof() of every
struct against the values the compiled library reports.
"""
import ctypes as C

RT_ABI_VERSION = 6

RT_OK = 0
RT_ERR_INVALID_ARGUMENT = -1
RT_ERR_CUDA = -2
RT_ERR_NO_DEVICE = -3
RT_ERR_UNSUPPORTED = -4
RT_ERR_DEGENERATE = -5
RT_ERR_IO = -6

# RtShape — Hittable cases, RayTracing/Hittable.fs:3-6
RT_SHAPE_SPHERE = 0
RT_SHAPE_UNBOUNDED_SPHERE = 1
RT_SHAPE_INFINITE_PLANE = 2

# RtStyle — SphereStyle / InfinitePlaneStyle cases, RayTracing/Sphere.fs:10-37, InfinitePlane.fs:3-13
RT_STYLE_LIGHT_SOURCE = 0
RT_STYLE_LIGHT_SOURCE_CAP = 1
RT_STYLE_PURE_REFLECTION = 2
RT_STYLE_FUZZED_REFLECTION = 3
RT_STYLE_LAMBERT_REFLECTION = 4
RT_STYLE_DIELECTRIC = 5
RT_STYLE_GLASS = 6

# RtTextureKind — RayTracing/Texture.fs:5-22
RT_TEX_COLOUR = 0
RT_TEX_IMAGE = 1
RT_TEX_CHECKERED = 2

RT_MODE_MEGAKERNEL = 0
RT_MODE_WAVEFRONT = 1

RT_FLAG_COUNTERS = 1
RT_FLAG_NO_SMEM = 2
RT_FLAG_WIDE_BVH = 4
RT_FLAG_BVH2 = 8
RT_FLAG_LOCKSTEP = 16
RT_FLAG_FLOW = 32
RT_FLAG_NO_LEAN = 64
RT_FLAG_NOISE = 128  # rt_frame_begin only: keep the per-pixel sum of squares for rt_frame_noise

RT_COMM_ID_BYTES = 128

RT_BVH_SAH = 0
RT_BVH_REFERENCE = 1


class RtTexture(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("colour", C.c_uint8 * 3),
        ("_pad0", C.c_uint8),
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("rgb8", C.POINTER(C.c_uint8)),
        ("even", C.c_int32),
        ("odd", C.c_int32),
        ("grid_size", C.c_double),
        ("map_centre", C.c_double * 3),
        ("map_radius", C.c_double),
    ]


class RtHittable(C.Structure):
    _fields_ = [
        ("shape", C.c_int32),
        ("style", C.c_int32),
        ("p", C.c_double * 3),
        ("n", C.c_double * 3),
        ("radius", C.c_double),
        ("albedo", C.c_double),
        ("fuzz", C.c_double),
        ("ior", C.c_double),
        ("prob", C.c_double),
        ("texture", C.c_int32),
        ("colour", C.c_uint8 * 3),
        ("_pad0", C.c_uint8),
    ]


class RtCamera(C.Structure):
    _fields_ = [
        ("view_origin", C.c_double * 3),
        ("view_dir", C.c_double * 3),
        ("xaxis_origin", C.c_double * 3),
        ("xaxis_dir", C.c_double * 3),
        ("yaxis_dir", C.c_double * 3),
        ("viewport_width", C.c_double),
        ("viewport_height", C.c_double),
        ("focal_length", C.c_double),
        ("samples_per_pixel", C.c_int32),
        ("bounce_depth", C.c_int32),
    ]


class RtRenderOpts(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64),
        ("adaptive", C.c_int32),
        ("mode", C.c_int32),
        ("gamma", C.c_int32),
        ("flags", C.c_int32),
    ]


class RtStats(C.Structure):
    _fields_ = [
        ("paths", C.c_uint64),
        ("rays", C.c_uint64),
        ("box_tests", C.c_uint64),
        ("prim_tests", C.c_uint64),
        ("kernel_ms", C.c_double),
        ("total_ms", C.c_double),
        ("pixels_early_out", C.c_uint64),
        ("launches", C.c_int32),
        ("_pad0", C.c_int32),
        ("main_ms", C.c_double),
        ("main_rays", C.c_uint64),
        ("degenerate_paths", C.c_uint64),
    ]


class RtFrameProgress(C.Structure):
    _fields_ = [
        ("samples_done", C.c_int32),
        ("samples_target", C.c_int32),
        ("paths_done", C.c_uint64),
        ("paths_target", C.c_uint64),
        ("pixels_flagged", C.c_uint64),
        ("last_pass_ms", C.c_double),
        ("device_ms", C.c_double),
        ("passes", C.c_int32),
        ("done", C.c_int32),
    ]


class RtFrameNoise(C.Structure):
    _fields_ = [
        ("pixels", C.c_uint64),
        ("pixels_above", C.c_uint64),
        ("max_se", C.c_double),
        ("mean_se", C.c_double),
        ("tolerance", C.c_double),
    ]


class RtFrameConvergence(C.Structure):
    _fields_ = [
        ("tolerance", C.c_double),
        ("min_samples", C.c_int32),
        ("interval", C.c_int32),
        ("next_check", C.c_int32),
        ("checks", C.c_int32),
        ("pixels_active", C.c_uint64),
        ("pixels_converged", C.c_uint64),
    ]


class RtDenoiseOpts(C.Structure):
    _fields_ = [
        ("iterations", C.c_int32),
        ("feature_samples", C.c_int32),
        ("sigma_colour", C.c_double),
        ("sigma_normal", C.c_double),
        ("sigma_albedo", C.c_double),
        ("sigma_depth", C.c_double),
        ("gamma", C.c_int32),
        ("_pad0", C.c_int32),
    ]


class RtSceneRebuild(C.Structure):
    _fields_ = [
        ("objects_removed", C.c_int32),
        ("objects_appended", C.c_int32),
        ("n_objects", C.c_int32),
        ("n_bounded", C.c_int32),
        ("nodes", C.c_int32),
        ("depth", C.c_int32),
        ("on_device", C.c_int32),
        ("launches", C.c_int32),
        ("generation", C.c_uint64),
        ("device_ms", C.c_double),
    ]


class RtSceneUpdate(C.Structure):
    _fields_ = [
        ("objects", C.c_int32),
        ("textures", C.c_int32),
        ("spheres_moved", C.c_int32),
        ("nodes_refit", C.c_int32),
        ("generation", C.c_uint64),
        ("device_ms", C.c_double),
        ("launches", C.c_int32),
        ("_pad0", C.c_int32),
    ]


# snapshots of progressive frames (rt_frame_save / rt_frame_resume; the format is in include/rtfs_b200.h)
RT_SNAPSHOT_VERSION = 1
RT_FRAME_CAMERA = 0
RT_FRAME_VIEWS = 1
RT_FRAME_WINDOW = 2


class RtSnapshotHeader(C.Structure):
    _fields_ = [
        ("magic", C.c_char * 8),
        ("version", C.c_uint32),
        ("header_bytes", C.c_uint32),
        ("total_bytes", C.c_uint64),
        ("checksum", C.c_uint64),
        ("scene_fingerprint", C.c_uint64),
        ("n_objects", C.c_int32),
        ("n_textures", C.c_int32),
        ("kind", C.c_int32),
        ("n_views", C.c_int32),
        ("camera", RtCamera),
        ("max_width_coord", C.c_int32),
        ("max_height_coord", C.c_int32),
        ("window", C.c_int32 * 4),
        ("opts", RtRenderOpts),
        ("samples_per_pixel", C.c_int32),
        ("samples_done", C.c_int32),
        ("samples_target", C.c_int32),
        ("n_probe", C.c_int32),
        ("passes", C.c_int32),
        ("_pad0", C.c_int32),
        ("n_pixels", C.c_uint64),
        ("pixels_flagged", C.c_uint64),
        ("pixels_active", C.c_uint64),
        ("paths_done", C.c_uint64),
        ("conv_tolerance", C.c_double),
        ("conv_min", C.c_int32),
        ("conv_interval", C.c_int32),
        ("conv_checks", C.c_int32),
        ("pace_devices", C.c_int32),
        ("ms_per_sample", C.c_double),
    ]
