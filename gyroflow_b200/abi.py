"""ctypes mirror of include/gyroflow_cuda.h and loader of the product library.

The library is the hand-written sm_100a backend (gyroflow_b200/libgyroflow_cuda.so, built in-tree by
`make -C gyroflow_b200/csrc` / `__graft_entry__.build()`).  Loading fails loudly when it is missing:
there is no Python, PyTorch or CPU fallback for the warp.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GF_CUDA_LIB") or os.path.join(_HERE, "libgyroflow_cuda.so")    # GF_CUDA_LIB: an alternative build (tuning experiments)

MATRIX_STRIDE = 14
MESH_MAX_LEN = 839
KERNEL_PARAMS_SIZE = 368


class KernelParams(C.Structure):
    """`#[repr(C, packed(4))] struct KernelParams` — src/core/stabilization/mod.rs:101-150 (368 bytes)."""
    _pack_ = 4
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("stride", C.c_int32),
        ("output_width", C.c_int32), ("output_height", C.c_int32), ("output_stride", C.c_int32),
        ("matrix_count", C.c_int32), ("interpolation", C.c_int32), ("background_mode", C.c_int32),
        ("flags", C.c_int32), ("bytes_per_pixel", C.c_int32), ("pix_element_count", C.c_int32),
        ("background", C.c_float * 4), ("f", C.c_float * 2), ("c", C.c_float * 2), ("k", C.c_float * 12),
        ("fov", C.c_float), ("r_limit", C.c_float), ("lens_correction_amount", C.c_float),
        ("input_vertical_stretch", C.c_float), ("input_horizontal_stretch", C.c_float),
        ("background_margin", C.c_float), ("background_margin_feather", C.c_float), ("canvas_scale", C.c_float),
        ("input_rotation", C.c_float), ("output_rotation", C.c_float),
        ("translation2d", C.c_float * 2), ("translation3d", C.c_float * 4),
        ("source_rect", C.c_int32 * 4), ("output_rect", C.c_int32 * 4),
        ("digital_lens_params", C.c_float * 16), ("safe_area_rect", C.c_float * 4),
        ("max_pixel_value", C.c_float), ("distortion_model", C.c_int32), ("digital_lens", C.c_int32),
        ("pixel_value_limit", C.c_float), ("light_refraction_coefficient", C.c_float),
        ("plane_index", C.c_int32), ("reserved1", C.c_float), ("reserved2", C.c_float),
        ("ewa_coeffs_p", C.c_float * 4), ("ewa_coeffs_q", C.c_float * 4),
    ]

    def copy(self):
        o = KernelParams()
        C.memmove(C.byref(o), C.byref(self), C.sizeof(KernelParams))
        return o


assert C.sizeof(KernelParams) == KERNEL_PARAMS_SIZE


class BufferDesc(C.Structure):
    """gf_buffer_desc <- BufferDescription, src/core/gpu/mod.rs:17-24."""
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("stride", C.c_int32),
        ("has_rect", C.c_int32), ("rect", C.c_int32 * 4),
        ("has_rotation", C.c_int32), ("rotation", C.c_float),
        ("kind", C.c_int32), ("_pad", C.c_int32),
        ("ptr", C.c_void_p), ("len", C.c_size_t),
    ]


class QuatTrack(C.Structure):
    """gf_quat_track: sorted (timestamp us, unit quaternion w,i,j,k) arrays — TimeQuat, gyro_source/mod.rs:34."""
    _fields_ = [("ts_us", C.POINTER(C.c_int64)), ("quats", C.POINTER(C.c_double)), ("n", C.c_size_t)]


class KeyframeTrack(C.Structure):
    """gf_keyframe_track: one KeyframeManager track (keyframes.rs:83-90): ascending keys in us, value and easing (0..3) per key."""
    _fields_ = [("ts_us", C.POINTER(C.c_int64)), ("value", C.POINTER(C.c_double)), ("easing", C.POINTER(C.c_uint8)), ("n", C.c_size_t)]


KEYFRAME_TYPES = {"Fov": 0, "VideoRotation": 1, "ZoomingCenterX": 2, "ZoomingCenterY": 3, "BackgroundMargin": 4, "BackgroundFeather": 5,
                  "LensCorrectionStrength": 6, "LightRefractionCoeff": 7}      # GF_KF_* / KeyframeType (keyframes.rs:27-72)
EASING = {"NoEasing": 0, "EaseIn": 1, "EaseOut": 2, "EaseInOut": 3}             # keyframes.rs:74-81


class ComputeParams(C.Structure):
    """gf_compute_params: the slice of ComputeParams (compute_params.rs:13-69) FrameTransform::at_timestamp reads."""
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("output_width", C.c_int32), ("output_height", C.c_int32),
        ("camera_matrix", C.c_double * 9), ("distortion_coeffs", C.c_double * 12), ("radial_distortion_limit", C.c_double),
        ("input_horizontal_stretch", C.c_double), ("input_vertical_stretch", C.c_double), ("fov_scale", C.c_double),
        ("fovs", C.POINTER(C.c_double)), ("n_fovs", C.c_size_t), ("minimal_fovs", C.POINTER(C.c_double)), ("n_minimal_fovs", C.c_size_t),
        ("lens_optimal_fov", C.c_double), ("has_optimal_fov", C.c_int32),
        ("frame_readout_time", C.c_double), ("readout_horizontal", C.c_int32), ("readout_inverted", C.c_int32),
        ("framebuffer_inverted", C.c_int32), ("suppress_rotation", C.c_int32), ("fov_overview", C.c_int32),
        ("video_rotation", C.c_double), ("lens_correction_amount", C.c_double), ("light_refraction_coefficient", C.c_double),
        ("background_margin", C.c_double), ("background_margin_feather", C.c_double), ("background_mode", C.c_int32),
        ("adaptive_zoom_center_offset", C.c_double * 2),
        ("digital_lens_params", C.c_double * 16), ("n_digital_lens_params", C.c_int32),
        ("gyro_offset_ms", C.c_double), ("duration_ms", C.c_double),
        ("org", QuatTrack), ("smoothed", QuatTrack),
        # optional per-clip metadata (zero = absent)
        ("sync_offset_ts_us", C.POINTER(C.c_int64)), ("sync_offset_ms", C.POINTER(C.c_double)), ("n_sync_offsets", C.c_size_t),
        ("per_frame_time_offsets", C.POINTER(C.c_double)), ("n_per_frame_time_offsets", C.c_size_t),
        ("focal_length_smoothing_enabled", C.c_int32),
        ("focal_lengths", C.POINTER(C.c_double)), ("smoothed_focal_lengths", C.POINTER(C.c_double)), ("n_focal_lengths", C.c_size_t),
        ("readout_time_scale", C.c_double),
        ("camera_stab", C.c_void_p), ("n_camera_stab", C.c_size_t),
        ("keyframes", KeyframeTrack * 8), ("keyframe_timestamp_scale", C.c_double),
        ("lens_per_frame", C.c_void_p), ("n_lens_per_frame", C.c_size_t),
        ("distorting_mesh", C.c_void_p), ("n_distorting_mesh", C.c_size_t),
    ]


class MeshF64(C.Structure):
    """gf_mesh_f64: one frame's distorting mesh (file_metadata.mesh_correction[frame].0)."""
    _fields_ = [("data", C.POINTER(C.c_double)), ("len", C.c_size_t)]


class LensData(C.Structure):
    """gf_lens_data: one frame's get_lens_data_at_timestamp result (frame_transform.rs:82-163)."""
    _fields_ = [("camera_matrix", C.c_double * 9), ("distortion_coeffs", C.c_double * 12), ("radial_distortion_limit", C.c_double),
                ("input_horizontal_stretch", C.c_double), ("input_vertical_stretch", C.c_double)]


class CameraStab(C.Structure):
    """gf_camera_stab: CameraStabData (gyro_source/file_metadata.rs:41-48) with the Catmull-Rom points as flat arrays."""
    _fields_ = [
        ("offset", C.c_double), ("sensor_size", C.c_uint32 * 2), ("crop_area", C.c_float * 4), ("pixel_pitch", C.c_uint32 * 2),
        ("ibis_pos", C.POINTER(C.c_double)), ("ibis_xyz", C.POINTER(C.c_double)), ("n_ibis", C.c_size_t),
        ("ois_pos", C.POINTER(C.c_double)), ("ois_xyz", C.POINTER(C.c_double)), ("n_ois", C.c_size_t),
    ]


class StabConfig(C.Structure):
    """gf_stab_config: the fields of `Stabilization` get_frame_transform_at reads (stabilization/mod.rs:253-326)."""
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("output_width", C.c_int32), ("output_height", C.c_int32),
        ("interpolation", C.c_int32), ("pixel_type", C.c_int32), ("base_flags", C.c_int32), ("has_digital_lens", C.c_int32),
        ("light_refraction_keyframed", C.c_int32), ("has_ibis_data", C.c_int32), ("show_safe_area", C.c_int32),
        ("background", C.c_float * 4), ("canvas_scale", C.c_float), ("adaptive_zoom_window", C.c_double),
    ]


class PlaneSpec(C.Structure):
    """gf_plane_spec: one plane of a decoder frame (rendering/mod.rs:563-651): pixel type, size, `yuvi` list, value limit."""
    _fields_ = [("pixel_type", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("n_ind", C.c_int32), ("ind", C.c_int32 * 4),
                ("max_value", C.c_float)]


class QueueConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int32), ("distortion_model", C.c_int32), ("digital_lens", C.c_int32), ("depth", C.c_int32),
        ("pin_numa", C.c_int32), ("checksum", C.c_int32), ("stab", StabConfig),
    ]


# KernelParamsFlags — stabilization/mod.rs:85-98
FLAG_FIX_COLOR_RANGE, FLAG_HAS_DIGITAL_LENS, FLAG_FILL_WITH_BACKGROUND, FLAG_DRAWING_ENABLED = 1, 2, 4, 8
FLAG_HORIZONTAL_RS, FLAG_HAS_SOURCE_RECT, FLAG_HAS_OUTPUT_RECT, FLAG_FRAMEBUFFER_INVERTED = 16, 32, 64, 128
FLAG_HAS_IBIS_DATA, FLAG_HAS_MESH_DATA, FLAG_HAS_FPD_DATA, FLAG_ANY_UNDERWATER = 256, 512, 1024, 2048

INTERP = {"Bilinear": 2, "Bicubic": 4, "Lanczos4": 8, "EWA: RobidouxSharp": 10, "EWA: Robidoux": 11,
          "EWA: Mitchell": 12, "EWA: Catmull-Rom": 13}

LENS = {"none": 0, "opencv_fisheye": 1, "opencv_standard": 2, "poly3": 3, "poly5": 4, "ptlens": 5, "insta360": 6,
        "sony": 7, "generic_polynomial": 8, "gopro": 9, "gopro_superview": 10, "gopro_hyperview": 11,
        "gopro_warp": 12, "digital_stretch": 13, "gopro6_superview": 14}

# name -> (id, channel count, numpy scalar dtype string)
PIXEL_TYPES = {
    "Luma8": (0, 1, "u1"), "Luma16": (1, 1, "u2"), "RGB8": (2, 3, "u1"), "RGBA8": (3, 4, "u1"), "BGRA8": (4, 4, "u1"),
    "RGB16": (5, 3, "u2"), "RGBA16": (6, 4, "u2"), "AYUV16": (7, 4, "u2"), "RGBAf": (8, 4, "f4"), "RGBAf16": (9, 4, "f2"),
    "R32f": (10, 1, "f4"), "UV8": (11, 2, "u1"), "UV16": (12, 2, "u2"),
}

BUF_NONE, BUF_HOST, BUF_DEVICE = 0, 1, 2

# GF_FRAME_*: the decoder frame formats of rendering/mod.rs:563-651, in the header's order
FRAME_FORMATS = {name: i for i, name in enumerate([
    "NV12", "NV21", "P010LE", "P016LE", "P210LE", "P216LE", "P410LE", "P416LE", "YUV420P", "YUVJ420P",
    "YUV420P10LE", "YUV420P12LE", "YUV420P14LE", "YUV420P16LE", "YUV422P10LE", "YUV422P12LE", "YUV422P14LE", "YUV422P16LE",
    "YUV444P10LE", "YUV444P12LE", "YUV444P14LE", "YUV444P16LE", "YUVA444P10LE", "YUVA444P12LE", "YUVA444P16LE",
    "GBRAPF32LE", "GBRPF32LE", "AYUV64LE", "RGB24", "RGBA", "RGB48BE", "RGBA64BE"])}
FRAME_MAX_PLANES = 4

ERRORS = {0: "Ok", -1: "BadParams", -2: "SizeTooSmall", -3: "SizeMismatch", -4: "InvalidStride",
          -5: "UnsupportedCombo", -6: "CudaError", -7: "BufferTooSmall", -8: "NoStabilizationData"}

# every symbol include/gyroflow_cuda.h declares: (name, restype, argtypes)
_P = C.POINTER
EXPORTS = [
    ("gf_cuda_device_count", C.c_int, []),
    ("gf_cuda_device_name", C.c_int, [C.c_int, C.c_char_p, C.c_size_t]),
    ("gf_cuda_supports", C.c_int, [_P(BufferDesc), _P(BufferDesc)]),
    ("gf_cuda_version", C.c_char_p, []),
    ("gf_lens_from_name", C.c_int, [C.c_char_p]),
    ("gf_lens_name", C.c_char_p, [C.c_int]),
    ("gf_pixel_bytes", C.c_int, [C.c_int]),
    ("gf_combo_supported", C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int]),
    ("gf_cuda_create", C.c_int, [_P(C.c_void_p), C.c_int, _P(KernelParams), C.c_int, C.c_int, C.c_int,
                                 _P(BufferDesc), _P(BufferDesc), C.c_size_t]),
    ("gf_cuda_destroy", None, [C.c_void_p]),
    ("gf_cuda_undistort_image", C.c_int, [C.c_void_p, _P(BufferDesc), _P(BufferDesc), _P(KernelParams),
                                          C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                          C.c_void_p, C.c_size_t, C.c_void_p]),
    ("gf_cuda_undistort_image_dev", C.c_int, [C.c_void_p, _P(BufferDesc), _P(BufferDesc), _P(KernelParams),
                                              C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("gf_cuda_undistort_image_async", C.c_int, [C.c_void_p, _P(BufferDesc), _P(BufferDesc), _P(KernelParams),
                                                C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("gf_cuda_validate_tables_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    ("gf_cuda_undistort_points", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_size_t, C.c_int, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("gf_cuda_stmap_distort_dev", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("gf_cuda_generate_stmap", C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                          C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("gf_cuda_undistort_planes_dev", C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("gf_cuda_undistort_planes", C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    ("gf_cuda_selftest_exhaustive", C.c_int, [C.c_int, C.POINTER(C.c_ulonglong)]),
    ("gf_cuda_selftest_filter", C.c_int, [C.c_int, C.c_ulonglong, C.c_int, C.c_int, C.POINTER(C.c_ulonglong)]),
    ("gf_cuda_plan", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_size_t]),
    ("gf_cuda_synchronize", C.c_int, [C.c_void_p]),
    ("gf_cuda_set_overlays", C.c_int, [C.c_void_p, C.c_int]),
    ("gf_cuda_last_error", C.c_char_p, [C.c_void_p]),
    ("gf_cuda_backend_name", C.c_char_p, []),
    ("gf_cuda_launch_count", C.c_uint64, [C.c_void_p]),
    ("gf_cuda_filter_counts", C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    ("gf_cuda_selftest", C.c_int, [C.c_int, C.c_ulonglong, C.c_ulonglong, _P(C.c_ulonglong)]),
    ("gf_frame_transform_at_timestamp", C.c_int, [_P(ComputeParams), C.c_double, C.c_size_t, _P(KernelParams), C.c_void_p, C.c_size_t,
                                                  _P(C.c_size_t), _P(C.c_double), _P(C.c_double)]),
    ("gf_cuda_gyro_upload", C.c_int, [_P(C.c_void_p), C.c_int, _P(ComputeParams)]),
    ("gf_cuda_gyro_free", None, [C.c_void_p]),
    ("gf_cuda_frame_transform_dev", C.c_int, [C.c_void_p, _P(ComputeParams), C.c_double, C.c_size_t, _P(KernelParams), C.c_void_p, C.c_size_t,
                                              _P(C.c_size_t), _P(C.c_double), _P(C.c_double), C.c_void_p]),
    ("gf_cuda_find_fovs", C.c_int, [C.c_void_p, _P(ComputeParams), C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_float, C.c_void_p, C.c_void_p]),
    ("gf_zoom_dynamic_compute", C.c_int, [C.c_void_p, C.c_size_t, C.c_double, C.c_double, C.c_int, C.c_void_p]),
    ("gf_cuda_scan_tables_dev", C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("gf_cuda_undistort_image_dev_flagged", C.c_int, [C.c_void_p, _P(BufferDesc), _P(BufferDesc), _P(KernelParams),
                                                      C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("gf_cuda_undistort_planes_dev_flagged", C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                                       C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("gf_cuda_frame_transform_dev_flagged", C.c_int, [C.c_void_p, _P(ComputeParams), C.c_double, C.c_size_t, _P(KernelParams), C.c_void_p, C.c_size_t,
                                                      C.c_void_p, _P(C.c_size_t), _P(C.c_double), _P(C.c_double), C.c_void_p]),
    ("gf_table_flags_host", C.c_uint32, [C.c_void_p, C.c_size_t]),
    ("gf_get_frame_transform_at", C.c_int, [_P(StabConfig), _P(ComputeParams), _P(BufferDesc), _P(BufferDesc), C.c_void_p, C.c_size_t,
                                            C.c_double, C.c_size_t, C.c_double, _P(KernelParams)]),
    ("gf_abi_struct_size", C.c_size_t, [C.c_int]),
    ("gf_keyframe_value_at", C.c_int, [C.c_void_p, C.c_double, C.c_double, _P(C.c_double)]),
    ("gf_cuda_queue_create", C.c_int, [_P(C.c_void_p), _P(QueueConfig), _P(ComputeParams), _P(BufferDesc), _P(BufferDesc)]),
    ("gf_cuda_queue_submit", C.c_int, [C.c_void_p, C.c_size_t, C.c_double, _P(BufferDesc), _P(BufferDesc), C.c_void_p, C.c_size_t]),
    ("gf_cuda_queue_wait", C.c_int, [C.c_void_p, _P(C.c_size_t), _P(C.c_uint64)]),
    ("gf_cuda_queue_drain", C.c_int, [C.c_void_p]),
    ("gf_cuda_queue_launches", C.c_uint64, [C.c_void_p]),
    ("gf_cuda_queue_destroy", None, [C.c_void_p]),
    ("gf_cuda_queue_last_error", C.c_char_p, [C.c_void_p]),
    ("gf_cuda_bind_thread_to_device", C.c_int, [C.c_int]),
    ("gf_cuda_checksum_dev", C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    ("gf_cuda_host_register", C.c_int, [C.c_void_p, C.c_size_t]),
    ("gf_cuda_host_unregister", C.c_int, [C.c_void_p]),
    ("gf_frame_layout", C.c_int, [C.c_int, C.c_int32, C.c_int32, _P(PlaneSpec), _P(C.c_size_t)]),
    ("gf_background_for_plane", C.c_int, [C.c_int, _P(C.c_float), _P(C.c_int32), C.c_size_t, C.c_int, _P(C.c_float)]),
    ("gf_cuda_queue_create_frame", C.c_int, [_P(C.c_void_p), _P(QueueConfig), _P(ComputeParams), C.c_int, C.c_int, C.c_size_t,
                                             _P(BufferDesc), _P(BufferDesc)]),
    ("gf_cuda_queue_submit_frame", C.c_int, [C.c_void_p, C.c_size_t, C.c_double, C.c_size_t, _P(BufferDesc), _P(BufferDesc),
                                             C.c_void_p, C.c_size_t, C.c_int]),
    ("gf_cuda_queue_wait_frame", C.c_int, [C.c_void_p, _P(C.c_size_t), _P(C.c_uint64), C.c_size_t]),
]

_lib = None


class BackendMissing(RuntimeError):
    pass


def load_library(path=None):
    """dlopen the product library and bind every declared entry point.  Raises BackendMissing if it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise BackendMissing(
            "%s is missing: build it with `make -C gyroflow_b200/csrc` (or __graft_entry__.build()). "
            "There is no CPU fallback for the warp." % p)
    lib = C.CDLL(p)
    for name, restype, argtypes in EXPORTS:
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if path is None:
        _lib = lib
    return lib
