/* gyroflow_cuda.h — C ABI of the B200 (sm_100a) backend for Gyroflow's per-pixel warp.
 *
 * This header is the drop-in boundary.  Every entry point replaces one method of the
 * reference's backend-wrapper convention (there is no C ABI in the reference; the
 * convention is `<Backend>Wrapper::{new, undistort_image, list_devices, ...}` driven by
 * `Stabilization::{init_backends, process_pixels}`).  Citations are relative to the
 * reference tree (gyroflow/gyroflow @ b5e8828):
 *
 *   gf_kernel_params            <- KernelParams            src/core/stabilization/mod.rs:101-150
 *   GF_FLAG_*                   <- KernelParamsFlags       src/core/stabilization/mod.rs:83-99
 *   GF_INTERP_*                 <- Interpolation           src/core/stabilization/mod.rs:24-34
 *   GF_LENS_*                   <- DistortionModel ids     src/core/stabilization/distortion_models/mod.rs:92-110
 *                                  (numeric ids follow gpu/stabilize_spirv/src/distortion_models/mod.rs:62-80)
 *   GF_PIX_*                    <- PixelType impls         src/core/stabilization/pixel_formats.rs:50-302
 *   gf_buffer_desc              <- BufferDescription       src/core/gpu/mod.rs:17-24 (+ BufferSource::{Cpu,CUDABuffer} 34,67-70)
 *   matrices: rows x 14 f32     <- FrameTransform.matrices src/core/stabilization/frame_transform.rs:13,301-307
 *   mesh: <= 839 f32            <- FrameTransform.mesh_data src/core/gyro_source/splines.rs:88-89, sony.rs:483-548
 *
 * No torch / C++ types cross this boundary: plain pointers, sizes and PODs only.
 * There is NO CPU fallback behind these calls; when no CUDA device is usable every
 * compute entry point returns GF_ERR_CUDA.
 */
#ifndef GYROFLOW_CUDA_H
#define GYROFLOW_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#  define GF_API __declspec(dllexport)
#else
#  define GF_API __attribute__((visibility("default")))
#endif

/* ------------------------------------------------------------------------------------------
 * KernelParams — byte-for-byte mirror of `#[repr(C, packed(4))] struct KernelParams`
 * (src/core/stabilization/mod.rs:103-148).  368 bytes, every member 4-byte aligned.
 * ---------------------------------------------------------------------------------------- */
#pragma pack(push, 4)
typedef struct gf_kernel_params {
    int32_t width;                       /*   0 */
    int32_t height;                      /*   4 */
    int32_t stride;                      /*   8  input stride in bytes */
    int32_t output_width;                /*  12 */
    int32_t output_height;               /*  16 */
    int32_t output_stride;               /*  20  output stride in bytes */
    int32_t matrix_count;                /*  24  1 = no rolling-shutter correction */
    int32_t interpolation;               /*  28  GF_INTERP_* */
    int32_t background_mode;             /*  32  0 colour, 1 edge repeat, 2 edge mirror, 3 margin+feather */
    int32_t flags;                       /*  36  GF_FLAG_* */
    int32_t bytes_per_pixel;             /*  40 */
    int32_t pix_element_count;           /*  44 */
    float   background[4];               /*  48 */
    float   f[2];                        /*  64  focal length in pixels */
    float   c[2];                        /*  72  principal point */
    float   k[12];                       /*  80  distortion coefficients */
    float   fov;                         /* 128 */
    float   r_limit;                     /* 132 */
    float   lens_correction_amount;      /* 136 */
    float   input_vertical_stretch;      /* 140 */
    float   input_horizontal_stretch;    /* 144 */
    float   background_margin;           /* 148 */
    float   background_margin_feather;   /* 152 */
    float   canvas_scale;                /* 156 */
    float   input_rotation;              /* 160 */
    float   output_rotation;             /* 164 */
    float   translation2d[2];            /* 168 */
    float   translation3d[4];            /* 176 */
    int32_t source_rect[4];              /* 192  x, y, w, h */
    int32_t output_rect[4];              /* 208  x, y, w, h */
    float   digital_lens_params[16];     /* 224 */
    float   safe_area_rect[4];           /* 288 */
    float   max_pixel_value;             /* 304 */
    int32_t distortion_model;            /* 308  (unused by the CPU path; informational) */
    int32_t digital_lens;                /* 312  (unused by the CPU path; informational) */
    float   pixel_value_limit;           /* 316 */
    float   light_refraction_coefficient;/* 320 */
    int32_t plane_index;                 /* 324 */
    float   reserved1;                   /* 328 */
    float   reserved2;                   /* 332 */
    float   ewa_coeffs_p[4];             /* 336 */
    float   ewa_coeffs_q[4];             /* 352 */
} gf_kernel_params;                      /* 368 */
#pragma pack(pop)

#define GF_KERNEL_PARAMS_SIZE 368
#define GF_MATRIX_STRIDE      14     /* f32 per row: 3x3 inverse, sx, sy, ra, ox, oy */
#define GF_MESH_MAX_LEN       839    /* 9 + 9*9*2 + 9*9*4*2 + 20, splines.rs:88-89 */

#if defined(__cplusplus)
static_assert(sizeof(gf_kernel_params) == GF_KERNEL_PARAMS_SIZE, "KernelParams ABI drift");
#else
_Static_assert(sizeof(gf_kernel_params) == GF_KERNEL_PARAMS_SIZE, "KernelParams ABI drift");
#endif

/* KernelParamsFlags — src/core/stabilization/mod.rs:85-98 */
enum {
    GF_FLAG_FIX_COLOR_RANGE      = 1 << 0,
    GF_FLAG_HAS_DIGITAL_LENS     = 1 << 1,
    GF_FLAG_FILL_WITH_BACKGROUND = 1 << 2,
    GF_FLAG_DRAWING_ENABLED      = 1 << 3,
    GF_FLAG_HORIZONTAL_RS        = 1 << 4,
    GF_FLAG_HAS_SOURCE_RECT      = 1 << 5,
    GF_FLAG_HAS_OUTPUT_RECT      = 1 << 6,
    GF_FLAG_FRAMEBUFFER_INVERTED = 1 << 7,
    GF_FLAG_HAS_IBIS_DATA        = 1 << 8,
    GF_FLAG_HAS_MESH_DATA        = 1 << 9,
    GF_FLAG_HAS_FPD_DATA         = 1 << 10,
    GF_FLAG_ANY_UNDERWATER       = 1 << 11
};

/* Interpolation — src/core/stabilization/mod.rs:25-34 */
enum {
    GF_INTERP_BILINEAR       = 2,
    GF_INTERP_BICUBIC        = 4,
    GF_INTERP_LANCZOS4       = 8,
    GF_INTERP_ROBIDOUX_SHARP = 10,
    GF_INTERP_ROBIDOUX       = 11,
    GF_INTERP_MITCHELL       = 12,
    GF_INTERP_CATMULL_ROM    = 13
};

/* Lens-model plugin ids.  String ids are the reference's `DistortionModel::id()`
 * (distortion_models/mod.rs:92-110); integers 0..13 follow the `#[repr(i32)]` order in
 * gpu/stabilize_spirv/src/distortion_models/mod.rs:62-80, gopro6_superview (absent there) is 14. */
enum {
    GF_LENS_NONE               = 0,   /* also: "no digital lens" */
    GF_LENS_OPENCV_FISHEYE     = 1,
    GF_LENS_OPENCV_STANDARD    = 2,
    GF_LENS_POLY3              = 3,
    GF_LENS_POLY5              = 4,
    GF_LENS_PTLENS             = 5,
    GF_LENS_INSTA360           = 6,
    GF_LENS_SONY               = 7,
    GF_LENS_GENERIC_POLYNOMIAL = 8,
    GF_LENS_GOPRO              = 9,
    GF_LENS_GOPRO_SUPERVIEW    = 10,
    GF_LENS_GOPRO_HYPERVIEW    = 11,
    GF_LENS_GOPRO_WARP         = 12,
    GF_LENS_DIGITAL_STRETCH    = 13,
    GF_LENS_GOPRO6_SUPERVIEW   = 14,
    GF_LENS_COUNT              = 15
};

/* Pixel formats — the PixelType impls of pixel_formats.rs.  Formats that share a memory
 * layout and conversion (BGRA8 == RGBA8, AYUV16 == RGBA16) keep distinct ids for callers. */
enum {
    GF_PIX_LUMA8   = 0,   /* pixel_formats.rs:64-81   */
    GF_PIX_LUMA16  = 1,   /* :82-99   */
    GF_PIX_RGB8    = 2,   /* :100-117 */
    GF_PIX_RGBA8   = 3,   /* :118-135 */
    GF_PIX_BGRA8   = 4,   /* :136-153 */
    GF_PIX_RGB16   = 5,   /* :154-171 */
    GF_PIX_RGBA16  = 6,   /* :172-189 */
    GF_PIX_AYUV16  = 7,   /* :190-207 */
    GF_PIX_RGBAF   = 8,   /* :208-225 */
    GF_PIX_RGBAF16 = 9,   /* :231-248 */
    GF_PIX_R32F    = 10,  /* :249-266 */
    GF_PIX_UV8     = 11,  /* :267-284 */
    GF_PIX_UV16    = 12,  /* :285-302 */
    GF_PIX_COUNT   = 13
};

/* Error codes.  0 = ok.  The Rust side maps them onto GyroflowCoreError (src/core/lib.rs:2098-2141):
 * SIZE_TOO_SMALL -> SizeTooSmall, SIZE_MISMATCH -> SizeMismatch, BAD_STRIDE -> InvalidStride,
 * NO_DATA -> NoStabilizationData, everything else -> Unknown. */
enum {
    GF_OK                    =  0,
    GF_ERR_BAD_PARAMS        = -1,
    GF_ERR_SIZE_TOO_SMALL    = -2,   /* height < 4, stabilization/mod.rs:613, opencl.rs:179 */
    GF_ERR_SIZE_MISMATCH     = -3,   /* stabilization/mod.rs:636-637 */
    GF_ERR_BAD_STRIDE        = -4,   /* stabilization/mod.rs:639-640 */
    GF_ERR_UNSUPPORTED_COMBO = -5,
    GF_ERR_CUDA              = -6,   /* no device / driver error; see gf_cuda_last_error */
    GF_ERR_BUFFER_TOO_SMALL  = -7,   /* opencl.rs:336,352,355 "Buffer size mismatch" */
    GF_ERR_NO_DATA           = -8
};

/* BufferDescription + BufferSource::{Cpu, CUDABuffer} — src/core/gpu/mod.rs:17-24,34,67-70 */
enum { GF_BUF_NONE = 0, GF_BUF_HOST = 1, GF_BUF_DEVICE = 2 };

typedef struct gf_buffer_desc {
    int32_t  width, height, stride;  /* size: (w, h, stride in bytes) */
    int32_t  has_rect;               /* rect: Option<(x, y, w, h)> */
    int32_t  rect[4];
    int32_t  has_rotation;           /* rotation: Option<f32>, degrees */
    float    rotation;
    int32_t  kind;                   /* GF_BUF_HOST (BufferSource::Cpu) or GF_BUF_DEVICE (BufferSource::CUDABuffer) */
    int32_t  _pad;
    void*    ptr;                    /* host pointer or CUdeviceptr; borrowed for the call only */
    size_t   len;                    /* bytes reachable from ptr */
} gf_buffer_desc;

typedef struct gf_cuda_ctx gf_cuda_ctx;   /* opaque; one per host thread / stream, like the thread-local LRU (mod.rs:62-66) */

/* ---- capability probe: OclWrapper::list_devices opencl.rs:60, wgpu.rs:77,99,113 ---------- */
GF_API int         gf_cuda_device_count(void);
GF_API int         gf_cuda_device_name(int device, char* buf, size_t buf_len);   /* "[CUDA] NVIDIA B200" style name */
GF_API int         gf_cuda_supports(const gf_buffer_desc* in, const gf_buffer_desc* out); /* is_buffer_supported opencl.rs:451 */
GF_API const char* gf_cuda_version(void);
/* sizeof() of the structs that cross this ABI, for binding generators and their tests: 0 gf_kernel_params, 1 gf_buffer_desc,
 * 2 gf_compute_params, 3 gf_camera_stab, 4 gf_keyframe_track, 5 gf_stab_config, 6 gf_queue_config, 7 gf_lens_data, 8 gf_mesh_f64; 0 for any other index. */
GF_API size_t gf_abi_struct_size(int which);

/* ---- lens plugin surface: DistortionModel::from_name / id  distortion_models/mod.rs:79-90 -- */
GF_API int         gf_lens_from_name(const char* id);     /* unknown -> GF_LENS_OPENCV_FISHEYE, like from_name's default */
GF_API const char* gf_lens_name(int lens_id);             /* NULL if out of range */
GF_API int         gf_pixel_bytes(int pixel_type);        /* COUNT * SCALAR_BYTES, 0 if unknown */
GF_API int         gf_combo_supported(int pixel_type, int distortion_model, int digital_lens, int interpolation);

/* ---- construct: OclWrapper::new opencl.rs:178 / WgpuWrapper::new wgpu.rs:147 ----------------
 * Validates (height >= 4, stride >= 1, width <= 16384 — opencl.rs:179, wgpu.rs:150), selects the
 * pre-compiled kernel instantiation for (pixel_type, distortion_model, digital_lens, interpolation)
 * and allocates device staging for params / matrices (14*max(W,H) f32) / mesh (839 f32) / drawing,
 * plus src/dst staging when the buffers are HOST.  `digital_lens` = GF_LENS_NONE for Option::None. */
GF_API int gf_cuda_create(gf_cuda_ctx** out_ctx, int device,
                          const gf_kernel_params* params, int pixel_type,
                          int distortion_model, int digital_lens,
                          const gf_buffer_desc* in, const gf_buffer_desc* out,
                          size_t drawing_len);
GF_API void gf_cuda_destroy(gf_cuda_ctx* ctx);

/* ---- run: OclWrapper::undistort_image opencl.rs:330 / WgpuWrapper::undistort_image wgpu.rs:454
 * `params`, `matrices`, `mesh`, `drawing` are HOST pointers (they come out of FrameTransform).
 * HOST image buffers: H2D -> kernel -> D2H -> stream sync before return (opencl.rs:359,413).
 * DEVICE image buffers: everything is enqueued on `cu_stream` and the call returns without synchronising.
 * `cu_stream` is a CUstream/cudaStream_t handle; NULL selects the context's own non-blocking stream (NOT the
 * legacy default stream — pass cudaStreamLegacy (0x1) or cudaStreamPerThread (0x2) to name those explicitly). */
GF_API int gf_cuda_undistort_image(gf_cuda_ctx* ctx,
                                   const gf_buffer_desc* in, const gf_buffer_desc* out,
                                   const gf_kernel_params* params,
                                   const float* matrices, size_t matrix_rows,
                                   const float* mesh, size_t mesh_len,
                                   const uint8_t* drawing, size_t drawing_len,
                                   void* cu_stream);

/* Same, but `matrices_dev` / `mesh_dev` already live in device memory (frame-sharded render queue:
 * tables are broadcast once, see DESIGN.md "multi-GPU").  No reference counterpart. */
GF_API int gf_cuda_undistort_image_dev(gf_cuda_ctx* ctx,
                                       const gf_buffer_desc* in, const gf_buffer_desc* out,
                                       const gf_kernel_params* params,
                                       const float* matrices_dev, size_t matrix_rows,
                                       const float* mesh_dev, size_t mesh_len,
                                       void* cu_stream);

/* gf_cuda_undistort_image without the final stream synchronisation: with HOST buffers the H2D copy, the kernel and the
 * D2H copy are only enqueued.  The host buffers must be page-locked and stay valid until gf_cuda_synchronize(ctx).
 * Round-robin over a few contexts pipelines frame i+1's upload under frame i's kernel and frame i-1's download (the
 * reference's render loop is strictly sequential per device, rendering/mod.rs:451,657-661).  No reference counterpart. */
GF_API int gf_cuda_undistort_image_async(gf_cuda_ctx* ctx,
                                         const gf_buffer_desc* in, const gf_buffer_desc* out,
                                         const gf_kernel_params* params,
                                         const float* matrices, size_t matrix_rows,
                                         const float* mesh, size_t mesh_len, void* cu_stream);

/* Multi-plane frames (SURVEY f3).  The reference renders planar formats one plane at a time, each with its own Stabilization
 * object (rendering/mod.rs:484-548, 596-629), recomputing every pixel's source coordinate per plane.  When the planes share one
 * geometry — the four R32f planes of GBRAPF32, the U and V planes of planar YUV: all KernelParams fields equal except plane_index
 * and background, same buffer sizes/strides/rects — this call computes the coordinates once into a device map and then samples
 * each plane from it (1 + n launches — 3 + n for the EWA resamplers — bit-identical to n separate calls).  Otherwise it degrades
 * to n ordinary calls.  DEVICE buffers and device tables; `in`, `out`, `params` are arrays of n_planes. */
GF_API int         gf_cuda_undistort_planes_dev(gf_cuda_ctx* ctx, size_t n_planes, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                                const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                                const float* mesh_dev, size_t mesh_len, void* cu_stream);

/* The same for planes in HOST memory with host tables — what the render path hands over for planar software frames
 * (rendering/mod.rs:596-629: every plane a BufferSource::Cpu slice): every plane is staged to the device, the planes are rendered as
 * above (one coordinate pass when they share a geometry), every plane is copied back; synchronous like gf_cuda_undistort_image. */
GF_API int         gf_cuda_undistort_planes(gf_cuda_ctx* ctx, size_t n_planes, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                            const gf_kernel_params* params, const float* matrices, size_t matrix_rows,
                                            const float* mesh, size_t mesh_len, void* cu_stream);

/* Table trust for DEVICE-resident tables.  The packed kernel has a fast path that assumes every matrix entry is zero or of
 * moderate magnitude (2^-40..2^40) and that no row carries IBIS data; otherwise it keeps per-pixel guards.  Which path runs is
 * decided ON THE DEVICE from a verdict word that travels with the table (0 = tame and IBIS-free), read by the kernel at entry and
 * ordered by the stream like the table itself — there is no host-side cache keyed by pointer:
 *   - host tables (gf_cuda_undistort_image): scanned on the host while they are staged;
 *   - gf_cuda_frame_transform_dev: writes the verdict of the table it produces into `table_flags_dev`;
 *   - caller-owned device tables: gf_cuda_scan_tables_dev(matrices_dev, rows, table_flags_dev, stream) — asynchronous, one small
 *     kernel on `cu_stream` (which must be ordered after the writes of the table);
 *   - gf_cuda_undistort_image_dev (no verdict word): always the guarded path.
 * The verdict must cover at least params->matrix_count rows.  Whoever rewrites the table must rewrite the word (or pass NULL).
 * gf_cuda_validate_tables_dev is the synchronous query form: it waits for the device, scans, and returns 0, a positive bit mask
 * (1 = wild entry, 2 = IBIS rows) or a negative GF_ERR_*; it remembers nothing. */
GF_API int         gf_cuda_scan_tables_dev(const float* matrices_dev, size_t matrix_rows, uint32_t* table_flags_dev, void* cu_stream);
GF_API int         gf_cuda_undistort_image_dev_flagged(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                                       const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                                       const float* mesh_dev, size_t mesh_len, const uint32_t* table_flags_dev, void* cu_stream);
GF_API int         gf_cuda_undistort_planes_dev_flagged(gf_cuda_ctx* ctx, size_t n_planes, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                                        const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                                        const float* mesh_dev, size_t mesh_len, const uint32_t* table_flags_dev, void* cu_stream);
GF_API int         gf_cuda_validate_tables_dev(gf_cuda_ctx* ctx, const float* matrices_dev, size_t matrix_rows);

/* Host-only planning query (no CUDA call): which kernel variant would render a frame with these parameters.
 * table_flags: what the verdict word will hold — 0 = tame and IBIS-free, else non-zero.
 * Returns 0 general, 1 lean, 2 packed, 3 packed with trusted tables, OR-ed with 0x10 when the two-pass path is used; < 0 on error. */
GF_API int         gf_cuda_plan(const gf_kernel_params* params, int pixel_type, int distortion_model, int digital_lens,
                                const gf_buffer_desc* in, const gf_buffer_desc* out, size_t mesh_len, uint32_t table_flags, size_t n_planes);

/* Preview overlays of the reference's GPU kernels — draw_pixel + draw_safe_area, src/core/gpu/opencl_undistort.cl:109-154, buffer
 * produced by gpu/drawing.rs:8-50 (SURVEY §8 f4).  OFF by default: the CPU path, the parity target, draws none
 * (cpu_undistort.rs:234-251).  When on, gf_cuda_undistort_image uses its `drawing` argument (if KernelParams.flags has DRAWING_ENABLED):
 * entries with stage bit 0 are drawn onto the device copy of the input before the warp (the .cl draws them onto every source tap),
 * entries with stage bit 1 and the safe-area shading (safe_area_rect) onto the output after it.  The caller's input buffer is never
 * modified.  Single-plane calls only. */
GF_API int         gf_cuda_set_overlays(gf_cuda_ctx* ctx, int enabled);

/* Waits for the context's own stream AND for the stream of the most recent call that named one. */
GF_API int         gf_cuda_synchronize(gf_cuda_ctx* ctx);
GF_API const char* gf_cuda_last_error(gf_cuda_ctx* ctx);     /* ctx may be NULL: last global error */
GF_API const char* gf_cuda_backend_name(void);               /* ProcessedInfo.backend: "CUDA" (mod.rs:195-201) */
GF_API uint64_t    gf_cuda_launch_count(gf_cuda_ctx* ctx);   /* warp / coordinate / sampling kernels launched by this ctx so far: 1 per bilinear
                                                              * frame, 2 for bicubic / Lanczos4 (coordinate pass + sampling pass), 4 for EWA */
/* Counters of the most recent frame on the packed fisheye kernel's filtered rolling-shutter pre-pass (waits for the ctx's work first):
 * out[0] pairs sent to the tail launch (uncertified row choice, or the final pass left the exact fast sequences' window),
 * out[1] pixels sent to the tail launch (8-bit bilinear footprint not interior), out[2] non-zero if a queue was full (the tail launch
 * then re-rendered the whole frame), out[3] the part of out[0] deferred by the final pass.  All zero before the first such frame. */
GF_API int         gf_cuda_filter_counts(gf_cuda_ctx* ctx, uint32_t out[4]);

/* Device self-test of the exact packed-f32x2 primitives (division, square root, atanf, uniform-divisor division)
 * against the scalar IEEE operations they replace: n pseudo-random operand sets, mismatch counts in out4[0..3].
 * No reference counterpart (test hook). */
GF_API int         gf_cuda_selftest(int device, unsigned long long n, unsigned long long seed, unsigned long long* out4);
/* Exhaustive variant (seconds): every input of the packed atanf ([2^-28, 2^24)) and of the packed square root ([2^-56, 2^48));
 * out2 = mismatch counts.  Test hook. */
GF_API int         gf_cuda_selftest_exhaustive(int device, unsigned long long* out2);
/* Certificate of the filtered rolling-shutter pre-pass (DESIGN.md §4): n_cfg random fisheye lenses / mid-row matrices / frame sizes, every
 * `step`-th pixel evaluated by the approximate and by the exact chain on the device.  out4 = { pixels inside the regime, pixels whose
 * difference exceeds the proven bound (must be 0), pixels the certificate leaves uncertain, max difference / bound in 1e-6 units }. */
GF_API int         gf_cuda_selftest_filter(int device, unsigned long long seed, int n_cfg, int step, unsigned long long* out4);


/* ------------------------------------------------------------------------------------------
 * Per-frame transform producer — FrameTransform::at_timestamp, src/core/stabilization/frame_transform.rs:165-350,
 * with GyroSource::quat_at_timestamp, src/core/gyro_source/mod.rs:857-879.  f64 like the reference.
 * Scope: everything at_timestamp computes from numbers — readout timing incl. the capture-area scale and per-frame time offsets,
 * focal-length FOV compensation, multi-point sync offsets, the per-row quaternion product, the IBIS / OIS spline rows.  What it
 * reads through Rust objects stays in Rust (INTEGRATION.md): keyframe curves (pass the per-timestamp values in the scalar fields),
 * lens-profile interpolation (pass the resulting camera matrix / coefficients), mesh extraction (pass mesh_data to the warp).  The 3x3 pinv(K_new * R) is an analytic f64 inverse (nalgebra
 * uses an SVD; both round to the same f32 except for last-ulp cases — `matrices` are *inputs* of the bit-exact contract).
 * ---------------------------------------------------------------------------------------- */
typedef struct gf_quat_track {          /* TimeQuat = BTreeMap<i64 us, UnitQuaternion<f64>> (gyro_source/mod.rs:34) as sorted arrays */
    const int64_t* ts_us;
    const double*  quats;               /* n x 4: w, i, j, k */
    size_t         n;
} gf_quat_track;

/* One KeyframeManager track (src/core/keyframes.rs:83-90, the BTreeMap<i64, Keyframe> of one KeyframeType): keys ascending in
 * microseconds, easing per key (keyframes.rs:74-81: 0 NoEasing, 1 EaseIn, 2 EaseOut, 3 EaseInOut).  A custom_provider closure
 * (keyframes.rs:112, :170-176) has no C form: bake it into a track on the Rust side. */
typedef struct gf_keyframe_track { const int64_t* ts_us; const double* value; const uint8_t* easing; size_t n; } gf_keyframe_track;
enum { GF_KF_FOV = 0, GF_KF_VIDEO_ROTATION, GF_KF_ZOOMING_CENTER_X, GF_KF_ZOOMING_CENTER_Y, GF_KF_BACKGROUND_MARGIN, GF_KF_BACKGROUND_FEATHER,
       GF_KF_LENS_CORRECTION_STRENGTH, GF_KF_LIGHT_REFRACTION_COEFF, GF_KF_COUNT };
/* KeyframeManager::value_at_video_timestamp (keyframes.rs:169-205) for one track: returns 1 and writes *out for Some(value), 0 for None.
 * Between two keys the value is eased with Easing::get / Easing::interpolate (keyframes.rs:279-303; simple_easing 1.0.2 sine_in /
 * sine_out / sine_in_out in f32). */
GF_API int gf_keyframe_value_at(const gf_keyframe_track* track, double timestamp_ms, double timestamp_scale, double* out);

typedef struct gf_compute_params {      /* the slice of ComputeParams (compute_params.rs:13-69) + lens data at_timestamp reads */
    int32_t width, height, output_width, output_height;
    double  camera_matrix[9];           /* row-major, already scaled to the frame (get_lens_data_at_timestamp :95-160) */
    double  distortion_coeffs[12];
    double  radial_distortion_limit;
    double  input_horizontal_stretch, input_vertical_stretch;   /* <= 0.01 means 1.0 (:146-147) */
    double  fov_scale;
    const double* fovs;          size_t n_fovs;                  /* adaptive-zoom result, may be empty */
    const double* minimal_fovs;  size_t n_minimal_fovs;
    double  lens_optimal_fov;    int32_t has_optimal_fov;
    double  frame_readout_time;                                  /* ms; 0 = no rolling-shutter correction */
    int32_t readout_horizontal, readout_inverted;                /* ReadoutDirection::is_horizontal / is_inverted */
    int32_t framebuffer_inverted, suppress_rotation, fov_overview;
    double  video_rotation;                                      /* degrees */
    double  lens_correction_amount, light_refraction_coefficient;
    double  background_margin, background_margin_feather;
    int32_t background_mode;
    double  adaptive_zoom_center_offset[2];
    double  digital_lens_params[16]; int32_t n_digital_lens_params;
    double  gyro_offset_ms;                                      /* offset_at_video_timestamp for a single sync point */
    double  duration_ms;                                         /* <= 0: quat_at_timestamp returns identity (:858) */
    gf_quat_track org, smoothed;                                 /* quaternions / smoothed_quaternions (stored form smooth^-1 * org) */
    /* ---- optional per-clip metadata (zero-initialised = absent) -------------------------------------------------------------- */
    const int64_t* sync_offset_ts_us; const double* sync_offset_ms; size_t n_sync_offsets;   /* GyroSource::offsets_adjusted, sorted by
                                                                  * key (gyro_source/mod.rs:884-909); n == 0: gyro_offset_ms alone */
    const double* per_frame_time_offsets; size_t n_per_frame_time_offsets;                   /* file_metadata.per_frame_time_offsets (:224) */
    int32_t focal_length_smoothing_enabled;                      /* focal_length_fov_compensation (:70-80); NaN or <= 0 = None */
    const double* focal_lengths; const double* smoothed_focal_lengths; size_t n_focal_lengths;
    double  readout_time_scale;                                  /* capture_area_size.1 / sensor_size_px.1 of the lens_params entry closest
                                                                  * to the timestamp (get_frame_readout_time :26-29); 0 = none (1.0) */
    const struct gf_camera_stab* camera_stab; size_t n_camera_stab;   /* file_metadata.camera_stab_data, one entry per frame (:227-236, :269-287) */
    /* keyframed scalars at_timestamp evaluates per frame (frame_transform.rs:53, :167-174): a track with n > 0 replaces the constant above */
    gf_keyframe_track keyframes[GF_KF_COUNT];
    double  keyframe_timestamp_scale;                            /* KeyframeManager::timestamp_scale; 0 = None (1.0) */
    /* per-frame result of get_lens_data_at_timestamp (:82-163) for clips whose lens changes over time (interpolated lens profiles,
     * telemetry lens_params of zoom lenses): entry `frame` replaces camera_matrix / distortion_coeffs / radial_distortion_limit /
     * input_*_stretch above in at_timestamp, and camera_matrix / distortion_coeffs in the single-timestamp point path (gf_cuda_undistort_points,
     * ST maps); gf_cuda_find_fovs keeps the constants.  Rust evaluates it once per job; NULL = the constants above for every frame. */
    const struct gf_lens_data* lens_per_frame; size_t n_lens_per_frame;
    /* file_metadata.mesh_correction[frame].0 — the DISTORTING mesh (f64, sony.rs:483-511 layout) the point path applies
     * (frame_transform.rs:369-373, cpu_undistort.rs:712-746: adaptive zoom, undistort_points, the redistort ST map).  The warp itself takes
     * the undistorting mesh (.1, f32) as a call argument.  NULL = no mesh; an entry with len == 0 = none for that frame. */
    const struct gf_mesh_f64* distorting_mesh; size_t n_distorting_mesh;
} gf_compute_params;
typedef struct gf_mesh_f64 { const double* data; size_t len; } gf_mesh_f64;
typedef struct gf_lens_data {
    double camera_matrix[9]; double distortion_coeffs[12]; double radial_distortion_limit;
    double input_horizontal_stretch, input_vertical_stretch;
} gf_lens_data;

/* CameraStabData (src/core/gyro_source/file_metadata.rs:41-48): IBIS / OIS motion of one frame as Catmull-Rom splines over the
 * sensor row (gyro_source/splines.rs:8-83).  Points are (position, Vector3) pairs: `*_pos[n]` ascending, `*_xyz[n][3]`. */
typedef struct gf_camera_stab {
    double   offset;
    uint32_t sensor_size[2];
    float    crop_area[4];
    uint32_t pixel_pitch[2];
    const double* ibis_pos; const double* ibis_xyz; size_t n_ibis;
    const double* ois_pos;  const double* ois_xyz;  size_t n_ois;
} gf_camera_stab;

/* Host producer.  Fills the fields at_timestamp sets in `out_params` (everything else zeroed: `..Default::default()`),
 * writes rows x 14 f32 to `out_matrices` (rows = 1, height, or width for horizontal readout).  Returns GF_OK or
 * GF_ERR_BUFFER_TOO_SMALL when max_rows is too small. */
GF_API int gf_frame_transform_at_timestamp(const gf_compute_params* cp, double timestamp_ms, size_t frame,
                                           gf_kernel_params* out_params, float* out_matrices, size_t max_rows,
                                           size_t* out_rows, double* out_fov, double* out_minimal_fov);

/* Device producer: the quaternion tracks live in HBM (uploaded / broadcast once per job), one small kernel per frame
 * writes the rows x 14 table straight into device memory — no per-frame host SVD loop, no per-frame table upload. */
typedef struct gf_cuda_gyro gf_cuda_gyro;
GF_API int  gf_cuda_gyro_upload(gf_cuda_gyro** out, int device, const gf_compute_params* cp);
GF_API void gf_cuda_gyro_free(gf_cuda_gyro* g);
GF_API int  gf_cuda_frame_transform_dev(gf_cuda_gyro* g, const gf_compute_params* cp, double timestamp_ms, size_t frame,
                                        gf_kernel_params* out_params, float* matrices_dev, size_t max_rows,
                                        size_t* out_rows, double* out_fov, double* out_minimal_fov, void* cu_stream);
/* Same, and the kernel also leaves the table's trust verdict (0 = tame and IBIS-free; see gf_cuda_undistort_image_dev_flagged) in
 * `table_flags_dev` — produced with the table, ordered with it on the stream, no host round trip.
 * STREAM ORDERING (both forms): with cu_stream == NULL the kernel runs on the gyro object's own stream and the call waits for it
 * before returning, so any later consumer may read the table; with a stream the call only enqueues — give the warp call the same
 * stream (or order the two with an event). */
GF_API int  gf_cuda_frame_transform_dev_flagged(gf_cuda_gyro* g, const gf_compute_params* cp, double timestamp_ms, size_t frame,
                                                gf_kernel_params* out_params, float* matrices_dev, size_t max_rows, uint32_t* table_flags_dev,
                                                size_t* out_rows, double* out_fov, double* out_minimal_fov, void* cu_stream);
/* the same verdict for a host table (what the staging path of gf_cuda_undistort_image computes) */
GF_API uint32_t gf_table_flags_host(const float* matrices, size_t rows);

/* ------------------------------------------------------------------------------------------
 * Adaptive-zoom companion — zooming::FovIterative (src/core/zooming/fov_iterative.rs:31-189) over
 * undistort_points_with_rolling_shutter (src/core/stabilization/cpu_undistort.rs:636-858).
 * gf_cuda_find_fovs: one CTA per frame warps the 120 frame-edge points (+ <= 4 refinement rounds of 63) and reduces them to
 * the minimal FOV; the calculate_fovs adjustments (zooming/mod.rs:41-49) are applied inside.
 * gf_zoom_dynamic_compute: the temporal filter over the per-frame vector (zoom_dynamic.rs:56-76; method 0 gaussian,
 * 1 envelope follower), sequential, on the host like the reference.
 * ---------------------------------------------------------------------------------------- */
GF_API int gf_cuda_find_fovs(gf_cuda_gyro* g, const gf_compute_params* cp, int distortion_model, int digital_lens,
                             const double* timestamps_ms, size_t n, float fov_algorithm_margin,
                             double* out_fov_minimal, void* cu_stream);
/* undistort_points_with_rolling_shutter for an arbitrary list of (x, y) points — cpu_undistort.rs:636-641 (host in/out, synchronous). */
GF_API int gf_cuda_undistort_points(gf_cuda_gyro* g, const gf_compute_params* cp, int distortion_model, int digital_lens,
                                    double timestamp_ms, size_t frame, int use_fovs, double lens_correction_amount,
                                    const float* points_xy, size_t n, float* out_xy, void* cu_stream);

/* ST maps (SURVEY f4) — generate_stmaps, src/core/stmap.rs:6-146, for one frame, without the EXR container: both maps are raw
 * RGB f32 images in device memory (x / width, 1 - y / height, 0 — stmap.rs:131-135).
 *   dist   : width x height, undistort_points of every pixel (the "redistort" map, :112-116)
 *   undist : new_width x new_height (the bounding box of the undistorted frame edge, :58-77), rotate_and_distort of every pixel (:86-109)
 * Call once with NULL buffers to get new_width / new_height, then with buffers of width*height*3 and new_width*new_height*3 floats.
 * `cp` is the user's ComputeParams; the adjustments of :24-35 (suppress_rotation, fovs cleared, per_frame == 0 -> no readout time)
 * are applied inside.  Synchronous. */
GF_API int gf_cuda_stmap_distort_dev(gf_cuda_gyro* g, const gf_compute_params* cp, int distortion_model, int digital_lens,
                                     double timestamp_ms, size_t frame, float* out_rgb_dev, void* cu_stream);
GF_API int gf_cuda_generate_stmap(gf_cuda_gyro* g, const gf_compute_params* cp, int distortion_model, int digital_lens,
                                  int per_frame, size_t frame, double timestamp_ms, int32_t* out_new_width, int32_t* out_new_height,
                                  float* dist_rgb_dev, size_t dist_capacity_floats, float* undist_rgb_dev, size_t undist_capacity_floats,
                                  void* cu_stream);

GF_API int gf_zoom_dynamic_compute(const double* fov_minimal, size_t n, double window_s, double fps, int method, double* out);

/* ------------------------------------------------------------------------------------------
 * Stabilization::get_frame_transform_at<T> — src/core/stabilization/mod.rs:253-326 (with get_kernel_flags :226-251 and
 * get_rect :209-224): completes the KernelParams FrameTransform::at_timestamp produced with the per-buffer fields — pixel limits,
 * sizes and strides, interpolation, background, bytes per pixel, flags, EWA coefficients, safe-area rect, buffer rotations,
 * source / output rects.  Host only, no CUDA call.  `kp` in: the fields at_timestamp sets (gf_frame_transform_at_timestamp /
 * gf_cuda_frame_transform_dev); out: complete.
 * ---------------------------------------------------------------------------------------- */
typedef struct gf_stab_config {            /* the fields of `Stabilization` the function reads */
    int32_t width, height;                 /* self.size */
    int32_t output_width, output_height;   /* self.output_size */
    int32_t interpolation;                 /* Interpolation as i32: 2, 4, 8, 10..13 */
    int32_t pixel_type;                    /* GF_PIX_*: T::COUNT, T::SCALAR_BYTES, T::default_max_value() */
    int32_t base_flags;                    /* self.kernel_flags: FIX_COLOR_RANGE / FILL_WITH_BACKGROUND / DRAWING_ENABLED as set by the caller */
    int32_t has_digital_lens;              /* compute_params.digital_lens.is_some() */
    int32_t light_refraction_keyframed;    /* keyframes.is_keyframed(LightRefractionCoeff) */
    int32_t has_ibis_data;                 /* file_metadata.camera_stab_data.len() > frame (cp->camera_stab is consulted as well) */
    int32_t show_safe_area;                /* compute_params.show_safe_area */
    float   background[4];                 /* compute_params.background */
    float   canvas_scale;                  /* self.drawing.scale */
    double  adaptive_zoom_window;          /* compute_params.adaptive_zoom_window */
} gf_stab_config;
GF_API int gf_get_frame_transform_at(const gf_stab_config* stab, const gf_compute_params* cp, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                     const float* mesh, size_t mesh_len, double timestamp_ms, size_t frame, double minimal_fov, gf_kernel_params* kp);
/* timestamp_ms: the frame's video timestamp — only the Fov keyframe of the safe-area rectangle reads it (mod.rs:299). */

/* ------------------------------------------------------------------------------------------
 * Frame-sharded render queue (SURVEY §8e; the shape of rendering/mod.rs:451,531-542,657-661 with rendering/render_queue.rs:550-612
 * turned inside out: instead of whole jobs in parallel, the frames of one job run `depth` deep on one GPU, and `i -> GPU i mod G`
 * across the processes of a box).  One queue = one device: `depth` slots, each with its own stream, device table + verdict word,
 * and (HOST buffers) device staging.  Per submitted frame, all on the slot's stream, nothing synchronous:
 *     gf_cuda_frame_transform_dev_flagged (table + verdict on the device)  ->  [H2D]  ->  warp  ->  [checksum]  ->  [D2H]
 * gf_cuda_queue_submit never blocks: with `depth` frames already in flight it fails with GF_ERR_BAD_PARAMS ("queue full") — call
 * gf_cuda_queue_wait first; gf_cuda_queue_wait blocks until the OLDEST frame is done and returns frames in submission order.  HOST buffers must be page-locked and stay valid until the
 * frame has been waited for.  `cp` is copied shallowly: the arrays it points to (tracks are uploaded at creation; fovs, offsets, focal lengths,
 * camera_stab, keyframe tracks, lens_per_frame are read per frame on the host) must stay valid until gf_cuda_queue_destroy.  The optional checksum is sum(word[i] * (2 i + 1)) mod 2^64 over the output buffer's 32-bit words.
 * ---------------------------------------------------------------------------------------- */
typedef struct gf_cuda_queue gf_cuda_queue;
typedef struct gf_queue_config {
    int32_t device;
    int32_t distortion_model, digital_lens;   /* GF_LENS_* (digital_lens: GF_LENS_NONE for Option::None) */
    int32_t depth;                            /* frames in flight, 1..16 */
    int32_t pin_numa;                         /* non-zero: gf_cuda_bind_thread_to_device(device) before any staging is allocated */
    int32_t checksum;                         /* non-zero: compute the per-frame output checksum */
    gf_stab_config stab;
} gf_queue_config;
GF_API int      gf_cuda_queue_create(gf_cuda_queue** out, const gf_queue_config* cfg, const gf_compute_params* cp,
                                     const gf_buffer_desc* in_proto, const gf_buffer_desc* out_proto);
GF_API int      gf_cuda_queue_submit(gf_cuda_queue* q, size_t frame, double timestamp_ms, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                     const float* mesh, size_t mesh_len);
GF_API int      gf_cuda_queue_wait(gf_cuda_queue* q, size_t* out_frame, uint64_t* out_checksum);   /* GF_ERR_NO_DATA when nothing is in flight */
GF_API int      gf_cuda_queue_drain(gf_cuda_queue* q);                                             /* wait for everything, discard the results */
GF_API uint64_t gf_cuda_queue_launches(gf_cuda_queue* q);                                          /* warp + producer (+ checksum) kernels launched */
GF_API void     gf_cuda_queue_destroy(gf_cuda_queue* q);
GF_API const char* gf_cuda_queue_last_error(gf_cuda_queue* q);

/* Bind the calling thread to the CPUs of the NUMA node the GPU hangs off (/sys/bus/pci/devices/<bdf>/local_cpulist), so that
 * page-locked staging allocated afterwards — by this library or by the caller — is node-local and the copy threads do not cross
 * the socket interconnect.  Returns the number of CPUs in the mask, 0 if the topology is unknown (nothing changed), < 0 on error. */
GF_API int      gf_cuda_bind_thread_to_device(int device);
/* Page-lock an existing host allocation (a decoder frame pool, a long-lived Vec<u8> — what BufferSource::Cpu borrows from) so that
 * HOST-buffer calls copy at the link's rate instead of through the driver's bounce buffers.  cudaHostRegister / cudaHostUnregister;
 * the caller owns the lifetime: unregister before freeing.  Registering twice is not an error. */
GF_API int      gf_cuda_host_register(void* ptr, size_t len);
GF_API int      gf_cuda_host_unregister(void* ptr);
/* sum(word[i] * (2 i + 1)) mod 2^64 over len / 4 words of device memory, accumulated into *out_dev (zeroed first), on `cu_stream` */
GF_API int      gf_cuda_checksum_dev(const void* ptr_dev, size_t len, uint64_t* out_dev, void* cu_stream);

#ifdef __cplusplus
}
#endif
#endif /* GYROFLOW_CUDA_H */
