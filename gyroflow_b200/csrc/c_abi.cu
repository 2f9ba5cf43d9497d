// c_abi.cu — extern "C" boundary of the CUDA backend (include/gyroflow_cuda.h).
//
// Mirrors the reference's backend-wrapper life cycle:
//   gf_cuda_create          <- OclWrapper::new        src/core/gpu/opencl.rs:178  (WgpuWrapper::new wgpu.rs:147)
//   gf_cuda_undistort_image <- OclWrapper::undistort_image opencl.rs:330-448 (wgpu.rs:454-559)
//   gf_cuda_destroy         <- Drop / clear_gpu_cache_current_thread  stabilization/mod.rs:72-81
// plus the validation `Stabilization::process_pixels` performs before dispatch (stabilization/mod.rs:612-640).
// There is no CPU fallback: without a usable CUDA device every compute call fails with GF_ERR_CUDA.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <cmath>
#include <algorithm>
#include <string>
#include <vector>

#include "kernel_registry.h"
#include "c_abi_internal.h"
#include <nvtx3/nvToolsExt.h>

using namespace gf;

namespace {

thread_local std::string g_last_error;

struct Slot {                 // one in-flight set of per-frame tables
    float* h_mat = nullptr;   // pinned
    float* d_mat = nullptr;
    float* h_mesh = nullptr;  // pinned
    float* d_mesh = nullptr;
    double* d_mesh64 = nullptr;   // the mesh widened to f64 once per frame, like cpu_undistort.rs:539
    cudaEvent_t done = nullptr;
};
constexpr int kSlots = 4;

} // namespace

struct gf_cuda_ctx {
    int device = 0;
    int pixel_type = 0, distortion_model = 0, digital_lens = 0, interpolation = 0;
    int layout = 0, bpp = 0;
    int width = 0, height = 0, output_width = 0, output_height = 0;    // Stabilization.size / output_size
    KernelFn fn = nullptr;        // general instantiation (run-time feature tests)
    KernelFn fn_lean = nullptr;   // rare features compiled out
    KernelFn fn_x2 = nullptr;     // lean + two pixels per thread on the packed f32x2 pipe; trusted / guarded path picked from a device word
    KernelFn fn_x2c = nullptr;    // the packed kernel writing a coordinate map (pass 1 of the two-pass path)
    KernelFn fn_x2f = nullptr;    // the packed kernel's main launch for filtered frames (fn_x2 renders their tail)
    uint32_t* d_const_flags = nullptr;   // two device words {0, 1}: the verdict of the host scan of host tables, as the kernel wants it
    uint32_t* d_vflags = nullptr;        // scratch verdict word of gf_cuda_validate_tables_dev
    cudaStream_t last_stream = nullptr;  // the stream of the most recent call (gf_cuda_synchronize waits for it too)
    // filtered rolling-shutter pre-pass (packed fisheye kernel): queues of deferred pixel pairs and pixels + two ping-pong sets of
    // GF_FLT_WORDS counters; defer_cap / defer_cap_px: queue capacities, GF_X2_DEFER_CAP overrides both (tests of the full-queue path)
    uint32_t* d_defer_q = nullptr; uint4* d_defer_px = nullptr; unsigned* d_defer_count = nullptr;
    uint32_t defer_cap = 1u << 20, defer_cap_px = 1u << 20; unsigned long long filter_frames = 0;
    bool no_filter = false;
    int block_y = GF_BLOCK_Y, x2_block_y = 4;   // tuning knobs GF_BLOCK_Y / GF_X2_BLOCK_Y, read once per context at creation
    // preview overlays (overlay.cu), off unless gf_cuda_set_overlays: device copy of the drawing buffer, private copy of a DEVICE input
    int overlays = 0;
    uint8_t* h_drawing = nullptr; uint8_t* d_drawing = nullptr; size_t drawing_cap = 0;
    uint8_t* d_src_ovl = nullptr; size_t d_src_ovl_len = 0;
    // HOST multi-plane frames (gf_cuda_undistort_planes): one device staging pair per plane beyond what d_src / d_dst hold
    std::vector<uint8_t*> d_plane_src, d_plane_dst; std::vector<size_t> d_plane_src_len, d_plane_dst_len;
    uint2* d_coords = nullptr; size_t d_coords_len = 0;   // multi-plane mode: the frame's coordinate map
    KernelFn fn_shade = nullptr;
    unsigned long long aux_launches = 0;   // helper kernels (mesh widening, table scans): not counted by gf_cuda_launch_count
    unsigned long long x2_launches = 0;
    unsigned long long lean_launches = 0;
    cudaStream_t stream = nullptr;
    size_t max_rows = 0;
    Slot slots[kSlots];
    int next_slot = 0;
    uint8_t* d_src = nullptr; size_t d_src_len = 0;     // staging when buffers are HOST
    uint8_t* d_dst = nullptr; size_t d_dst_len = 0;
    size_t drawing_len = 0;
    unsigned long long launches = 0;
    std::string last_error;
};

namespace {

int fail(gf_cuda_ctx* ctx, int code, const std::string& msg) {
    g_last_error = msg;
    if (ctx) ctx->last_error = msg;
    return code;
}
int cuda_fail(gf_cuda_ctx* ctx, cudaError_t e, const char* what) {
    return fail(ctx, GF_ERR_CUDA, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call); } while (0)

bool pix_layout(int pixel_type, int* layout, int* bpp) {
    switch (pixel_type) {
    case GF_PIX_LUMA8:   *layout = LAY_1U8;  *bpp = 1;  return true;
    case GF_PIX_UV8:     *layout = LAY_2U8;  *bpp = 2;  return true;
    case GF_PIX_RGB8:    *layout = LAY_3U8;  *bpp = 3;  return true;
    case GF_PIX_RGBA8:
    case GF_PIX_BGRA8:   *layout = LAY_4U8;  *bpp = 4;  return true;
    case GF_PIX_LUMA16:  *layout = LAY_1U16; *bpp = 2;  return true;
    case GF_PIX_UV16:    *layout = LAY_2U16; *bpp = 4;  return true;
    case GF_PIX_RGB16:   *layout = LAY_3U16; *bpp = 6;  return true;
    case GF_PIX_RGBA16:
    case GF_PIX_AYUV16:  *layout = LAY_4U16; *bpp = 8;  return true;
    case GF_PIX_R32F:    *layout = LAY_1F32; *bpp = 4;  return true;
    case GF_PIX_RGBAF:   *layout = LAY_4F32; *bpp = 16; return true;
    case GF_PIX_RGBAF16: *layout = LAY_4F16; *bpp = 8;  return true;
    default: return false;
    }
}

KernelFn find_kernel(int lens, int digital, int layout, int interp, int lean) {
    switch (lens) {
    case GF_LENS_OPENCV_FISHEYE:     return gf_kernel_opencv_fisheye(digital, layout, interp, lean);
    case GF_LENS_OPENCV_STANDARD:    return gf_kernel_opencv_standard(digital, layout, interp, lean);
    case GF_LENS_POLY3:              return gf_kernel_poly3(digital, layout, interp, lean);
    case GF_LENS_POLY5:              return gf_kernel_poly5(digital, layout, interp, lean);
    case GF_LENS_PTLENS:             return gf_kernel_ptlens(digital, layout, interp, lean);
    case GF_LENS_INSTA360:           return gf_kernel_insta360(digital, layout, interp, lean);
    case GF_LENS_SONY:               return gf_kernel_sony(digital, layout, interp, lean);
    case GF_LENS_GENERIC_POLYNOMIAL: return gf_kernel_generic_polynomial(digital, layout, interp, lean);
    case GF_LENS_GOPRO:              return gf_kernel_gopro(digital, layout, interp, lean);
    default: return nullptr;
    }
}

const char* const kLensNames[GF_LENS_COUNT] = {
    "none", "opencv_fisheye", "opencv_standard", "poly3", "poly5", "ptlens", "insta360", "sony", "generic_polynomial",
    "gopro", "gopro_superview", "gopro_hyperview", "gopro_warp", "digital_stretch", "gopro6_superview" };

// process_pixels / OclWrapper::new validation (stabilization/mod.rs:613,636-640; opencl.rs:179; wgpu.rs:150)
int validate(gf_cuda_ctx* ctx, const gf_kernel_params* p, const gf_buffer_desc* in, const gf_buffer_desc* out, int bpp) {
    if (!p || !in || !out) return fail(ctx, GF_ERR_BAD_PARAMS, "null argument");
    if (in->height < 4 || out->height < 4 || p->height < 4 || p->output_height < 4)
        return fail(ctx, GF_ERR_SIZE_TOO_SMALL, "SizeTooSmall: height < 4");
    if (p->stride < 1 || p->output_stride < 1) return fail(ctx, GF_ERR_BAD_STRIDE, "InvalidStride: stride < 1");
    if (p->width > 16384 || p->output_width > 16384 || p->width < 1 || p->output_width < 1)
        return fail(ctx, GF_ERR_BAD_PARAMS, "width out of range (1..16384)");
    if (in->width > p->stride)         return fail(ctx, GF_ERR_BAD_STRIDE, "InvalidStride: input width > stride");
    if (out->width > p->output_stride) return fail(ctx, GF_ERR_BAD_STRIDE, "InvalidStride: output width > output_stride");
    if (p->stride != in->stride || p->output_stride != out->stride)
        return fail(ctx, GF_ERR_BAD_STRIDE, "InvalidStride: KernelParams stride differs from the buffer description");
    if (p->bytes_per_pixel != bpp) return fail(ctx, GF_ERR_BAD_PARAMS, "bytes_per_pixel does not match the pixel type");
    if (p->matrix_count < 1) return fail(ctx, GF_ERR_BAD_PARAMS, "matrix_count < 1");
    if ((in->kind != GF_BUF_HOST && in->kind != GF_BUF_DEVICE) || (out->kind != GF_BUF_HOST && out->kind != GF_BUF_DEVICE) || !in->ptr || !out->ptr)
        return fail(ctx, GF_ERR_BAD_PARAMS, "unsupported buffer source");
    // every tap the kernel may read must be inside the input buffer (Rust would panic on the slice index)
    const long long x0 = p->source_rect[0], y0 = p->source_rect[1], x1 = x0 + p->source_rect[2], y1 = y0 + p->source_rect[3];
    if (p->source_rect[2] > 0 && p->source_rect[3] > 0) {
        if (x0 < 0 || y0 < 0) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "source_rect has a negative origin");
        const unsigned long long last = (unsigned long long)(y1 - 1) * (unsigned long long)p->stride + (unsigned long long)x1 * (unsigned long long)bpp;
        if (last > in->len) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch input: source_rect exceeds the input buffer");
    }
    if (out->len == 0) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "empty output buffer");
    return GF_OK;
}

// map_coord's per-frame-uniform pieces (util.rs:144-147), same float operations as the reference evaluates per pixel
MapC make_map(float in_min, float in_max, float out_min, float out_max, float max_abs_int_coord) {
    MapC m;
    m.in_min = in_min;
    m.mul = out_max - out_min;
    m.div = in_max - in_min;
    m.rcp = 1.0f / m.div;
    m.add = out_min;
    const float ad = fabsf(m.div);
    m.fast_div = (std::isfinite(m.div) && ad >= 0x1p-40f && ad <= 0x1p40f) ? 1 : 0;
    // integer-valued x: (x - in_min) and (x - in_min) * mul are exact below 2^24, and exact / div == (x - in_min) when mul == div
    m.identity = (max_abs_int_coord >= 0.0f && m.mul == m.div && m.mul > 0.0f && in_min == truncf(in_min) &&
                  (max_abs_int_coord + fabsf(in_min)) * m.mul < 16777216.0f) ? 1 : 0;
    return m;
}

// "tame": zero, or finite with 2^-40 <= |v| <= 2^40 — the magnitudes for which the packed kernel's unguarded numerators are safe
inline bool tame(float v) { const float a = fabsf(v); return v == 0.0f || (a >= 0x1p-40f && a <= 0x1p40f); }
enum : uint32_t { TBL_WILD = 1u, TBL_IBIS = 2u };
uint32_t scan_tables_host(const float* m, size_t rows) {
    uint32_t f = 0;
    for (size_t r = 0; r < rows; ++r) {
        const float* p = m + r * GF_MATRIX_STRIDE;
        for (int i = 0; i < 9; ++i) if (!tame(p[i])) f |= TBL_WILD;
        for (int i = 9; i < 14; ++i) if (!(p[i] == 0.0f)) f |= TBL_IBIS;
    }
    return f;
}
// f32 mesh -> f64 once per frame (cpu_undistort.rs:539) + the per-frame constants of MeshAux, all on the device so that
// device-resident meshes never touch the host.  o has room for GF_MESH_MAX_LEN doubles followed by one MeshAux.
__device__ MapC make_map_dev(float in_min, float in_max, float out_min, float out_max) {
    MapC m;
    m.in_min = in_min; m.mul = out_max - out_min; m.div = in_max - in_min; m.rcp = 1.0f / m.div; m.add = out_min;
    const float ad = fabsf(m.div);
    m.fast_div = (isfinite(m.div) && ad >= 0x1p-40f && ad <= 0x1p40f) ? 1 : 0;
    m.identity = 0;
    return m;
}
__global__ void widen_mesh_kernel(const float* __restrict__ m, double* __restrict__ o, int n, float width_f, float height_f) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) o[i] = (double)m[i];
    if (i == 0 && n >= 9) {
        MeshAux* aux = reinterpret_cast<MeshAux*>(o + GF_MESH_MAX_LEN);
        const double size_y = (double)m[4];
        const double h = size_y / 8.0;
        aux->h = h; aux->inv_h = 1.0 / h; aux->three_inv_h = 3.0 * aux->inv_h; aux->h_over_3 = h / 3.0; aux->inv_3h = 1.0 / (3.0 * h);
        // `mesh[5] as f32` etc.: the f64 value is the widened f32, so the narrowing is the identity
        const float origin_x = m[5], origin_y = m[6], crop_w = m[7], crop_h = m[8];
        aux->to_crop_x  = make_map_dev(0.0f, width_f,  origin_x, origin_x + crop_w);
        aux->to_crop_y  = make_map_dev(0.0f, height_f, origin_y, origin_y + crop_h);
        aux->to_frame_x = make_map_dev(origin_x, origin_x + crop_w, 0.0f, width_f);
        aux->to_frame_y = make_map_dev(origin_y, origin_y + crop_h, 0.0f, height_f);
    }
}
// one block: every thread ORs its rows, the block reduces, thread 0 WRITES the verdict (no prior memset, no atomics on the word)
__global__ void __launch_bounds__(1024) scan_tables_kernel(const float* __restrict__ m, size_t rows, uint32_t* flags) {
    __shared__ unsigned warp_or[32];
    unsigned f = 0;
    const size_t n = rows * GF_MATRIX_STRIDE;
    for (size_t i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = m[i], a = fabsf(v);
        const unsigned col = (unsigned)(i % GF_MATRIX_STRIDE);
        if (col < 9u) { if (!(v == 0.0f || (a >= 0x1p-40f && a <= 0x1p40f))) f |= TBL_WILD; }
        else if (!(v == 0.0f)) f |= TBL_IBIS;
    }
    f = __reduce_or_sync(0xffffffffu, f);
    if ((threadIdx.x & 31u) == 0u) warp_or[threadIdx.x >> 5] = f;
    __syncthreads();
    if (threadIdx.x < 32u) {
        f = threadIdx.x < (blockDim.x >> 5) ? warp_or[threadIdx.x] : 0u;
        f = __reduce_or_sync(0xffffffffu, f);
        if (threadIdx.x == 0u) *flags = f;
    }
}

bool lens_noop(int lens, const gf_kernel_params* p) {
    const float* k = p->k;
    switch (lens) {
    case GF_LENS_OPENCV_FISHEYE:
    case GF_LENS_SONY:               return k[0] == 0.0f && k[1] == 0.0f && k[2] == 0.0f && k[3] == 0.0f;
    case GF_LENS_GENERIC_POLYNOMIAL: { for (int i = 0; i < 12; ++i) if (!(k[i] == 0.0f)) return false; return true; }
    case GF_LENS_GOPRO:              return k[1] == 0.0f;
    default: return false;
    }
}

// Everything the reference recomputes per pixel from per-frame constants (cpu_undistort.rs:421-528), computed once, on the
// host, with the same IEEE float operations (this TU is built with -ffp-contract=off; sin/cos come from gf_math.cuh, the
// same code the device runs).
void fill_uniforms(WarpArgs& A, const gf_cuda_ctx* ctx, const uint8_t* src, const uint8_t* dst) {
    const gf_kernel_params* p = &A.p;
    const int bpp = ctx->bpp;
    const int align = (bpp == 1 || bpp == 2 || bpp == 4 || bpp == 8 || bpp == 16) ? bpp : (bpp == 3 ? 1 : 2);
    uint32_t f = 0;
    if (p->matrix_count > 1) f |= F_RS;
    if ((p->flags & 16) == 16) f |= F_HRS;
    A.r_limit_sq = p->r_limit * p->r_limit;                                      // :521
    if (A.r_limit_sq > 0.0f) f |= F_RLIMIT;
    if (p->light_refraction_coefficient != 1.0f && p->light_refraction_coefficient > 0.0f) f |= F_REFRACT;
    if (A.mesh_len > 0) f |= F_MESH;
    if ((p->flags & 2) == 2 && ctx->digital_lens != GF_LENS_NONE) f |= F_DIGITAL;
    if (p->input_horizontal_stretch > 0.001f && p->input_horizontal_stretch != 1.0f) f |= F_HSTRETCH;
    if (p->input_vertical_stretch   > 0.001f && p->input_vertical_stretch   != 1.0f) f |= F_VSTRETCH;
    if (p->lens_correction_amount < 1.0f) f |= F_LCA;
    if (p->input_rotation != 0.0f) f |= F_INROT;
    if (p->background_mode == 1) f |= F_BG1;
    if (p->background_mode == 2) f |= F_BG2;
    if (p->background_mode == 3) f |= F_BG3;
    if ((p->flags & 1) == 1) f |= F_FIXRANGE;
    if ((p->flags & 4) == 4) f |= F_FILLBG;
    if (lens_noop(ctx->distortion_model, p)) f |= F_LENS_NOOP;
    if ((reinterpret_cast<uintptr_t>(src) % (uintptr_t)align) == 0 && (p->stride % align) == 0) f |= F_SRC_VEC;
    if ((f & F_SRC_VEC) && (reinterpret_cast<uintptr_t>(src) % 8u) == 0 && (p->stride % 8) == 0 && (A.src_len % 8ull) == 0) f |= F_SRC_VEC8;
    if ((reinterpret_cast<uintptr_t>(dst) % (uintptr_t)align) == 0 && (p->output_stride % align) == 0) f |= F_DST_VEC;
    if ((p->flags & 128) == 128) f |= F_FB_INV;
    if (p->plane_index == 0) f |= F_IS_Y;
    if (p->translation3d[0] != 0.0f || p->translation3d[1] != 0.0f || p->translation3d[2] != 0.0f) f |= F_T3D;
    const float maxv = ctx->bpp > 0 && (ctx->layout <= LAY_4U8) ? 255.0f : ((ctx->layout <= LAY_4U16) ? 65535.0f : 3.402823466e38f);
    if (!(p->pixel_value_limit >= maxv)) f |= F_PIXLIMIT;
    {   // magnitudes the packed kernel's fast paths rely on (otherwise the scalar lean kernel, which has no such assumptions, runs)
        bool wild = false;
        for (int i = 0; i < 12; ++i) if (!(std::isfinite(p->k[i]) && fabsf(p->k[i]) <= 0x1p40f)) wild = true;
        if (!(fabsf(p->translation2d[0]) < 0x1p19f && fabsf(p->translation2d[1]) < 0x1p19f)) wild = true;
        if (!(tame(p->f[0]) && tame(p->f[1]) && std::isfinite(p->c[0]) && std::isfinite(p->c[1]))) wild = true;
        // packed gopro lens: k1 is a divisor (paraxial guess of the Newton inversion) and the 89-degree cut-off is a literal
        if (ctx->distortion_model == GF_LENS_GOPRO && (!(tame(p->k[1]) && p->k[1] != 0.0f) || gf_tanf(1.5533f) != 0x1.c9315ap+5f)) wild = true;
        if (ctx->digital_lens == GF_LENS_GOPRO_WARP) for (int i = 0; i < 16; ++i) if (!(std::isfinite(p->digital_lens_params[i]) && fabsf(p->digital_lens_params[i]) <= 0x1p40f)) wild = true;
        if (wild) f |= F_WILD;
    }
    A.feat = f;

    for (int i = 0; i < 4; ++i) A.bg[i] = p->background[i] * p->max_pixel_value;  // :523
    const float factor = fmaxf(1.0f - p->lens_correction_amount, 0.001f);         // :526
    A.out_c[0] = (float)p->output_width / 2.0f; A.out_c[1] = (float)p->output_height / 2.0f;   // :527
    A.out_f[0] = p->f[0] / p->fov / factor;      A.out_f[1] = p->f[1] / p->fov / factor;        // :528

    A.width_f = (float)p->width; A.height_f = (float)p->height;
    A.frame_w = A.width_f; A.frame_h = A.height_f;
    A.rot_cos = 1.0f; A.rot_sin = 0.0f;
    if (p->input_rotation != 0.0f) {                                              // :485-489 (rotate_point :262-265)
        const float rotation = p->input_rotation * (3.14159274101257324f / 180.0f);
        A.rot_cos = gf_cosf(rotation); A.rot_sin = gf_sinf(rotation);
        const float fx = A.rot_cos * (A.width_f - 0.0f) - A.rot_sin * (A.height_f - 0.0f) + 0.0f;
        const float fy = A.rot_sin * (A.width_f - 0.0f) + A.rot_cos * (A.height_f - 0.0f) + 0.0f;
        A.frame_w = rs_round(fabsf(fx)); A.frame_h = rs_round(fabsf(fy));
    }
    A.omap_x = make_map((float)p->output_rect[0], (float)(p->output_rect[0] + p->output_rect[2]), 0.0f, (float)p->output_width,  (float)A.out_cols);
    A.omap_y = make_map((float)p->output_rect[1], (float)(p->output_rect[1] + p->output_rect[3]), 0.0f, (float)p->output_height, (float)A.out_rows);
    A.smap_x = make_map(0.0f, A.frame_w, (float)p->source_rect[0], (float)(p->source_rect[0] + p->source_rect[2]), -1.0f);
    A.smap_y = make_map(0.0f, A.frame_h, (float)p->source_rect[1], (float)(p->source_rect[1] + p->source_rect[3]), -1.0f);
    A.rs_lim = (p->flags & 16) == 16 ? p->width : p->height;
    const float lim = p->pixel_value_limit;
    A.u8_limit = (lim != lim) ? 255 : (lim < 0.0f ? 0 : (lim >= 255.0f ? 255 : (int)lim));
    A.src_rect[0] = p->source_rect[0]; A.src_rect[1] = p->source_rect[1];
    A.src_rect[2] = p->source_rect[0] + p->source_rect[2]; A.src_rect[3] = p->source_rect[1] + p->source_rect[3];
    A.interior_span[0] = A.src_rect[2] - 2 - A.src_rect[0]; A.interior_span[1] = A.src_rect[3] - 2 - A.src_rect[1];
    if (A.interior_span[0] < 0 || A.interior_span[1] < 0 || A.interior_span[0] >= (1 << 17) || A.interior_span[1] >= (1 << 17) || A.rs_lim >= (1 << 22)) { A.interior_span[0] = 0; A.interior_span[1] = 0; A.feat |= F_WILD; }   // no interior at all
    // source-rect maps of the packed kernel (see map_apply_x2): in_min == 0, moderate non-zero scale, divisor <= 2^20, |c| >= 2^-10,
    // source rect inside [0, 2^16) so that every coordinate the rounding shortcut cannot represent is outside the image anyway
    auto smap_ok = [](const MapC& m) { return m.fast_div && m.in_min == 0.0f && m.mul != 0.0f && tame(m.mul) && m.div > 0.0f && m.div <= 0x1p20f && std::isfinite(m.add) && fabsf(m.add) <= 0x1p16f; };
    if (!(smap_ok(A.smap_x) && smap_ok(A.smap_y) && fabsf(p->c[0]) >= 0x1p-10f && fabsf(p->c[1]) >= 0x1p-10f &&
          A.src_rect[0] >= 0 && A.src_rect[1] >= 0 && A.src_rect[2] <= (1 << 16) && A.src_rect[3] <= (1 << 16))) A.feat |= F_WILD;
    // pixel-index maps of the packed kernel: identity, or a positive moderate scale (map_apply_int_lean in warp_kernel_x2.cuh)
    auto int_map_ok = [](const MapC& m) {
        return m.identity || (m.fast_div && m.mul > 0.0f && m.div > 0.0f && tame(m.mul) && std::isfinite(m.add) && fabsf(m.in_min) <= 0x1p20f);
    };
    if (!(int_map_ok(A.omap_x) && int_map_ok(A.omap_y))) A.feat |= F_WILD;
    // integer prologue of the packed kernel: identity maps -> opx = (x - in_min) + add with integer in_min / add
    A.hot.rect[0] = A.src_rect[0]; A.hot.rect[1] = A.src_rect[1]; A.hot.rect[2] = A.interior_span[0]; A.hot.rect[3] = A.interior_span[1];
    if (A.omap_x.identity && A.omap_y.identity && A.omap_x.add == truncf(A.omap_x.add) && A.omap_y.add == truncf(A.omap_y.add) &&
        fabsf(A.omap_x.add) < 0x1p20f && fabsf(A.omap_y.add) < 0x1p20f && fabsf(A.omap_x.in_min) < 0x1p20f && fabsf(A.omap_y.in_min) < 0x1p20f) {
        const int bpp = ctx->bpp;
        A.hot.x_off = (int)A.omap_x.add - (int)A.omap_x.in_min; A.hot.y_off = (int)A.omap_y.add - (int)A.omap_y.in_min;
        // :551 — opx >= 0 && (opx as i32) < output_width  <=>  0 <= x + x_off < output_width
        A.hot.x0 = std::max(0, -A.hot.x_off); A.hot.x1 = std::min(A.out_cols, p->output_width - A.hot.x_off);
        A.hot.y0 = std::max(0, -A.hot.y_off); A.hot.y1 = std::min(A.out_rows, p->output_height - A.hot.y_off);
        A.hot.full_rows = (int)std::min<size_t>(A.dst_len / (size_t)p->output_stride, (size_t)A.out_rows);
        const size_t tail = A.dst_len - (size_t)A.hot.full_rows * (size_t)p->output_stride;
        A.hot.last_cols = (A.hot.full_rows < A.out_rows) ? (int)std::min<size_t>(tail / (size_t)bpp, (size_t)A.out_cols) : 0;
        A.feat |= F_INTPRO;
    }
}

} // namespace

extern "C" {

GF_API int gf_cuda_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { g_last_error = std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e); (void)cudaGetLastError(); return 0; }
    return n;
}

GF_API int gf_cuda_device_name(int device, char* buf, size_t buf_len) {
    if (!buf || buf_len == 0) return GF_ERR_BAD_PARAMS;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return fail(nullptr, GF_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e)); }
    snprintf(buf, buf_len, "[CUDA] %s", prop.name);      // listed like "[OpenCL] ..." / "[wgpu] ..." (stabilization/mod.rs:399-410)
    return GF_OK;
}

GF_API int gf_cuda_supports(const gf_buffer_desc* in, const gf_buffer_desc* out) {
    if (!in || !out) return 0;
    const bool i = in->kind == GF_BUF_HOST || in->kind == GF_BUF_DEVICE;
    const bool o = out->kind == GF_BUF_HOST || out->kind == GF_BUF_DEVICE;
    return (i && o) ? 1 : 0;
}

GF_API const char* gf_cuda_version(void) { return "gyroflow-b200 0.1 (sm_100a)"; }
GF_API size_t gf_abi_struct_size(int which) {
    switch (which) {
    case 0: return sizeof(gf_kernel_params);  case 1: return sizeof(gf_buffer_desc);    case 2: return sizeof(gf_compute_params);
    case 3: return sizeof(gf_camera_stab);    case 4: return sizeof(gf_keyframe_track); case 5: return sizeof(gf_stab_config);
    case 6: return sizeof(gf_queue_config);   case 7: return sizeof(gf_lens_data);
    case 8: return sizeof(gf_mesh_f64);       case 9: return sizeof(gf_plane_spec);
    default: return 0;
    }
}
GF_API const char* gf_cuda_backend_name(void) { return "CUDA"; }

GF_API int gf_lens_from_name(const char* id) {
    if (id) for (int i = 1; i < GF_LENS_COUNT; ++i) if (!strcmp(id, kLensNames[i])) return i;
    return GF_LENS_OPENCV_FISHEYE;     // DistortionModel::from_name falls back to the default model
}
GF_API const char* gf_lens_name(int lens_id) { return (lens_id >= 0 && lens_id < GF_LENS_COUNT) ? kLensNames[lens_id] : nullptr; }
GF_API int gf_pixel_bytes(int pixel_type) { int l, b; return pix_layout(pixel_type, &l, &b) ? b : 0; }
GF_API int gf_combo_supported(int pixel_type, int distortion_model, int digital_lens, int interpolation) {
    int l, b;
    if (!pix_layout(pixel_type, &l, &b)) return 0;
    return find_kernel(distortion_model, digital_lens, l, interpolation, 0) != nullptr ? 1 : 0;
}

GF_API int gf_cuda_create(gf_cuda_ctx** out_ctx, int device, const gf_kernel_params* params, int pixel_type,
                          int distortion_model, int digital_lens,
                          const gf_buffer_desc* in, const gf_buffer_desc* out, size_t drawing_len) {
    if (!out_ctx) return fail(nullptr, GF_ERR_BAD_PARAMS, "out_ctx is null");
    *out_ctx = nullptr;
    int layout = 0, bpp = 0;
    if (!pix_layout(pixel_type, &layout, &bpp)) return fail(nullptr, GF_ERR_BAD_PARAMS, "unknown pixel type");
    { int rc = validate(nullptr, params, in, out, bpp); if (rc != GF_OK) return rc; }
    KernelFn fn = find_kernel(distortion_model, digital_lens, layout, params->interpolation, 0);
    KernelFn fn_lean = find_kernel(distortion_model, digital_lens, layout, params->interpolation, 1);
    const bool no_x2 = getenv("GF_DISABLE_X2") != nullptr;      // read per context (tests flip it between contexts)
    const bool no_filter = getenv("GF_DISABLE_FILTER") != nullptr;
    KernelFn fn_x2 = no_x2 ? nullptr : find_kernel(distortion_model, digital_lens, layout, params->interpolation, 2);
    if (!fn) return fail(nullptr, GF_ERR_UNSUPPORTED_COMBO, "no kernel compiled for this (lens, digital lens, pixel type, interpolation)");

    gf_cuda_ctx* ctx = new gf_cuda_ctx();
    ctx->device = device; ctx->pixel_type = pixel_type; ctx->distortion_model = distortion_model; ctx->digital_lens = digital_lens;
    ctx->interpolation = params->interpolation; ctx->layout = layout; ctx->bpp = bpp; ctx->fn = fn; ctx->fn_lean = fn_lean; ctx->fn_x2 = fn_x2; ctx->fn_shade = gf_shade_kernel(layout);
    if (!no_x2) ctx->fn_x2c = find_kernel(distortion_model, digital_lens, layout, GF_INTERP_BILINEAR, 4);
    if (!no_x2) ctx->fn_x2f = find_kernel(distortion_model, digital_lens, layout, params->interpolation, 5);
    ctx->width = params->width; ctx->height = params->height; ctx->output_width = params->output_width; ctx->output_height = params->output_height;
    ctx->drawing_len = drawing_len; ctx->no_filter = no_filter;
    { const char* e = getenv("GF_BLOCK_Y"); const int v = e ? atoi(e) : GF_BLOCK_Y; ctx->block_y = (v == 1 || v == 2 || v == 4 || v == 8) ? v : GF_BLOCK_Y; }
    { const char* e = getenv("GF_X2_BLOCK_Y"); const int v = e ? atoi(e) : 4; ctx->x2_block_y = (v == 1 || v == 2 || v == 4 || v == 8) ? v : 4; }
    { const char* e = getenv("GF_X2_DEFER_CAP"); const long v = e ? atol(e) : 0; if (v > 0 && v < (1l << 20)) ctx->defer_cap = ctx->defer_cap_px = (uint32_t)v; }
    auto bail = [&](int rc) { std::string m = ctx->last_error; gf_cuda_destroy(ctx); g_last_error = m; return rc; };

    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { cuda_fail(ctx, e, "cudaSetDevice"); return bail(GF_ERR_CUDA); }
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { cuda_fail(ctx, e, "cudaStreamCreate"); return bail(GF_ERR_CUDA); }
    // matrices: 14 * max(W, H) f32 (rows = height, or width for horizontal rolling shutter) — opencl.rs:268, wgpu.rs:260
    size_t rows = (size_t)std::max(std::max(params->width, params->height), std::max(params->output_width, params->output_height));
    rows = std::max(rows, (size_t)params->matrix_count);
    ctx->max_rows = rows;
    {
        const uint32_t words[2] = { 0u, 1u };
        if ((e = cudaMalloc(&ctx->d_const_flags, sizeof(words))) != cudaSuccess ||
            (e = cudaMemcpy(ctx->d_const_flags, words, sizeof(words), cudaMemcpyHostToDevice)) != cudaSuccess ||
            (e = cudaMalloc(&ctx->d_vflags, sizeof(uint32_t))) != cudaSuccess) { cuda_fail(ctx, e, "table-verdict words"); return bail(GF_ERR_CUDA); }
    }
    for (int s = 0; s < kSlots; ++s) {
        Slot& sl = ctx->slots[s];
        if ((e = cudaMallocHost(&sl.h_mat, rows * GF_MATRIX_STRIDE * sizeof(float))) != cudaSuccess ||
            (e = cudaMalloc(&sl.d_mat, rows * GF_MATRIX_STRIDE * sizeof(float))) != cudaSuccess ||
            (e = cudaMallocHost(&sl.h_mesh, GF_MESH_MAX_LEN * sizeof(float))) != cudaSuccess ||
            (e = cudaMalloc(&sl.d_mesh, GF_MESH_MAX_LEN * sizeof(float))) != cudaSuccess ||
            (e = cudaMalloc(&sl.d_mesh64, GF_MESH_MAX_LEN * sizeof(double) + sizeof(MeshAux))) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming)) != cudaSuccess) {
            cuda_fail(ctx, e, "table staging allocation"); return bail(GF_ERR_CUDA);
        }
    }
    if (in->kind == GF_BUF_HOST)  { if ((e = cudaMalloc(&ctx->d_src, in->len)) != cudaSuccess)  { cuda_fail(ctx, e, "cudaMalloc(src staging)"); return bail(GF_ERR_CUDA); } ctx->d_src_len = in->len; }
    if (out->kind == GF_BUF_HOST) { if ((e = cudaMalloc(&ctx->d_dst, out->len)) != cudaSuccess) { cuda_fail(ctx, e, "cudaMalloc(dst staging)"); return bail(GF_ERR_CUDA); } ctx->d_dst_len = out->len; }
    *out_ctx = ctx;
    return GF_OK;
}

GF_API void gf_cuda_destroy(gf_cuda_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int s = 0; s < kSlots; ++s) {
        Slot& sl = ctx->slots[s];
        if (sl.h_mat) cudaFreeHost(sl.h_mat);
        if (sl.d_mat) cudaFree(sl.d_mat);
        if (sl.h_mesh) cudaFreeHost(sl.h_mesh);
        if (sl.d_mesh) cudaFree(sl.d_mesh);
        if (sl.d_mesh64) cudaFree(sl.d_mesh64);
        if (sl.done) cudaEventDestroy(sl.done);
    }
    if (ctx->d_src) cudaFree(ctx->d_src);
    if (ctx->d_dst) cudaFree(ctx->d_dst);
    if (ctx->d_vflags) cudaFree(ctx->d_vflags);
    if (ctx->d_const_flags) cudaFree(ctx->d_const_flags);
    for (uint8_t* q : ctx->d_plane_src) if (q) cudaFree(q);
    for (uint8_t* q : ctx->d_plane_dst) if (q) cudaFree(q);
    if (ctx->h_drawing) cudaFreeHost(ctx->h_drawing);
    if (ctx->d_drawing) cudaFree(ctx->d_drawing);
    if (ctx->d_src_ovl) cudaFree(ctx->d_src_ovl);
    if (ctx->d_defer_q) cudaFree(ctx->d_defer_q);
    if (ctx->d_defer_px) cudaFree(ctx->d_defer_px);
    if (ctx->d_defer_count) cudaFree(ctx->d_defer_count);
    if (ctx->d_coords) cudaFree(ctx->d_coords);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    (void)cudaGetLastError();
    delete ctx;
}

// Filtered rolling-shutter pre-pass (warp_kernel_x2.cuh, Lens2<opencv_fisheye>::approx_v): the host side of its contract.
// The certificate |tv_approx - tv_exact| <= rho |tv - c_y| + 2^-22 |tv| assumes that the polynomial s = 1 + k0 t^2 + k1 t^4 + k2 t^6 +
// k3 t^8 stays within [3/4, 5/4] (its rounding error and its sensitivity to the error of t are then bounded, DESIGN.md §4):
// a_cap = tan^2(t_cap) with t_cap the largest angle (<= 1.55 rad) for which sum |k_i| t^(2i+2) <= 1/4.  Returns 0 when the lens is too
// strongly curved for the filter to be worth it (t_cap < 0.5 rad).
static float filter_a_cap(const float* k) {
    auto B = [&](double t) { const double t2 = t * t; return t2 * (fabs((double)k[0]) + t2 * (fabs((double)k[1]) + t2 * (fabs((double)k[2]) + t2 * fabs((double)k[3])))); };
    for (int i = 0; i < 4; ++i) if (!std::isfinite(k[i])) return 0.0f;
    double lo = 0.0, hi = 1.55;
    if (B(hi) > 0.25) { for (int it = 0; it < 60; ++it) { const double mid = 0.5 * (lo + hi); if (B(mid) <= 0.25) lo = mid; else hi = mid; } }
    else lo = hi;
    if (lo < 0.5) return 0.0f;
    const double a = tan(lo) * tan(lo);
    return (float)std::min(a * 0.999, 16000.0);                 // stay inside the table (r^2 < 2^14) and below the exact bound
}

// Which kernel renders a frame with these uniforms?  Shared by run_warp and gf_cuda_plan (the host-only query the CPU tests use).
enum { PLAN_GENERAL = 0, PLAN_LEAN = 1, PLAN_PACKED = 2, PLAN_PACKED_TRUSTED = 3, PLAN_TWO_PASS = 0x10 };
static int select_variant(bool has_lean, bool has_packed, int ctx_digital_lens, const WarpArgs& A, uint32_t table_flags, bool two_pass, int n_maps) {
    // lean instantiation iff no general-only feature is on, vector access is legal, and the digital-lens flag matches the template
    const bool lean_ok = has_lean && (A.feat & F_GENERAL_ONLY) == 0 && (A.feat & F_LEAN_REQUIRED) == F_LEAN_REQUIRED &&
                         (((A.feat & F_DIGITAL) != 0) == (ctx_digital_lens != GF_LENS_NONE));
    // packed kernel: the trusted code path runs when the table's verdict word is 0 (host scan of host tables, or the device word the
    // table's producer / gf_cuda_scan_tables_dev wrote); table_flags here is what the HOST knows (non-zero = unknown or guarded)
    // (two-pass: the coordinate-writing variant, except for EWA whose probe positions only the scalar kernels evaluate)
    const bool packed_ok = lean_ok && has_packed && (A.feat & F_WILD) == 0 && !(two_pass && n_maps != 1);
    const int v = packed_ok ? (table_flags == 0 ? PLAN_PACKED_TRUSTED : PLAN_PACKED) : (lean_ok ? PLAN_LEAN : PLAN_GENERAL);
    return v | (two_pass ? PLAN_TWO_PASS : 0);
}

// `more_planes` > 0: multi-plane mode — in/out/p are arrays of 1 + more_planes planes that share one geometry (checked by the caller);
// the coordinates are computed once (pass 1, into ctx->d_coords) and every plane is then sampled from them (pass 2).
static int run_warp(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out, const gf_kernel_params* p,
                    const float* matrices, size_t matrix_rows, const float* mesh, size_t mesh_len,
                    bool tables_on_device, void* cu_stream, bool sync_host = true, size_t more_planes = 0, bool coord_only = false,
                    const uint32_t* table_flags_dev = nullptr, uint64_t* checksum_dev = nullptr,
                    const uint8_t* drawing = nullptr, size_t drawing_len = 0) {
    if (!ctx) return fail(nullptr, GF_ERR_BAD_PARAMS, "ctx is null");
    { int rc = validate(ctx, p, in, out, ctx->bpp); if (rc != GF_OK) return rc; }
    if (!matrices) return fail(ctx, GF_ERR_NO_DATA, "NoStabilizationData: matrices is null");
    if (p->width != ctx->width || p->height != ctx->height || p->output_width != ctx->output_width || p->output_height != ctx->output_height)
        return fail(ctx, GF_ERR_SIZE_MISMATCH, "SizeMismatch: KernelParams size differs from the size this context was created for");
    if (p->interpolation != ctx->interpolation)
        return fail(ctx, GF_ERR_UNSUPPORTED_COMBO, "interpolation differs from the one this context was created for");
    if ((size_t)p->matrix_count > matrix_rows) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch matrices: matrix_count > rows supplied");
    if (!tables_on_device && matrix_rows > ctx->max_rows) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch matrices");
    if (mesh_len > GF_MESH_MAX_LEN) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch buf_mesh_data");
    if (mesh_len > 0 && !mesh) return fail(ctx, GF_ERR_BAD_PARAMS, "mesh is null");
    if (mesh_len > 0 && mesh_len < 9) return fail(ctx, GF_ERR_BAD_PARAMS, "mesh shorter than its 9-value header (the reference would index out of bounds)");
    if (in->kind == GF_BUF_HOST && in->len > ctx->d_src_len)   return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch input");
    if (out->kind == GF_BUF_HOST && out->len > ctx->d_dst_len) return fail(ctx, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch output");
    if (tables_on_device && (reinterpret_cast<uintptr_t>(matrices) & 7u)) return fail(ctx, GF_ERR_BAD_PARAMS, "device matrices must be 8-byte aligned");

    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = cu_stream ? (cudaStream_t)cu_stream : ctx->stream;
    ctx->last_stream = st;

    WarpArgs A;
    memset(&A, 0, sizeof(A));
    A.p = *p;
    uint32_t table_flags = TBL_WILD;       // unknown device tables are not trusted until validated
    const bool use_slot = !tables_on_device || mesh_len > 0;   // device tables still need a slot for the widened mesh
    Slot& sl = ctx->slots[ctx->next_slot];
    if (use_slot) {
        ctx->next_slot = (ctx->next_slot + 1) % kSlots;
        CK(cudaEventSynchronize(sl.done));                     // the slot's previous frame has consumed its tables
    }
    if (tables_on_device) {
        // the verdict travels with the data: a device word written on this stream (or ordered before it) by whoever produced the table
        A.table_flags = table_flags_dev ? table_flags_dev : ctx->d_const_flags + 1;
        A.matrices = matrices;
        A.mesh = mesh_len ? mesh : nullptr;
    } else {
        memcpy(sl.h_mat, matrices, (size_t)p->matrix_count * GF_MATRIX_STRIDE * sizeof(float));
        table_flags = scan_tables_host(sl.h_mat, (size_t)p->matrix_count);
        A.table_flags = ctx->d_const_flags + (table_flags ? 1 : 0);
        CK(cudaMemcpyAsync(sl.d_mat, sl.h_mat, (size_t)p->matrix_count * GF_MATRIX_STRIDE * sizeof(float), cudaMemcpyHostToDevice, st));
        A.matrices = sl.d_mat;
        if (mesh_len) {
            memcpy(sl.h_mesh, mesh, mesh_len * sizeof(float));
            CK(cudaMemcpyAsync(sl.d_mesh, sl.h_mesh, mesh_len * sizeof(float), cudaMemcpyHostToDevice, st));
            A.mesh = sl.d_mesh;
        }
        // recorded after the launch below
    }
    A.mesh_len = (int)mesh_len;
    if (mesh_len) {                                            // cpu_undistort.rs:539 — `mesh_data.iter().map(|x| *x as f64)`, once per frame
        widen_mesh_kernel<<<(unsigned)((mesh_len + 255) / 256), 256, 0, st>>>(A.mesh, sl.d_mesh64, (int)mesh_len, (float)p->width, (float)p->height);
        CK(cudaGetLastError());
        A.mesh64 = sl.d_mesh64; A.mesh_aux = reinterpret_cast<const MeshAux*>(sl.d_mesh64 + GF_MESH_MAX_LEN); ctx->aux_launches++;
    }

    const uint8_t* src = (const uint8_t*)in->ptr;
    uint8_t* dst = (uint8_t*)out->ptr;
    if (in->kind == GF_BUF_HOST) {                             // opencl.rs:359 `self.src.write(buffer)`
        nvtxRangePushA("gf_h2d_frame");
        cudaError_t e_h2d = cudaMemcpyAsync(ctx->d_src, in->ptr, in->len, cudaMemcpyHostToDevice, st);
        nvtxRangePop();
        CK(e_h2d);
        src = ctx->d_src;
    }
    // Does the kernel write every pixel of [0,w) x [0,h)?  (output_rect == whole buffer == output size: the bounds test of
    // cpu_undistort.rs:551 then passes everywhere.)  If so only those bytes travel back; otherwise the untouched pixels
    // must keep their previous content, like on the CPU path, so the buffer is uploaded first.
    const bool full_cover = p->output_rect[0] == 0 && p->output_rect[1] == 0 && p->output_rect[2] == out->width && p->output_rect[3] == out->height &&
                            out->width == p->output_width && out->height == p->output_height && (p->flags & 4) == 0 &&
                            (size_t)out->height * (size_t)p->output_stride <= out->len + (size_t)(p->output_stride - out->width * ctx->bpp);
    if (out->kind == GF_BUF_HOST) {
        if (!full_cover) CK(cudaMemcpyAsync(ctx->d_dst, out->ptr, out->len, cudaMemcpyHostToDevice, st));
        dst = ctx->d_dst;
    }
    // preview overlays, input stage: drawing entries with stage bit 0 are drawn onto the device copy of the input
    const uint8_t* drawing_dev = nullptr;
    int ovl_count = 0, ovl_scalar = 0;
    if (ctx->overlays && more_planes == 0 && !coord_only) {
        ovl_count = ctx->layout <= LAY_4U8 ? ctx->layout + 1 : (ctx->layout <= LAY_4U16 ? ctx->layout - LAY_1U16 + 1 : (ctx->layout == LAY_1F32 ? 1 : 4));
        ovl_scalar = ctx->layout <= LAY_4U8 ? 0 : (ctx->layout <= LAY_4U16 ? 1 : (ctx->layout == LAY_4F16 ? 3 : 2));
        bool any_input_stage = false;
        if ((p->flags & GF_FLAG_DRAWING_ENABLED) && drawing && drawing_len) {
            if (drawing_len > ctx->drawing_cap) {
                CK(cudaStreamSynchronize(st));
                for (uint8_t* q : ctx->d_plane_src) if (q) cudaFree(q);
    for (uint8_t* q : ctx->d_plane_dst) if (q) cudaFree(q);
    if (ctx->h_drawing) cudaFreeHost(ctx->h_drawing);
                if (ctx->d_drawing) cudaFree(ctx->d_drawing);
                ctx->h_drawing = nullptr; ctx->d_drawing = nullptr; ctx->drawing_cap = 0;
                CK(cudaMallocHost(&ctx->h_drawing, drawing_len));
                CK(cudaMalloc(&ctx->d_drawing, drawing_len));
                ctx->drawing_cap = drawing_len;
            } else {
                CK(cudaStreamSynchronize(st));                 // the previous frame's upload has left the pinned copy
            }
            for (size_t i = 0; i < drawing_len; ++i) { const uint8_t d = drawing[i]; ctx->h_drawing[i] = d; any_input_stage |= (d != 0 && (d & 1u) == 0u); }
            CK(cudaMemcpyAsync(ctx->d_drawing, ctx->h_drawing, drawing_len, cudaMemcpyHostToDevice, st));   // opencl.rs: buf_drawing.write(drawing_buffer)
            drawing_dev = ctx->d_drawing;
        }
        if (any_input_stage) {
            if (in->kind == GF_BUF_DEVICE) {                   // never draw into the caller's buffer: private copy
                if (in->len > ctx->d_src_ovl_len) {
                    if (ctx->d_src_ovl) { CK(cudaStreamSynchronize(st)); cudaFree(ctx->d_src_ovl); ctx->d_src_ovl = nullptr; ctx->d_src_ovl_len = 0; }
                    CK(cudaMalloc(&ctx->d_src_ovl, in->len)); ctx->d_src_ovl_len = in->len;
                }
                CK(cudaMemcpyAsync(ctx->d_src_ovl, in->ptr, in->len, cudaMemcpyDeviceToDevice, st));
                src = ctx->d_src_ovl;
            }
            if (gf_internal_draw_overlays((void*)st, const_cast<uint8_t*>(src), in->len, in->width, in->height, p->stride, p, ovl_count, ovl_scalar, 1,
                                          drawing_dev, drawing_len) != GF_OK) return fail(ctx, GF_ERR_CUDA, "overlay kernel (input stage) failed");
            ctx->aux_launches++;
        }
    }
    A.src = src; A.dst = dst; A.src_len = in->len; A.dst_len = out->len;
    const int bpp = ctx->bpp;
    A.out_rows = (int)((out->len + (size_t)p->output_stride - 1) / (size_t)p->output_stride);
    A.out_cols = p->output_stride / bpp;
    fill_uniforms(A, ctx, src, dst);

    const int sby = ctx->block_y;
    const dim3 block(GF_BLOCK_X, sby);
    const dim3 grid((A.out_cols + GF_BLOCK_X - 1) / GF_BLOCK_X, (A.out_rows + sby - 1) / sby);
    if (grid.x == 0 || grid.y == 0 || grid.y > 65535) return fail(ctx, GF_ERR_BAD_PARAMS, "output buffer geometry out of range");
    // Two-pass mode: coordinates into a device map (pass 1), then sampling from the map (pass 2, shade_from_coords_kernel).  Used for
    // multi-plane frames, for every resampler other than bilinear (so that the 16/64-tap and EWA code lives in 11 sampling kernels
    // instead of every lens instantiation) and for ST maps (pass 1 only).  EWA needs three coordinate maps (pixel + two probes).
    const bool ewa = p->interpolation > 8;
    const bool two_pass = more_planes > 0 || coord_only || p->interpolation != GF_INTERP_BILINEAR;
    const int n_maps = (ewa && !coord_only) ? 3 : 1;
    const size_t map_len = (size_t)A.out_cols * (size_t)A.out_rows;
    if (two_pass) {
        if (!ctx->fn_shade && !coord_only) return fail(ctx, GF_ERR_UNSUPPORTED_COMBO, "no sampling kernel for this pixel layout");
        const size_t need = map_len * (size_t)n_maps;
        if (need > ctx->d_coords_len) {
            if (ctx->d_coords) { CK(cudaStreamSynchronize(st)); cudaFree(ctx->d_coords); ctx->d_coords = nullptr; ctx->d_coords_len = 0; }
            CK(cudaMalloc(&ctx->d_coords, need * sizeof(uint2)));
            ctx->d_coords_len = need;
        }
        A.coord_out = ctx->d_coords;
    }
    nvtxRangePushA("gf_warp_launch");
    struct NvtxPop { ~NvtxPop() { nvtxRangePop(); } } nvtx_pop_;
    const bool has_packed = two_pass ? (ctx->fn_x2c != nullptr) : (ctx->fn_x2 != nullptr);
    const int variant = select_variant(ctx->fn_lean != nullptr, has_packed, ctx->digital_lens, A, table_flags, two_pass, n_maps) & 0xf;
    const bool lean_ok = variant != PLAN_GENERAL;
    KernelFn x2 = (variant == PLAN_PACKED_TRUSTED || variant == PLAN_PACKED) ? (two_pass ? ctx->fn_x2c : ctx->fn_x2) : nullptr;
    // Packed-kernel launches use programmatic stream serialization: the grid may be scheduled while the previous kernel on the stream
    // (the frame's producer kernel, the previous frame's tail, ...) is still draining; every CTA executes griddepcontrol.wait before it
    // touches memory, so the dependency itself is unchanged and only the kernel-to-kernel launch gap disappears.
    auto launch_pdl = [&](KernelFn fn, dim3 g, dim3 b, const WarpArgs& args) -> cudaError_t {
        cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = g; cfg.blockDim = b; cfg.dynamicSmemBytes = 0; cfg.stream = st;      // 0 bytes: f32x2.cuh's opaque zero depends on it
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        void* kargs[1] = { (void*)&args };
        return cudaLaunchKernelExC(&cfg, (const void*)fn, kargs);
    };
    if (lean_ok && x2) {
        // 32 x 4 threads (4 x 8 output rows... 32 x 8 pixels) per block measured 2 % faster than 32 x 8 threads (finer tail); GF_X2_BLOCK_Y overrides
        const int by = ctx->x2_block_y;
        const dim3 block2(GF_BLOCK_X, by), grid2(grid.x, (A.out_rows + 2 * by - 1) / (2 * by));
        // filtered pre-pass: fisheye without a digital lens, rolling shutter on, geometry that fits the queue's 16 + 16 bit entries
        const float a_cap = (ctx->distortion_model == GF_LENS_OPENCV_FISHEYE && ctx->digital_lens == GF_LENS_NONE && (A.feat & F_RS) && !ctx->no_filter &&
                             A.out_cols <= 65536 && A.out_rows <= 131072 && (two_pass || ctx->fn_x2f) &&
                             (tables_on_device || table_flags == 0)) ? filter_a_cap(p->k) : 0.0f;      // host tables known to be wild / IBIS: guarded path, no tail launch
        if (a_cap > 0.0f) {
            if (!ctx->d_defer_q) {
                // 1 M pairs (4 MB, a quarter of a 4K frame's pairs) and 1 M pixels (16 MB, an eighth of a 4K frame); a full queue costs
                // the frame a second, exact rendering in the tail launch (COORD frames: the pairs past the end take the exact pre-pass inline)
                CK(cudaMalloc(&ctx->d_defer_q, (size_t)ctx->defer_cap * sizeof(uint32_t)));
                CK(cudaMalloc(&ctx->d_defer_px, (size_t)ctx->defer_cap_px * sizeof(uint4)));
                CK(cudaMalloc(&ctx->d_defer_count, 2 * GF_FLT_WORDS * sizeof(unsigned)));
                CK(cudaMemsetAsync(ctx->d_defer_count, 0, 2 * GF_FLT_WORDS * sizeof(unsigned), st));
            }
            const unsigned cur = (unsigned)(ctx->filter_frames & 1ull);
            ctx->filter_frames++;
            A.feat |= F_FILTER;
            A.flt.q = ctx->d_defer_q; A.flt.cap = ctx->defer_cap;
            A.flt.qpx = ctx->d_defer_px; A.flt.cap_px = ctx->defer_cap_px;
            A.flt.count = ctx->d_defer_count + cur * GF_FLT_WORDS; A.flt.count_next = ctx->d_defer_count + (cur ^ 1u) * GF_FLT_WORDS;
            A.flt.rho = 0x1p-17f; A.flt.a_cap = a_cap; A.flt.tail = 0;
            CK(launch_pdl(two_pass ? x2 : ctx->fn_x2f, grid2, block2, A)); ctx->x2_launches++;
            A.flt.tail = 1;                                            // the deferred pairs and pixels; also re-arms the other counters
            // one thread per deferred entry for up to 2 % of a 4K frame's pairs in a single wave of tiny blocks (idle blocks exit at once);
            // more entries than threads are covered by the grid-stride loop
            CK(launch_pdl(x2, dim3(148 * 16, 1), block2, A));
            ctx->launches++;
        } else {
            CK(launch_pdl(x2, grid2, block2, A)); ctx->x2_launches++;
        }
    }
    else {
        for (int mi = 0; mi < n_maps; ++mi) {                  // one launch, or three for EWA (pixel, x-probe, y-probe)
            if (two_pass) { A.coord_out = ctx->d_coords + (size_t)mi * map_len; A.coord_shift = mi; }
            if (lean_ok) { ctx->fn_lean<<<grid, block, 0, st>>>(A); ctx->lean_launches++; }
            else         { ctx->fn<<<grid, block, 0, st>>>(A); }
            CK(cudaGetLastError());
            if (mi > 0) ctx->launches++;
        }
    }
    CK(cudaGetLastError());
    ctx->launches++;
    if (two_pass && !coord_only) {                             // pass 2: one sampling-only launch per plane
        for (size_t i = 0; i <= more_planes; ++i) {
            WarpArgs B = A;
            B.p = p[i];
            B.coord_out = nullptr; B.coord_in = ctx->d_coords; B.coord_maps = n_maps; B.coord_shift = 0;
            if (more_planes > 0) { B.src = (const uint8_t*)in[i].ptr; B.dst = (uint8_t*)out[i].ptr; B.src_len = in[i].len; B.dst_len = out[i].len; }
            fill_uniforms(B, ctx, B.src, B.dst);
            ctx->fn_shade<<<grid, block, 0, st>>>(B);
            CK(cudaGetLastError());
            ctx->launches++;
        }
    }
    if (use_slot) CK(cudaEventRecord(sl.done, st));
    if (ctx->overlays && more_planes == 0 && !coord_only) {    // output stage: stage-1 drawing entries + safe area, on the final pixels
        if (gf_internal_draw_overlays((void*)st, dst, out->len, out->width, out->height, p->output_stride, p, ovl_count, ovl_scalar, 0,
                                      drawing_dev, drawing_len) != GF_OK) return fail(ctx, GF_ERR_CUDA, "overlay kernel (output stage) failed");
        ctx->aux_launches++;
    }
    if (checksum_dev) {                                        // render queue: per-frame output checksum, before the result leaves the device
        if (gf_cuda_checksum_dev(dst, std::min<size_t>(out->len, (size_t)out->height * (size_t)p->output_stride), checksum_dev, (void*)st) != GF_OK)
            return fail(ctx, GF_ERR_CUDA, "checksum kernel failed");
        ctx->aux_launches++;
    }
    if (out->kind == GF_BUF_HOST) {                                                                                  // opencl.rs:413
        nvtxRangePushA("gf_d2h_frame");
        cudaError_t e_d2h;
        if (full_cover) e_d2h = cudaMemcpy2DAsync(out->ptr, (size_t)p->output_stride, ctx->d_dst, (size_t)p->output_stride,
                                                  (size_t)out->width * (size_t)bpp, (size_t)out->height, cudaMemcpyDeviceToHost, st);
        else            e_d2h = cudaMemcpyAsync(out->ptr, ctx->d_dst, out->len, cudaMemcpyDeviceToHost, st);
        nvtxRangePop();
        CK(e_d2h);
    }
    if (sync_host && (in->kind == GF_BUF_HOST || out->kind == GF_BUF_HOST)) CK(cudaStreamSynchronize(st));
    return GF_OK;
}

} // extern "C"

int gf_internal_run_frame(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out, const gf_kernel_params* params,
                          const float* matrices_dev, size_t matrix_rows, const float* mesh_dev, size_t mesh_len,
                          const uint32_t* table_flags_dev, void* cu_stream, uint64_t* checksum_dev) {
    return run_warp(ctx, in, out, params, matrices_dev, matrix_rows, mesh_dev, mesh_len, true, cu_stream, false, 0, false, table_flags_dev, checksum_dev);
}

extern "C" {

GF_API int gf_cuda_undistort_image(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                   const gf_kernel_params* params, const float* matrices, size_t matrix_rows,
                                   const float* mesh, size_t mesh_len, const uint8_t* drawing, size_t drawing_len, void* cu_stream) {
    // the CPU path (the parity target) draws no overlay (cpu_undistort.rs:234-251,607,617): `drawing` is used only after
    // gf_cuda_set_overlays(ctx, 1) — then like the reference's GPU kernels (opencl_undistort.cl:121-154, overlay.cu)
    return run_warp(ctx, in, out, params, matrices, matrix_rows, mesh, mesh_len, false, cu_stream, true, 0, false, nullptr, nullptr, drawing, drawing_len);
}

GF_API int gf_cuda_undistort_image_dev(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                       const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                       const float* mesh_dev, size_t mesh_len, void* cu_stream) {
    return run_warp(ctx, in, out, params, matrices_dev, matrix_rows, mesh_dev, mesh_len, true, cu_stream);
}

GF_API int gf_cuda_undistort_image_dev_flagged(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                               const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                               const float* mesh_dev, size_t mesh_len, const uint32_t* table_flags_dev, void* cu_stream) {
    return run_warp(ctx, in, out, params, matrices_dev, matrix_rows, mesh_dev, mesh_len, true, cu_stream, true, 0, false, table_flags_dev);
}

GF_API int gf_cuda_scan_tables_dev(const float* matrices_dev, size_t matrix_rows, uint32_t* table_flags_dev, void* cu_stream) {
    if (!matrices_dev || !table_flags_dev || matrix_rows == 0) return fail(nullptr, GF_ERR_BAD_PARAMS, "null argument");
    scan_tables_kernel<<<1, 1024, 0, (cudaStream_t)cu_stream>>>(matrices_dev, matrix_rows, table_flags_dev);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(nullptr, e, "scan_tables_kernel");
    return GF_OK;
}

GF_API int gf_cuda_undistort_image_async(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                         const gf_kernel_params* params, const float* matrices, size_t matrix_rows,
                                         const float* mesh, size_t mesh_len, void* cu_stream) {
    return run_warp(ctx, in, out, params, matrices, matrix_rows, mesh, mesh_len, false, cu_stream, false);
}

// ------------------------------------------------------------------------------------------
// ST maps — src/core/stmap.rs:6-146 without the EXR container: the two maps are returned as raw RGB f32 images
// (SpecificChannels::rgb of :131-135: x / width, 1 - y / height, 0).
// ------------------------------------------------------------------------------------------
__global__ void stmap_rgb_kernel(const uint2* __restrict__ coords, int w, int h, int pitch, float* __restrict__ out) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const uint2 e = coords[(size_t)y * pitch + x];
    float cx = 0.0f, cy = 0.0f;                              // `coords` starts zeroed and stays so where the closure returns None (:121-127)
    if (e.x != GF_COORD_MARK) { cx = __uint_as_float(e.x); cy = __uint_as_float(e.y); }
    float* o = out + ((size_t)y * w + x) * 3;
    o[0] = cx / (float)w; o[1] = 1.0f - (cy / (float)h); o[2] = 0.0f;
}

extern "C" int gf_cuda_undistort_points(gf_cuda_gyro* g, const gf_compute_params* cp, int distortion_model, int digital_lens,
                                        double timestamp_ms, size_t frame, int use_fovs, double lens_correction_amount,
                                        const float* points_xy, size_t n, float* out_xy, void* cu_stream);
extern "C" int gf_cuda_stmap_distort_dev(gf_cuda_gyro* g, const gf_compute_params* cp, int distortion_model, int digital_lens,
                                         double timestamp_ms, size_t frame, float* out_rgb_dev, void* cu_stream);

GF_API int gf_cuda_generate_stmap(gf_cuda_gyro* g, const gf_compute_params* cp_user, int distortion_model, int digital_lens,
                                  int per_frame, size_t frame, double timestamp_ms, int32_t* out_new_width, int32_t* out_new_height,
                                  float* dist_rgb_dev, size_t dist_capacity_floats, float* undist_rgb_dev, size_t undist_capacity_floats,
                                  void* cu_stream) {
    if (!g || !cp_user || !out_new_width || !out_new_height) return fail(nullptr, GF_ERR_BAD_PARAMS, "null argument");
    gf_compute_params cp = *cp_user;                                                         // stmap.rs:24-35
    const int width = cp.width, height = cp.height;
    if (width < 4 || height < 4) return fail(nullptr, GF_ERR_SIZE_TOO_SMALL, "SizeTooSmall");
    if (!per_frame) cp.frame_readout_time = 0.0;
    cp.suppress_rotation = 1; cp.fovs = nullptr; cp.n_fovs = 0; cp.minimal_fovs = nullptr; cp.n_minimal_fovs = 0;
    cp.fov_scale = 1.0; cp.output_width = width; cp.output_height = height;                  // :44-46

    // bbox of the undistorted frame edge: points_around_rect(width, height, 31, 31) with fov_algorithm_margin = 0 (:58-60, fov_iterative.rs:154-175)
    std::vector<float> rect, und;
    {
        const float w = (float)width, h = (float)height;
        const int wcnt = 30, hcnt = 30;
        const float wstep = w / (float)wcnt, hstep = h / (float)hcnt;
        for (int i = 0; i < wcnt; ++i) { rect.push_back((float)i * wstep); rect.push_back(0.0f); }
        for (int i = 0; i < hcnt; ++i) { rect.push_back(w); rect.push_back((float)i * hstep); }
        for (int i = 0; i < wcnt; ++i) { rect.push_back((float)(wcnt - i) * wstep); rect.push_back(h); }
        for (int i = 0; i < hcnt; ++i) { rect.push_back(0.0f); rect.push_back((float)(hcnt - i) * hstep); }
        for (float& v : rect) v += 0.0f;
    }
    und.resize(rect.size());
    int rc = gf_cuda_undistort_points(g, &cp, distortion_model, digital_lens, timestamp_ms, frame, 0, 1.0, rect.data(), rect.size() / 2, und.data(), cu_stream);
    if (rc != GF_OK) return fail(nullptr, rc, "gf_cuda_undistort_points failed");
    float min_x = 0.0f, min_y = 0.0f, max_x = 0.0f, max_y = 0.0f;                             // :62-71 (f32::min / max ignore NaN)
    for (size_t i = 0; i < und.size(); i += 2) {
        min_x = fminf(und[i], min_x); min_y = fminf(und[i + 1], min_y);
        max_x = fmaxf(und[i], max_x); max_y = fmaxf(und[i + 1], max_y);
    }
    const float fw = ceilf(max_x - min_x), fh = ceilf(max_y - min_y);
    // `as usize`: truncating, saturating, NaN -> 0
    const long long new_w = fw != fw ? 0 : (fw <= 0.0f ? 0 : (fw >= 2147483647.0f ? 2147483647LL : (long long)fw));
    const long long new_h = fh != fh ? 0 : (fh <= 0.0f ? 0 : (fh >= 2147483647.0f ? 2147483647LL : (long long)fh));
    *out_new_width = (int32_t)new_w; *out_new_height = (int32_t)new_h;
    if (new_w < 4 || new_h < 4 || new_w > 32768 || new_h > 32768) return fail(nullptr, GF_ERR_SIZE_MISMATCH, "ST map: undistorted frame size out of range");
    if (!dist_rgb_dev || !undist_rgb_dev) return GF_OK;                                      // size query
    if (dist_capacity_floats < (size_t)width * height * 3 || undist_capacity_floats < (size_t)new_w * new_h * 3)
        return fail(nullptr, GF_ERR_BUFFER_TOO_SMALL, "ST map output buffers too small");

    cp.fov_scale = (double)fmaxf((float)new_w / (float)width, (float)new_h / (float)height);  // :75
    cp.width = (int)new_w; cp.height = (int)new_h; cp.output_width = (int)new_w; cp.output_height = (int)new_h;
    gf_kernel_params kp;
    const size_t max_rows = (size_t)std::max(new_w, new_h);
    std::vector<float> mats(max_rows * GF_MATRIX_STRIDE);
    size_t rows = 0;
    rc = gf_frame_transform_at_timestamp(&cp, timestamp_ms, frame, &kp, mats.data(), max_rows, &rows, nullptr, nullptr);   // :79
    if (rc != GF_OK) return fail(nullptr, rc, "gf_frame_transform_at_timestamp failed");
    kp.width = (int)new_w; kp.height = (int)new_h; kp.output_width = (int)new_w; kp.output_height = (int)new_h;   // :80-84
    kp.flags = (digital_lens != GF_LENS_NONE ? GF_FLAG_HAS_DIGITAL_LENS : 0) | (cp.readout_horizontal ? GF_FLAG_HORIZONTAL_RS : 0);
    // The closure of :88-109 is undistort_coord's row selection + rotate_and_distort and nothing else: run the warp kernel in
    // coordinate mode with the optional stages switched off (no lens-correction blend, no source-rect map: background mode 3
    // defers that map to the sampling stage, which never runs here).
    gf_kernel_params kq = kp;
    kq.lens_correction_amount = 1.0f; kq.background_mode = 3; kq.input_rotation = 0.0f;
    kq.translation2d[0] = kq.translation2d[1] = 0.0f;
    kq.interpolation = GF_INTERP_BILINEAR; kq.bytes_per_pixel = 1; kq.pix_element_count = 1;
    kq.stride = (int)new_w; kq.output_stride = (int)new_w;
    kq.source_rect[0] = kq.source_rect[1] = 0; kq.source_rect[2] = (int)new_w; kq.source_rect[3] = (int)new_h;
    kq.output_rect[0] = kq.output_rect[1] = 0; kq.output_rect[2] = (int)new_w; kq.output_rect[3] = (int)new_h;
    kq.max_pixel_value = 255.0f; kq.pixel_value_limit = 255.0f;
    gf_buffer_desc d; memset(&d, 0, sizeof(d));
    d.width = (int)new_w; d.height = (int)new_h; d.stride = (int)new_w; d.kind = GF_BUF_DEVICE;
    d.ptr = undist_rgb_dev; d.len = (size_t)new_w * (size_t)new_h;                          // never dereferenced in coordinate mode
    gf_cuda_ctx* ctx = nullptr;
    int device = 0; cudaGetDevice(&device);
    rc = gf_cuda_create(&ctx, device, &kq, GF_PIX_LUMA8, distortion_model, digital_lens, &d, &d, 0);
    if (rc != GF_OK) return rc;
    cudaStream_t st = cu_stream ? (cudaStream_t)cu_stream : ctx->stream;
    rc = run_warp(ctx, &d, &d, &kq, mats.data(), rows, nullptr, 0, false, (void*)st, true, 0, true);
    if (rc == GF_OK) {
        const dim3 block(32, 8), grid(((unsigned)new_w + 31) / 32, ((unsigned)new_h + 7) / 8);
        stmap_rgb_kernel<<<grid, block, 0, st>>>(ctx->d_coords, (int)new_w, (int)new_h, (int)new_w, undist_rgb_dev);
        if (cudaGetLastError() != cudaSuccess) rc = GF_ERR_CUDA;
    }
    if (rc == GF_OK && cudaStreamSynchronize(st) != cudaSuccess) rc = GF_ERR_CUDA;
    gf_cuda_destroy(ctx);
    if (rc != GF_OK) return rc;

    cp.width = width; cp.height = height; cp.output_width = width; cp.output_height = height;   // :111-112 (fov_scale stays)
    rc = gf_cuda_stmap_distort_dev(g, &cp, distortion_model, digital_lens, timestamp_ms, frame, dist_rgb_dev, cu_stream);
    return rc;
}

// Planes of one frame that share their geometry (GBRAPF32's four R32f planes, the U and V planes of planar YUV, ...):
// every KernelParams field except plane_index and background must agree, as must buffer sizes, strides and rects.
static bool same_plane_geometry(const gf_kernel_params& pa, const gf_buffer_desc& ia, const gf_buffer_desc& oa,
                                const gf_kernel_params& pb, const gf_buffer_desc& ib, const gf_buffer_desc& ob) {
    gf_kernel_params a = pa, b = pb;
    a.plane_index = b.plane_index = 0;
    memset(a.background, 0, sizeof(a.background)); memset(b.background, 0, sizeof(b.background));
    if (memcmp(&a, &b, sizeof(a)) != 0) return false;
    const gf_buffer_desc* d[2][2] = {{&ia, &ib}, {&oa, &ob}};
    for (auto& q : d) {
        if (q[0]->width != q[1]->width || q[0]->height != q[1]->height || q[0]->stride != q[1]->stride || q[0]->len != q[1]->len ||
            q[0]->has_rect != q[1]->has_rect || memcmp(q[0]->rect, q[1]->rect, sizeof(q[0]->rect)) != 0 ||
            q[0]->has_rotation != q[1]->has_rotation || q[0]->rotation != q[1]->rotation || q[0]->kind != q[1]->kind) return false;
    }
    return true;
}
static bool planes_share_geometry(const gf_kernel_params* p, const gf_buffer_desc* in, const gf_buffer_desc* out, size_t n) {
    for (size_t i = 1; i < n; ++i) if (!same_plane_geometry(p[0], in[0], out[0], p[i], in[i], out[i])) return false;
    return true;
}
} // extern "C"

bool gf_internal_same_plane_geometry(const gf_kernel_params* pa, const gf_buffer_desc* ia, const gf_buffer_desc* oa,
                                     const gf_kernel_params* pb, const gf_buffer_desc* ib, const gf_buffer_desc* ob) {
    return same_plane_geometry(*pa, *ia, *oa, *pb, *ib, *ob);
}

extern "C" {

GF_API int gf_cuda_undistort_planes_dev(gf_cuda_ctx* ctx, size_t n_planes, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                        const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                        const float* mesh_dev, size_t mesh_len, void* cu_stream) {
    return gf_cuda_undistort_planes_dev_flagged(ctx, n_planes, in, out, params, matrices_dev, matrix_rows, mesh_dev, mesh_len, nullptr, cu_stream);
}

GF_API int gf_cuda_undistort_planes_dev_flagged(gf_cuda_ctx* ctx, size_t n_planes, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                                const gf_kernel_params* params, const float* matrices_dev, size_t matrix_rows,
                                                const float* mesh_dev, size_t mesh_len, const uint32_t* table_flags_dev, void* cu_stream) {
    if (!ctx || !in || !out || !params || n_planes == 0) return fail(ctx, GF_ERR_BAD_PARAMS, "null argument");
    for (size_t i = 0; i < n_planes; ++i) {
        if (in[i].kind != GF_BUF_DEVICE || out[i].kind != GF_BUF_DEVICE) return fail(ctx, GF_ERR_BAD_PARAMS, "gf_cuda_undistort_planes_dev takes DEVICE buffers");
        int rc = validate(ctx, &params[i], &in[i], &out[i], ctx->bpp); if (rc != GF_OK) return rc;
    }
    // one coordinate pass for all planes when they share a geometry
    const bool fuse = n_planes > 1 && ctx->fn_shade && planes_share_geometry(params, in, out, n_planes);
    if (fuse) return run_warp(ctx, in, out, params, matrices_dev, matrix_rows, mesh_dev, mesh_len, true, cu_stream, true, n_planes - 1, false, table_flags_dev);
    for (size_t i = 0; i < n_planes; ++i) {
        int rc = run_warp(ctx, &in[i], &out[i], &params[i], matrices_dev, matrix_rows, mesh_dev, mesh_len, true, cu_stream, true, 0, false, table_flags_dev);
        if (rc != GF_OK) return rc;
    }
    return GF_OK;
}

// The planes of one frame in HOST memory — what the render path hands over for planar software frames (rendering/mod.rs:596-629:
// every plane a BufferSource::Cpu slice): stage every plane to the device, render them like gf_cuda_undistort_planes_dev (one
// coordinate pass shared by the planes of one geometry), copy every plane back, synchronise.  Host tables, like gf_cuda_undistort_image.
GF_API int gf_cuda_undistort_planes(gf_cuda_ctx* ctx, size_t n_planes, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                    const gf_kernel_params* params, const float* matrices, size_t matrix_rows,
                                    const float* mesh, size_t mesh_len, void* cu_stream) {
    if (!ctx || !in || !out || !params || n_planes == 0) return fail(ctx, GF_ERR_BAD_PARAMS, "null argument");
    for (size_t i = 0; i < n_planes; ++i) {
        if (in[i].kind != GF_BUF_HOST || out[i].kind != GF_BUF_HOST) return fail(ctx, GF_ERR_BAD_PARAMS, "gf_cuda_undistort_planes takes HOST buffers (DEVICE: gf_cuda_undistort_planes_dev)");
        int rc = validate(ctx, &params[i], &in[i], &out[i], ctx->bpp); if (rc != GF_OK) return rc;
    }
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = cu_stream ? (cudaStream_t)cu_stream : ctx->stream;
    ctx->last_stream = st;
    if (ctx->d_plane_src.size() < n_planes) { ctx->d_plane_src.resize(n_planes, nullptr); ctx->d_plane_dst.resize(n_planes, nullptr); ctx->d_plane_src_len.resize(n_planes, 0); ctx->d_plane_dst_len.resize(n_planes, 0); }
    std::vector<gf_buffer_desc> din(in, in + n_planes), dout(out, out + n_planes);
    for (size_t i = 0; i < n_planes; ++i) {
        if (in[i].len > ctx->d_plane_src_len[i]) { if (ctx->d_plane_src[i]) { CK(cudaStreamSynchronize(st)); cudaFree(ctx->d_plane_src[i]); ctx->d_plane_src[i] = nullptr; } CK(cudaMalloc(&ctx->d_plane_src[i], in[i].len)); ctx->d_plane_src_len[i] = in[i].len; }
        if (out[i].len > ctx->d_plane_dst_len[i]) { if (ctx->d_plane_dst[i]) { CK(cudaStreamSynchronize(st)); cudaFree(ctx->d_plane_dst[i]); ctx->d_plane_dst[i] = nullptr; } CK(cudaMalloc(&ctx->d_plane_dst[i], out[i].len)); ctx->d_plane_dst_len[i] = out[i].len; }
        CK(cudaMemcpyAsync(ctx->d_plane_src[i], in[i].ptr, in[i].len, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->d_plane_dst[i], out[i].ptr, out[i].len, cudaMemcpyHostToDevice, st));   // untouched pixels keep their content, like on the CPU path
        din[i].kind = GF_BUF_DEVICE; din[i].ptr = ctx->d_plane_src[i];
        dout[i].kind = GF_BUF_DEVICE; dout[i].ptr = ctx->d_plane_dst[i];
    }
    const bool fuse = n_planes > 1 && ctx->fn_shade && planes_share_geometry(params, din.data(), dout.data(), n_planes);
    if (fuse) {
        int rc = run_warp(ctx, din.data(), dout.data(), params, matrices, matrix_rows, mesh, mesh_len, false, (void*)st, false, n_planes - 1);
        if (rc != GF_OK) return rc;
    } else {
        for (size_t i = 0; i < n_planes; ++i) {
            int rc = run_warp(ctx, &din[i], &dout[i], &params[i], matrices, matrix_rows, mesh, mesh_len, false, (void*)st, false);
            if (rc != GF_OK) return rc;
        }
    }
    for (size_t i = 0; i < n_planes; ++i) CK(cudaMemcpyAsync(out[i].ptr, ctx->d_plane_dst[i], out[i].len, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return GF_OK;
}

// Host-only: which kernel variant would render this frame (no CUDA call, no context).  table_flags: 0 = validated tame tables without
// IBIS rows, non-zero = anything else.  Returns PLAN_* (0 general, 1 lean, 2 packed, 3 packed + trusted tables; | 0x10 two-pass),
// or a negative GF_ERR_*.  A planning aid for integrators and the hook the CPU-only tests use to check the host logic.
GF_API int gf_cuda_plan(const gf_kernel_params* params, int pixel_type, int distortion_model, int digital_lens,
                        const gf_buffer_desc* in, const gf_buffer_desc* out, size_t mesh_len, uint32_t table_flags, size_t n_planes) {
    if (!params || !in || !out) return GF_ERR_BAD_PARAMS;
    int layout = 0, bpp = 0;
    if (!pix_layout(pixel_type, &layout, &bpp)) return GF_ERR_BAD_PARAMS;
    { int rc = validate(nullptr, params, in, out, bpp); if (rc != GF_OK) return rc; }
    if (!find_kernel(distortion_model, digital_lens, layout, params->interpolation, 0)) return GF_ERR_UNSUPPORTED_COMBO;
    gf_cuda_ctx ctx;                                           // plain host object: nothing below touches the device
    ctx.pixel_type = pixel_type; ctx.distortion_model = distortion_model; ctx.digital_lens = digital_lens;
    ctx.interpolation = params->interpolation; ctx.layout = layout; ctx.bpp = bpp;
    WarpArgs A; memset(&A, 0, sizeof(A));
    A.p = *params; A.mesh_len = (int)mesh_len;
    A.src = (const uint8_t*)in->ptr; A.dst = (uint8_t*)out->ptr; A.src_len = in->len; A.dst_len = out->len;
    A.out_rows = (int)((out->len + (size_t)params->output_stride - 1) / (size_t)params->output_stride);
    A.out_cols = params->output_stride / bpp;
    fill_uniforms(A, &ctx, A.src, A.dst);
    const bool two_pass = n_planes > 1 || params->interpolation != GF_INTERP_BILINEAR;
    const int n_maps = params->interpolation > 8 ? 3 : 1;
    const bool has_lean = find_kernel(distortion_model, digital_lens, layout, params->interpolation, 1) != nullptr;
    const bool has_packed = !getenv("GF_DISABLE_X2") && find_kernel(distortion_model, digital_lens, layout, GF_INTERP_BILINEAR, two_pass ? 4 : 2) != nullptr;
    return select_variant(has_lean, has_packed, digital_lens, A, table_flags, two_pass, n_maps);
}

GF_API int gf_cuda_validate_tables_dev(gf_cuda_ctx* ctx, const float* matrices_dev, size_t matrix_rows) {
    if (!ctx || !matrices_dev) return fail(ctx, GF_ERR_BAD_PARAMS, "null argument");
    CK(cudaSetDevice(ctx->device));
    // A synchronous QUERY: nothing is cached.  (Round 1 kept a pointer-keyed cache of verdicts; a table rewritten in place or an
    // allocation reused at the same address was then silently trusted.)  To render device tables on the trusted path pass a verdict
    // word to gf_cuda_undistort_image_dev_flagged — written by gf_cuda_scan_tables_dev or by gf_cuda_frame_transform_dev.
    CK(cudaDeviceSynchronize());                               // the table may have been written on any stream
    scan_tables_kernel<<<1, 1024, 0, ctx->stream>>>(matrices_dev, matrix_rows, ctx->d_vflags);
    CK(cudaGetLastError());
    uint32_t f = 0;
    CK(cudaMemcpyAsync(&f, ctx->d_vflags, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return (int)f;      // 0 = tame and IBIS-free; bit 0 = wild entry, bit 1 = IBIS rows present (both still render correctly, on the guarded path)
}

GF_API int gf_cuda_synchronize(gf_cuda_ctx* ctx) {
    if (!ctx) return fail(nullptr, GF_ERR_BAD_PARAMS, "ctx is null");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->last_stream && ctx->last_stream != ctx->stream) CK(cudaStreamSynchronize(ctx->last_stream));   // calls made with a caller-supplied stream
    return GF_OK;
}

GF_API int gf_cuda_set_overlays(gf_cuda_ctx* ctx, int enabled) {
    if (!ctx) return fail(nullptr, GF_ERR_BAD_PARAMS, "ctx is null");
    ctx->overlays = enabled ? 1 : 0;
    return GF_OK;
}

GF_API const char* gf_cuda_last_error(gf_cuda_ctx* ctx) { return ctx ? ctx->last_error.c_str() : g_last_error.c_str(); }
GF_API uint64_t gf_cuda_launch_count(gf_cuda_ctx* ctx) { return ctx ? ctx->launches : 0; }
GF_API int gf_cuda_filter_counts(gf_cuda_ctx* ctx, uint32_t* out) {
    if (!ctx || !out) return fail(ctx, GF_ERR_BAD_PARAMS, "null argument");
    memset(out, 0, GF_FLT_WORDS * sizeof(uint32_t));
    if (ctx->filter_frames == 0) return GF_OK;
    { const int rc = gf_cuda_synchronize(ctx); if (rc != GF_OK) return rc; }
    const unsigned cur = (unsigned)((ctx->filter_frames - 1) & 1ull);     // the latest frame's set: the next one zeroes the other
    CK(cudaMemcpy(out, ctx->d_defer_count + cur * GF_FLT_WORDS, GF_FLT_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return GF_OK;
}

} // extern "C"
