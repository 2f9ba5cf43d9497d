// warp_kernel.cuh — the fused undistort -> rotate (per-scanline) -> redistort -> sample kernel.
//
// One thread = one output pixel; x is the fastest thread index so that stores of a warp cover one
// contiguous 32*bpp-byte span and the 2x2 (or IxI) source taps of neighbouring lanes land in the same
// L1 lines.  Everything per-frame-uniform (the 368-byte KernelParams, derived constants) rides in the
// kernel's __grid_constant__ parameter block, i.e. the constant bank: no loads, uniform registers.
// The per-scanline matrices (rows x 14 f32) are read through the read-only L1 path: neighbouring
// pixels resolve to the same or adjacent rows, so a warp touches one or two 56-byte rows.
//
// Behavioural source (bit-exact target): src/core/stabilization/cpu_undistort.rs:133-228 (rotate_and_distort),
// :329-419 (sample_input_at), :421-517 (undistort_coord), :519-633 (main loop).  Compile with -fmad=false.
#pragma once
#include "lens_models.cuh"
#include "gf_coeffs_tables.h"
#include "f32x2.cuh"
#include <cuda_fp16.h>

namespace gf {

// map_coord (util.rs:144-147) with every per-frame-uniform piece evaluated once on the host, in the same float
// operations: map(x) = ((x - in_min) * mul) / div + add, mul = out_max - out_min, div = in_max - in_min.
struct MapC {
    float in_min, mul, div, rcp, add;   // rcp = 1.0f / div (correctly rounded), used by the exact fast division
    int   fast_div;                     // div is finite, normal and of moderate magnitude
    int   identity;                     // integer-valued x only: ((x - in_min) * mul) / div == x - in_min exactly (products < 2^24, mul == div)
};

// feature bits, decided once per launch on the host (all per-frame uniform)
enum : uint32_t {
    F_RS         = 1u << 0,   // matrix_count > 1
    F_HRS        = 1u << 1,   // flags & 16: horizontal rolling shutter
    F_RLIMIT     = 1u << 2,   // r_limit_sq > 0
    F_REFRACT    = 1u << 3,   // light_refraction_coefficient != 1 && > 0
    F_MESH       = 1u << 4,   // mesh_len > 0
    F_DIGITAL    = 1u << 5,   // flags & 2 (and a digital lens is compiled in)
    F_HSTRETCH   = 1u << 6,   // input_horizontal_stretch > 0.001 and != 1 (x / 1.0f == x exactly, so 1.0 is skipped)
    F_VSTRETCH   = 1u << 7,
    F_LCA        = 1u << 8,   // lens_correction_amount < 1
    F_INROT      = 1u << 9,   // input_rotation != 0
    F_BG1        = 1u << 10,  // background_mode == 1 / 2 / 3
    F_BG2        = 1u << 11,
    F_BG3        = 1u << 12,
    F_FIXRANGE   = 1u << 13,  // flags & 1
    F_FILLBG     = 1u << 14,  // flags & 4
    F_LENS_NOOP  = 1u << 15,  // the lens model's "all coefficients zero" early-out applies (fisheye/sony: k0..k3, generic: k0..k11, gopro: k1)
    F_SRC_VEC    = 1u << 16,  // whole-pixel vector loads / stores are legal (pointer and stride alignment)
    F_DST_VEC    = 1u << 17,
    F_FB_INV     = 1u << 18,  // flags & 128
    F_IS_Y       = 1u << 19,  // plane_index == 0
    F_T3D        = 1u << 20,  // translation3d != 0 (x + 0.0f only differs from x in the sign of zero, which no consumer sees)
    F_PIXLIMIT   = 1u << 21,  // pixel_value_limit below the format's maximum (the min() after sampling can bite)
    F_WILD       = 1u << 22,  // lens coefficients / translation2d / source mapping outside the magnitudes the packed fast paths assume
    F_INTPRO     = 1u << 23,  // packed kernel: both output maps are the identity -> integer prologue (X2Hot below)
    F_FILTER     = 1u << 24,  // packed kernel: filtered rolling-shutter pre-pass (approximate mid-row evaluation + deferred exact pairs)
    F_SRC_VEC8   = 1u << 25,  // source pointer, stride and length are multiples of 8: every aligned 8-byte word that holds a valid byte is readable
};

// Features the specialised ("lean") instantiation compiles out entirely.  The reference's OpenCL backend does the same
// thing at run time: it constant-folds every `(params->flags & N)` test into the program text before building it
// (src/core/gpu/opencl.rs:207-211).  A launch whose feature word has any of these bits uses the general instantiation.
constexpr uint32_t F_GENERAL_ONLY = F_HRS | F_RLIMIT | F_REFRACT | F_MESH | F_HSTRETCH | F_VSTRETCH | F_LCA | F_INROT |
                                    F_BG1 | F_BG2 | F_BG3 | F_FIXRANGE | F_FILLBG | F_LENS_NOOP | F_FB_INV | F_T3D | F_PIXLIMIT;
constexpr uint32_t F_LEAN_REQUIRED = F_SRC_VEC | F_DST_VEC;   // and F_DIGITAL iff a digital lens is compiled in

// has<GEN>(feat, bit): run-time test in the general kernel, compile-time constant in the lean one
template <bool GEN> __device__ __forceinline__ bool has(uint32_t feat, uint32_t bit) {
    if (GEN) return (feat & bit) != 0;
    if (bit & F_GENERAL_ONLY) return false;
    if (bit & (F_LEAN_REQUIRED | F_DIGITAL)) return true;
    return (feat & bit) != 0;        // F_RS, F_IS_Y stay dynamic
}

// per-frame counters of the filtered pre-pass (WarpArgs::X2Filter::count); appends are counted even when the queue is full
enum {
    GF_FLT_PAIRS    = 0,      // pairs appended to the deferred-pair queue (uncertified row or `bad`)
    GF_FLT_PIXELS   = 1,      // pixels appended to the deferred-pixel queue
    GF_FLT_OVERFLOW = 2,      // non-zero: a queue was full, the tail launch re-renders the whole frame
    GF_FLT_BAD      = 3,      // of GF_FLT_PAIRS, the pairs deferred because the final pass set `bad`
    GF_FLT_WORDS    = 4
};

struct WarpArgs {
    gf_kernel_params p;             // verbatim KernelParams
    const uint8_t* src;
    uint8_t*       dst;
    const float*   matrices;        // device, rows x 14, 8-byte aligned
    const float*   mesh;            // device f32 (nullptr when mesh_len == 0)
    const double*  mesh64;          // the same values widened to f64 by a helper kernel before the launch (cpu_undistort.rs:539)
    const struct MeshAux* mesh_aux; // per-frame constants derived from the mesh header by the same helper kernel
    uint2*         coord_out;       // multi-plane mode, pass 1: write the source coordinates of every output pixel here instead of sampling
    const uint2*   coord_in;        // pass 2 (shade_from_coords_kernel): read them back
    const uint32_t* table_flags;    // device word: 0 = the matrix table is tame and IBIS-free (packed kernel: trusted path), see warp_kernel_x2
    // filtered rolling-shutter pre-pass of the packed kernel (F_FILTER): the main launch appends what it does not finish to two queues
    // (pairs whose row choice the approximate evaluation cannot certify or whose fast sequences left their window; pixels whose 8-bit
    // footprint is not interior) and a second launch of the kernel in tail mode renders them
    struct X2Filter {
        uint32_t* q;                // deferred pairs: x | (y0 / 2) << 16
        uint4*    qpx;              // deferred pixels: {x, y, bits(u), bits(v)}, u and v exact
        unsigned* count;            // this frame's GF_FLT_WORDS counters (GF_FLT_* above)
        unsigned* count_next;       // the next frame's counters, zeroed by this frame's tail launch
        uint32_t  cap, cap_px;      // capacities of q and qpx (COORD frames: a full q makes the thread take the exact pre-pass inline)
        int       tail;             // 1 = this launch renders the queues
        float     rho;              // relative tolerance of the certificate
        float     a_cap;            // r^2 below which the tolerance holds for this lens (polynomial conditioning), <= 2^14
    } flt;
    int            coord_shift;     // pass 1: 0 = pixel (x, y); 1 = (x + 0.01, y); 2 = (x, y + 0.01) — the EWA Jacobian probes of :567-572
    int            coord_maps;      // pass 2: 1, or 3 when the two probe maps follow the first one (stride out_cols * out_rows)
    unsigned long long src_len, dst_len;
    int   mesh_len;
    int   out_rows;                 // ceil(dst_len / output_stride): rows the reference iterates (par_chunks_mut)
    int   out_cols;                 // floor(output_stride / bpp): pixels per full row (chunks_mut)
    uint32_t feat;                  // F_* bits
    // derived on the host with the same IEEE float ops as cpu_undistort.rs:521-528 / :421-517
    float r_limit_sq;
    float out_c[2], out_f[2];
    float bg[4];
    MapC  omap_x, omap_y;           // output_rect -> output size   (:422-423, :546-549)
    MapC  smap_x, smap_y;           // frame size  -> source_rect   (:510-515, :599-602)
    float width_f, height_f;        // (float)width / height
    float frame_w, frame_h;         // frame size after input_rotation (:485-489)
    float rot_cos, rot_sin;         // cos/sin(input_rotation * PI/180) via gf_cosf/gf_sinf
    int   rs_lim;                   // HRS ? width : height
    int   u8_limit;                 // trunc(min(pixel_value_limit, 255)) for the integer u8 sampler
    int   src_rect[4];              // rx0, ry0, rx1, ry1
    int   interior_span[2];         // rx1 - 2 - rx0, ry1 - 2 - ry0: a bilinear footprint at (sx, sy) is interior iff (unsigned)(sx - rx0) <= span (both axes)
    // packed kernel: per-frame integers that replace the float rect map + bounds test of :546-551 when both output maps are the
    // identity (F_INTPRO), and the sampler's rect constants side by side (one 128-bit constant load)
    struct X2Hot {
        int x_off, y_off;           // opx == (float)(x + x_off), opy likewise (exact: integers below 2^24)
        int x0, x1, y0, y1;         // pixel (x, y) is written iff x0 <= x < x1 and y0 <= y < y1 ...
        int full_rows, last_cols;   // ... and it fits the buffer: y < full_rows, or y == full_rows and x < last_cols (short last row)
        int rect[4];                // rx0, ry0, span_x, span_y
    } hot;
};

// ------------------------------------------------------------------------------------------
// Pixel formats (pixel_formats.rs): COUNT channels of a SCALAR type.
// ------------------------------------------------------------------------------------------
enum { SC_U8 = 0, SC_U16 = 1, SC_F32 = 2, SC_F16 = 3 };

template <int COUNT_, int SCALAR_> struct Pix {
    static constexpr int COUNT = COUNT_;
    static constexpr int SCALAR = SCALAR_;
    static constexpr int SBYTES = SCALAR_ == SC_U8 ? 1 : (SCALAR_ == SC_F32 ? 4 : 2);
    static constexpr int BYTES = COUNT_ * SBYTES;
    static constexpr bool POW2 = (BYTES == 1 || BYTES == 2 || BYTES == 4 || BYTES == 8 || BYTES == 16);
    static constexpr int ALIGN = POW2 ? BYTES : SBYTES;      // alignment F_SRC_VEC / F_DST_VEC vouch for

    static GF_DEV float scalar_to_float(uint32_t raw) {      // PixelType::to_float
        if (SCALAR == SC_F32) return __uint_as_float(raw);
        if (SCALAR == SC_F16) return __half2float(__ushort_as_half((unsigned short)raw));
        // u8 / u16 widen exactly: 2^23 + raw has raw in its mantissa, the subtraction is exact.  (float)raw compiles to I2F on
        // the quarter-rate XU pipe, which capped the 64-tap Lanczos4 sampler; this is one LOP3/PRMT + one FADD.
        return __uint_as_float(0x4b000000u | raw) - 8388608.0f;
    }
    static GF_DEV uint32_t float_to_scalar(float v) {        // PixelType::from_float: Rust `as` casts
        if (SCALAR == SC_F32) return __float_as_uint(v);
        if (SCALAR == SC_F16) return (uint32_t)__half_as_ushort(__float2half_rn(v));
        int i = __float2int_rz(v);                           // trunc, saturating, NaN -> 0
        const int hi = SCALAR == SC_U8 ? 255 : 65535;
        i = i < 0 ? 0 : (i > hi ? hi : i);
        return (uint32_t)i;
    }
    static GF_DEV uint32_t load_scalar(const uint8_t* __restrict__ p) {      // one aligned scalar
        if (SBYTES == 1) return __ldg(p);
        if (SBYTES == 2) return __ldg(reinterpret_cast<const unsigned short*>(p));
        return __ldg(reinterpret_cast<const unsigned int*>(p));
    }
    // aligned pixel -> COUNT raw scalars
    static GF_DEV void load_raw(const uint8_t* __restrict__ p, uint32_t (&r)[COUNT]) {
        if (!POW2) {
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) r[i] = load_scalar(p + i * SBYTES);
        } else if (BYTES <= 4) {
            const uint32_t w = BYTES == 1 ? (uint32_t)__ldg(p) : (BYTES == 2 ? (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) : __ldg(reinterpret_cast<const unsigned int*>(p)));
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) r[i] = COUNT == 1 ? w : ((w >> (8 * SBYTES * i)) & (SBYTES == 1 ? 0xffu : 0xffffu));
        } else if (BYTES == 8) {
            const uint2 w = __ldg(reinterpret_cast<const uint2*>(p));
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) { const uint32_t q = (i < 2) ? w.x : w.y; r[i] = (q >> (16 * (i & 1))) & 0xffffu; }
        } else {
            const uint4 w = __ldg(reinterpret_cast<const uint4*>(p));
            const uint32_t q[4] = {w.x, w.y, w.z, w.w};
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) r[i] = q[i & 3];
        }
    }
    // aligned pixel -> COUNT "magic" floats 2^23 + raw (integer formats only): the raw value sits in the mantissa, so the
    // caller's exact `- 2^23` yields PixelType::to_float.  One PRMT per channel straight from the loaded word.
    static GF_DEV void load_magic(const uint8_t* __restrict__ p, float (&m)[COUNT]) {
        if (SCALAR == SC_U8 && POW2) {
            const uint32_t w = BYTES == 1 ? (uint32_t)__ldg(p) : (BYTES == 2 ? (uint32_t)__ldg(reinterpret_cast<const unsigned short*>(p)) : __ldg(reinterpret_cast<const unsigned int*>(p)));
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) m[i] = __uint_as_float(__byte_perm(w, 0x4b000000u, 0x7540u + i));          // bytes: w[i], 00, 00, 4b
        } else if (SCALAR == SC_U16 && POW2) {
            uint32_t w[2] = {0u, 0u};
            if (BYTES == 2) w[0] = __ldg(reinterpret_cast<const unsigned short*>(p));
            else if (BYTES == 4) w[0] = __ldg(reinterpret_cast<const unsigned int*>(p));
            else { const uint2 q = __ldg(reinterpret_cast<const uint2*>(p)); w[0] = q.x; w[1] = q.y; }
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) m[i] = __uint_as_float(__byte_perm(w[i >> 1], 0x4b000000u, (i & 1) ? 0x7432u : 0x7410u));   // w.h[i], 00, 4b
        } else {
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) m[i] = __uint_as_float(0x4b000000u | load_scalar(p + i * SBYTES));
        }
    }
    static GF_DEV void load_vec(const uint8_t* __restrict__ p, float (&v)[COUNT]) {
        uint32_t r[COUNT];
        load_raw(p, r);
        #pragma unroll
        for (int i = 0; i < COUNT; ++i) v[i] = scalar_to_float(r[i]);
    }
    static GF_DEV void load_bytes(const uint8_t* __restrict__ p, float (&v)[COUNT]) {     // no alignment assumed
        #pragma unroll
        for (int i = 0; i < COUNT; ++i) {
            uint32_t raw = 0;
            #pragma unroll
            for (int b = 0; b < SBYTES; ++b) raw |= (uint32_t)__ldg(p + i * SBYTES + b) << (8 * b);
            v[i] = scalar_to_float(raw);
        }
    }
    // 8-bit formats: channel c in byte c of one word (aligned)
    static GF_DEV uint32_t load_packed(const uint8_t* __restrict__ p) {
        if (COUNT == 1) return __ldg(p);
        if (COUNT == 2) return __ldg(reinterpret_cast<const unsigned short*>(p));
        if (COUNT == 4) return __ldg(reinterpret_cast<const unsigned int*>(p));
        return (uint32_t)__ldg(p) | ((uint32_t)__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16);
    }
    static GF_DEV void store_scalars(uint8_t* __restrict__ p, bool vec_ok, const uint32_t (&s)[COUNT]) {
        if (vec_ok) {
            if (!POW2) {
                #pragma unroll
                for (int i = 0; i < COUNT; ++i) {
                    if (SBYTES == 1) p[i] = (uint8_t)s[i];
                    else if (SBYTES == 2) reinterpret_cast<unsigned short*>(p)[i] = (unsigned short)s[i];
                    else reinterpret_cast<unsigned int*>(p)[i] = s[i];
                }
            } else if (BYTES <= 4) {
                uint32_t w = 0;
                #pragma unroll
                for (int i = 0; i < COUNT; ++i) w |= s[i] << (8 * SBYTES * i);
                if (BYTES == 1) *p = (uint8_t)w;
                else if (BYTES == 2) *reinterpret_cast<unsigned short*>(p) = (unsigned short)w;
                else *reinterpret_cast<unsigned int*>(p) = w;
            } else if (BYTES == 8) {
                uint2 w = make_uint2(0u, 0u);
                #pragma unroll
                for (int i = 0; i < COUNT; ++i) { if (i < 2) w.x |= s[i] << (16 * (i & 1)); else w.y |= s[i] << (16 * (i & 1)); }
                *reinterpret_cast<uint2*>(p) = w;
            } else {
                *reinterpret_cast<uint4*>(p) = make_uint4(s[0], s[COUNT > 1 ? 1 : 0], s[COUNT > 2 ? 2 : 0], s[COUNT > 3 ? 3 : 0]);
            }
        } else {
            #pragma unroll
            for (int i = 0; i < COUNT; ++i) {
                #pragma unroll
                for (int b = 0; b < SBYTES; ++b) p[i * SBYTES + b] = (uint8_t)(s[i] >> (8 * b));
            }
        }
    }
    static GF_DEV void store(uint8_t* __restrict__ p, bool vec_ok, const float (&v)[COUNT]) {
        uint32_t s[COUNT];
        #pragma unroll
        for (int i = 0; i < COUNT; ++i) s[i] = float_to_scalar(v[i]);
        store_scalars(p, vec_ok, s);
    }
};

// ------------------------------------------------------------------------------------------
// Mesh correction (f64) — gyro_source/splines.rs:100-176, sony.rs:557-563.  The reference widens the
// f32 mesh to f64 once per frame (cpu_undistort.rs:539); here each element is widened on load.
// ------------------------------------------------------------------------------------------
#define GF_MAX_GRID 9
#ifndef GF_MESH9_INLINE
#define GF_MESH9_INLINE 1
#endif
#if GF_MESH9_INLINE
#define GF_MESH9_QUAL GF_DEV
#else
#define GF_MESH9_QUAL static __device__ __noinline__
#endif
struct MeshView {
    const double* __restrict__ m;
    GF_DEV double operator[](uint32_t i) const { return __ldg(m + i); }
};

// mu[] of the natural-spline solve (splines.rs:112-115) does not depend on the data: mu[0] = 0, mu[i] = 1 / (4 - mu[i-1]).
// The same IEEE double operations, evaluated at compile time.
namespace spline_mu {
constexpr double M0 = 0.0, M1 = 1.0 / (4.0 - M0), M2 = 1.0 / (4.0 - M1), M3 = 1.0 / (4.0 - M2), M4 = 1.0 / (4.0 - M3),
                 M5 = 1.0 / (4.0 - M4), M6 = 1.0 / (4.0 - M5), M7 = 1.0 / (4.0 - M6);
}

// Per-frame constants of the mesh block, computed once (helper kernel in c_abi.cu) with the operations the reference repeats
// per pixel: the spline step terms of splines.rs:101-105 for n = 9 and the four map_coord()s of cpu_undistort.rs:173-183 /
// :194-211 (frame <-> mesh-crop coordinates) in the uniform-divisor form of div_uniform.
struct MeshAux {
    double h, inv_h, three_inv_h, h_over_3, inv_3h;      // size_y / 8, 1 / h, 3 * inv_h, h / 3, 1 / (3 h)
    MapC to_crop_x, to_crop_y, to_frame_x, to_frame_y;
};

// BivariateSpline::interpolate for both maps (mesh_offset 0 and 1) of a grid with n_y == 9 rows — splines.rs:141-176.
// Same operations in the same order as the general routine below, restricted to what the result depends on:
// the tridiagonal forward sweep z[], the back-substitution c[] only down to the interval k that contains y, and b, d only at k
// (the extrapolation branches use k = 0 and k = n - 2).  Fully unrolled, everything in registers.
GF_MESH9_QUAL void mesh_interpolate9(const MeshView mesh, const MeshAux& aux, uint32_t n_x, double size_x, double size_y, double x, double y,
                                                       double& out_x, double& out_y) {
    using namespace spline_mu;
    constexpr uint32_t n = 9, grid = GF_MAX_GRID, block = GF_MAX_GRID * 4;
    uint32_t i = as_usize_small(((double)n_x - 1.0) * x / size_x);
    if (i > n_x - 2) i = n_x - 2;
    const double dx = x - size_x * (double)i / (double)(n_x - 1);
    const double dx2 = dx * dx;
    const double h = aux.h, inv_h = aux.inv_h, three_inv_h = aux.three_inv_h, h_over_3 = aux.h_over_3, inv_3h = aux.inv_3h;
    const int mode = y <= 0.0 ? 0 : (y >= size_y ? 2 : 1);
    uint32_t k = 0;
    if (mode == 1) { k = as_usize_small(((double)n - 1.0) * y / size_y); if (k > n - 2) k = n - 2; }
    else if (mode == 2) k = n - 2;
    const double dy = y - size_y * (double)k / (double)(n - 1);
    const double MU[8] = {M0, M1, M2, M3, M4, M5, M6, M7};
    // one base pointer, compile-time offsets from it: with 32-bit index arithmetic every one of the 72 loads carried its own
    // IMAD.WIDE (unsigned wrap-around has to be preserved); the element order and the arithmetic are unchanged
    const double* __restrict__ base = mesh.m + (9u + n_x * n * 2u + i);
    #pragma unroll 1
    for (uint32_t mo = 0; mo < 2; ++mo) {
        const double* __restrict__ rows = base + (size_t)mo * (n * block);
        double a[9];
        #pragma unroll
        for (int j = 0; j < (int)n; ++j) {
            const double* __restrict__ r = rows + j * (int)block;
            a[j] = __ldg(r) + __ldg(r + grid) * dx + __ldg(r + grid * 2) * dx2 + __ldg(r + grid * 3) * dx2 * dx;
        }
        double z[8];
        z[0] = 0.0;
        #pragma unroll
        for (uint32_t q = 1; q + 1 < n; ++q) {
            const double alpha = three_inv_h * (a[q + 1] - 2.0 * a[q] + a[q - 1]);
            z[q] = (alpha * inv_h - z[q - 1]) * MU[q];
        }
        double cur = 0.0, nxt = 0.0, ak = a[0], ak1 = a[1];               // cur = c[q], nxt = c[q + 1]
        #pragma unroll
        for (int q = (int)n - 2; q >= 0; --q) {                            // c[q] = z[q] - mu[q] * c[q+1], stop at q == k
            nxt = cur; cur = z[q] - MU[q] * cur;
            if ((uint32_t)q == k) { ak = a[q]; ak1 = a[q + 1]; break; }
        }
        const double bk = (ak1 - ak) * inv_h - h_over_3 * (nxt + 2.0 * cur);
        const double dk = (nxt - cur) * inv_3h;
        double r;
        if (mode == 0)      r = ak + bk * y;                                                   // a[0] + b[0] * x
        else if (mode == 2) r = ak1 + (bk + 2.0 * cur * h + 3.0 * dk * h * h) * (y - size_y);   // a[n-1] + slope * (x - size)
        else                r = ak + bk * dy + cur * dy * dy + dk * dy * dy * dy;
        if (mo == 0) out_x = r; else out_y = r;
    }
}

static __device__ __noinline__ double mesh_bivariate(const MeshView mesh, uint32_t n_x, uint32_t n_y, double size_x, double size_y,
                                              uint32_t mesh_offset, double x, double y) {
    double a[GF_MAX_GRID], b[GF_MAX_GRID], c[GF_MAX_GRID], d[GF_MAX_GRID], alpha[GF_MAX_GRID], mu[GF_MAX_GRID], z[GF_MAX_GRID];
    uint32_t i = as_usize_small(((double)n_x - 1.0) * x / size_x);
    if (i > n_x - 2) i = n_x - 2;
    const double dx = x - size_x * (double)i / (double)(n_x - 1);
    const double dx2 = dx * dx;
    const uint32_t grid = GF_MAX_GRID, raw_mesh_len = n_x * n_y * 2, block = grid * 4;
    const uint32_t offs = 9 + raw_mesh_len + (mesh_offset * n_y * block) + i;
    for (uint32_t j = 0; j < n_y; ++j) {
        const uint32_t rb = offs + j * block;
        a[j] = mesh[rb] + mesh[rb + grid] * dx + mesh[rb + grid * 2] * dx2 + mesh[rb + grid * 3] * dx2 * dx;   // intermediate_values[j]; cubic_spline_coefficients copies it into a[]
    }
    // cubic_spline_coefficients(intermediate, step 1, offset 0, size_y, n_y) — splines.rs:100-124
    const uint32_t n = n_y;
    const double h = size_y / (double)(n - 1);
    const double inv_h = 1.0 / h;
    const double three_inv_h = 3.0 * inv_h;
    const double h_over_3 = h / 3.0;
    const double inv_3h = 1.0 / (3.0 * h);
    for (uint32_t q = 1; q + 1 < n; ++q) alpha[q] = three_inv_h * (a[q + 1] - 2.0 * a[q] + a[q - 1]);
    mu[0] = 0.0; z[0] = 0.0;
    for (uint32_t q = 1; q + 1 < n; ++q) {
        mu[q] = 1.0 / (4.0 - mu[q - 1]);
        z[q] = (alpha[q] * inv_h - z[q - 1]) * mu[q];
    }
    c[n - 1] = 0.0;
    for (int q = (int)n - 2; q >= 0; --q) {
        c[q] = z[q] - mu[q] * c[q + 1];
        b[q] = (a[q + 1] - a[q]) * inv_h - h_over_3 * (c[q + 1] + 2.0 * c[q]);
        d[q] = (c[q + 1] - c[q]) * inv_3h;
    }
    // cubic_spline_interpolate — splines.rs:126-139
    if (y <= 0.0) return a[0] + b[0] * y;
    if (y >= size_y) {
        const double slope = b[n - 2] + 2.0 * c[n - 2] * h + 3.0 * d[n - 2] * h * h;
        return a[n - 1] + slope * (y - size_y);
    }
    uint32_t k = as_usize_small(((double)n - 1.0) * y / size_y);
    if (k > n - 2) k = n - 2;
    const double dy = y - size_y * (double)k / (double)(n - 1);
    return a[k] + b[k] * dy + c[k] * dy * dy + d[k] * dy * dy * dy;
}

// ------------------------------------------------------------------------------------------
// Exact division by a per-frame-uniform divisor: q = RN(a / d) from the precomputed rcp = RN(1/d).
// One Markstein correction step: with rcp the CORRECTLY ROUNDED reciprocal and q0 = RN(a * rcp) (within one ulp of a / d),
// RN(q0 + fma(-d, q0, a) * rcp) is the correctly rounded quotient for every a and d as long as no intermediate leaves the
// normal range (Markstein 1990; Muller et al., Handbook of Floating-Point Arithmetic, 2nd ed., Thm. 4.8) — the windows below
// guarantee that.  tools/udiv_check.c confirms it by brute force over every float `a` of the window for a list of divisors
// (tests/test_gf_math.py runs a strided sweep).  Outside the window — or when the host did not vouch for the divisor — the
// ordinary division is used.
// ------------------------------------------------------------------------------------------
GF_DEV float div_uniform(float a, const MapC& m) {
    const float aa = fabsf(a);
    if (m.fast_div && aa < 0x1p60f && aa > 0x1p-80f) {
        const float q0 = a * m.rcp;
        const float r0 = __fmaf_rn(-m.div, q0, a);
        return __fmaf_rn(r0, m.rcp, q0);
    }
    return a / m.div;
}
// map_coord for an integer-valued coordinate (pixel index)
GF_DEV float map_apply_int(float x, const MapC& m) {
    if (m.identity) return (x - m.in_min) + m.add;
    return div_uniform((x - m.in_min) * m.mul, m) + m.add;
}
GF_DEV float map_apply(float x, const MapC& m) {
    return div_uniform((x - m.in_min) * m.mul, m) + m.add;
}

// ------------------------------------------------------------------------------------------
// rotate_and_distort — cpu_undistort.rs:133-228
// ------------------------------------------------------------------------------------------
template <int LENS, int DIGITAL, bool GEN>
GF_DEV bool rotate_and_distort(float px, float py, uint32_t idx, const WarpArgs& A, float& ou, float& ov) {
    const gf_kernel_params& P = A.p;
    const uint32_t feat = A.feat;
    const float2* __restrict__ mp = reinterpret_cast<const float2*>(A.matrices + (size_t)idx * GF_MATRIX_STRIDE);
    const float2 m01 = __ldg(mp + 0), m23 = __ldg(mp + 1), m45 = __ldg(mp + 2), m67 = __ldg(mp + 3), m8_9 = __ldg(mp + 4);
    const float2 m10_11 = __ldg(mp + 5), m12_13 = __ldg(mp + 6);
    float _x = (px * m01.x) + (py * m01.y) + m23.x;
    float _y = (px * m23.y) + (py * m45.x) + m45.y;
    float _w = (px * m67.x) + (py * m67.y) + m8_9.x;
    if (has<GEN>(feat, F_T3D)) { _x += P.translation3d[0]; _y += P.translation3d[1]; _w += P.translation3d[2]; }   // :135-137
    if (!(_w > 0.0f)) return false;
    if (has<GEN>(feat, F_RLIMIT | F_REFRACT)) {
        if (has<GEN>(feat, F_RLIMIT) && (_x * _x + _y * _y) > A.r_limit_sq * _w) return false;          // :139 (sic: * _w)
        if (has<GEN>(feat, F_REFRACT)) {                                                                          // :143-152 (_w != 0 holds: _w > 0)
            const float r = sqrtf(_x * _x + _y * _y) / _w;
            const float sin_theta_d = (r / sqrtf(1.0f + r * r)) * P.light_refraction_coefficient;
            const float r_d = sin_theta_d / sqrtf(1.0f - sin_theta_d * sin_theta_d);
            if (r_d != 0.0f) _w *= r / r_d;
        }
    }

    float ux, uy;
    Lens<LENS>::distort(_x, _y, _w, P, has<GEN>(feat, F_LENS_NOOP), ux, uy);                             // :154
    ux = ux * P.f[0]; uy = uy * P.f[1];                                                                // :155

    // :157 — any of m[9..13] != 0.0 (NaN counts as non-zero; -0.0 does not): all bits but the sign
    if (((__float_as_uint(m8_9.y) | __float_as_uint(m10_11.x) | __float_as_uint(m10_11.y) |
          __float_as_uint(m12_13.x) | __float_as_uint(m12_13.y)) << 1) != 0u) {                        // :157-165
        const float ang_rad = m10_11.y;
        const float cos_a = gf_cosf(-ang_rad), sin_a = gf_sinf(-ang_rad);
        const float tx = cos_a * ux - sin_a * uy - m8_9.y   + m12_13.x;
        const float ty = sin_a * ux + cos_a * uy - m10_11.x + m12_13.y;
        ux = tx; uy = ty;
    }

    ux = ux + P.c[0]; uy = uy + P.c[1];                                                                // :167

    if (has<GEN>(feat, F_MESH)) {
        const MeshView mesh{A.mesh64};
        const MeshAux& aux = *A.mesh_aux;
        const bool inv = has<GEN>(feat, F_FB_INV);
        const double mesh0 = mesh[0];
        if (mesh0 > 10.0) {                                                                            // :169-185
            if (inv) uy = A.height_f - uy;
            ux = map_apply(ux, aux.to_crop_x);                 // map_coord(ux, 0, width_f,  origin_x, origin_x + crop_w)
            uy = map_apply(uy, aux.to_crop_y);                 // map_coord(uy, 0, height_f, origin_y, origin_y + crop_h)
            const uint32_t n_x = as_usize_small(mesh[1]), n_y = as_usize_small(mesh[2]);
            const double sx = mesh[3], sy = mesh[4];
            double nx, ny;
            if (n_y == 9 && n_x >= 2 && n_x <= 9) {
                mesh_interpolate9(mesh, aux, n_x, sx, sy, (double)ux, (double)uy, nx, ny);
            } else {
                nx = mesh_bivariate(mesh, n_x, n_y, sx, sy, 0, (double)ux, (double)uy);
                ny = mesh_bivariate(mesh, n_x, n_y, sx, sy, 1, (double)ux, (double)uy);
            }
            ux = map_apply((float)nx, aux.to_frame_x);         // map_coord(nx, origin_x, origin_x + crop_w, 0, width_f)
            uy = map_apply((float)ny, aux.to_frame_y);
            if (inv) uy = A.height_f - uy;
        }
        // FocalPlaneDistortion :188-214 (a missing FPD block means "none"; the reference would index out of bounds)
        const uint32_t o = as_usize_small(mesh0);
        if (mesh0 > 0.0 && o < (uint32_t)A.mesh_len && mesh[o] > 0.0) {
            const double stblz_grid = aux.h;                                                           // mesh_size_y / 8.0
            if (inv) uy = A.height_f - uy;
            ux = map_apply(ux, aux.to_crop_x);
            uy = map_apply(uy, aux.to_crop_y);
            const uint32_t idx2 = as_usize_small(fmin(fmax(floor((double)uy / stblz_grid), 0.0), 7.0));
            const double delta = (double)uy - stblz_grid * (double)idx2;
            ux -= (float)(mesh[o + 4 + idx2 * 2 + 0] * delta);
            uy -= (float)(mesh[o + 4 + idx2 * 2 + 1] * delta);
            for (uint32_t j = 0; j < idx2; ++j) {
                ux -= (float)(mesh[o + 4 + j * 2 + 0] * stblz_grid);
                uy -= (float)(mesh[o + 4 + j * 2 + 1] * stblz_grid);
            }
            ux = map_apply(ux, aux.to_frame_x);
            uy = map_apply(uy, aux.to_frame_y);
            if (inv) uy = A.height_f - uy;
        }
    }

    if (DIGITAL != GF_LENS_NONE && has<GEN>(feat, F_DIGITAL)) {                                        // :216-220
        float dx, dy;
        Lens<DIGITAL>::distort(ux, uy, 1.0f, P, false, dx, dy);
        ux = dx; uy = dy;
    }

    if (has<GEN>(feat, F_HSTRETCH | F_VSTRETCH)) {                                                     // :222-223
        if (has<GEN>(feat, F_HSTRETCH)) ux /= P.input_horizontal_stretch;
        if (has<GEN>(feat, F_VSTRETCH)) uy /= P.input_vertical_stretch;
    }

    ou = ux; ov = uy;
    return true;
}

// rotate_point (cpu_undistort.rs:262-265) with the frame-uniform cos/sin supplied
GF_DEV void rotate_point(float px, float py, float ca, float sa, float ox, float oy, float o2x, float o2y, float& rx, float& ry) {
    rx = ca * (px - ox) - sa * (py - oy) + o2x;
    ry = sa * (px - ox) + ca * (py - oy) + o2y;
}

// undistort_coord — cpu_undistort.rs:421-517.  (opx, opy) = out_pos after the output-rect mapping of :422-423.
template <int LENS, int DIGITAL, bool GEN>
GF_DEV bool undistort_coord(float opx, float opy, const WarpArgs& A, float& ru, float& rv) {
    const gf_kernel_params& P = A.p;
    const uint32_t feat = A.feat;
    opx += P.translation2d[0];
    opy += P.translation2d[1];

    if (has<GEN>(feat, F_LCA)) {                                                                       // :429-460
        float nx = opx, ny = opy;
        const float ocx = A.out_c[0], ocy = A.out_c[1], ofx = A.out_f[0], ofy = A.out_f[1];
        if (DIGITAL != GF_LENS_NONE && has<GEN>(feat, F_DIGITAL)) {
            const float uzx = (nx - ocx) * P.fov + ocx, uzy = (ny - ocy) * P.fov + ocy;
            float tx, ty;
            if (Lens<DIGITAL>::undistort(uzx, uzy, P, false, tx, ty)) {
                nx = (tx - ocx) / P.fov + ocx;
                ny = (ty - ocy) / P.fov + ocy;
            }
        }
        nx = (nx - ocx) / ofx; ny = (ny - ocy) / ofy;
        { float tx, ty; if (Lens<LENS>::undistort(nx, ny, P, has<GEN>(feat, F_LENS_NOOP), tx, ty)) { nx = tx; ny = ty; } }
        if (has<GEN>(feat, F_REFRACT)) {
            const float r = sqrtf(nx * nx + ny * ny);
            if (r != 0.0f) {
                const float sin_theta_d = (r / sqrtf(1.0f + r * r)) / P.light_refraction_coefficient;
                const float r_d = sin_theta_d / sqrtf(1.0f - sin_theta_d * sin_theta_d);
                const float factor = r_d / r;
                nx *= factor; ny *= factor;
            }
        }
        nx = (nx * ofx) + ocx; ny = (ny * ofy) + ocy;
        const float ia = 1.0f - P.lens_correction_amount;
        opx = nx * ia + (opx * P.lens_correction_amount);
        opy = ny * ia + (opy * P.lens_correction_amount);
    }

    // rolling-shutter row :465-482
    const bool hrs = has<GEN>(feat, F_HRS);
    const int lim = A.rs_lim;
    int sy = as_i32(rs_round(hrs ? opx : opy));
    sy = max(min(sy, lim), 0);
    if (has<GEN>(feat, F_RS)) {
        float tu, tv;
        if (rotate_and_distort<LENS, DIGITAL, GEN>(opx, opy, (uint32_t)P.matrix_count / 2u, A, tu, tv)) {
            const int v = as_i32(rs_round(hrs ? tu : tv));
            sy = max(min(v, lim), 0);
        }
    }
    const uint32_t idx = min((uint32_t)sy, (uint32_t)(P.matrix_count - 1));

    float u, v;
    if (!rotate_and_distort<LENS, DIGITAL, GEN>(opx, opy, idx, A, u, v)) return false;                      // :483

    if (has<GEN>(feat, F_INROT | F_BG1 | F_BG2)) {
        if (has<GEN>(feat, F_INROT)) {                                                                          // :485-491
            float nu, nv;
            rotate_point(u, v, A.rot_cos, A.rot_sin, A.width_f / 2.0f, A.height_f / 2.0f, A.frame_w / 2.0f, A.frame_h / 2.0f, nu, nv);
            u = nu; v = nv;
        }
        const float width_f = A.width_f, height_f = A.height_f;
        if (has<GEN>(feat, F_BG1)) {                                                                   // edge repeat :495-499
            u = rs_min(rs_max(u, 3.0f), width_f - 3.0f);
            v = rs_min(rs_max(v, 3.0f), height_f - 3.0f);
        } else if (has<GEN>(feat, F_BG2)) {                                                            // edge mirror :500-509
            const float rx = rs_round(u), ry = rs_round(v);
            const float width3 = width_f - 3.0f, height3 = height_f - 3.0f;
            if (rx > width3)  u = width3  - (rx - width3);
            if (rx < 3.0f)    u = 3.0f + width_f - (width3 + rx);
            if (ry > height3) v = height3 - (ry - height3);
            if (ry < 3.0f)    v = 3.0f + height_f - (height3 + ry);
        }
    }
    if (!has<GEN>(feat, F_BG3)) {                                                                      // :510-515
        u = map_apply(u, A.smap_x);
        v = map_apply(v, A.smap_y);
    }
    ru = u; rv = v;
    return true;
}

// ------------------------------------------------------------------------------------------
// sample_input_at, separable branch (I = 2, 4, 8) — cpu_undistort.rs:370-418
// ------------------------------------------------------------------------------------------
template <int I> GF_DEV void coeff_row(uint32_t frac, float (&c)[I]) {
    if (I == 2) { c[1] = (float)frac * 0.03125f; c[0] = 1.0f - c[1]; }                  // == COEFFS[frac*2 ..]: exact dyadics (k/32)
    else if (I == 4) { _Pragma("unroll") for (int i = 0; i < I; ++i) c[i] = __ldg(&GF_COEFFS_BICUBIC_DEV[(frac << 2) + i]); }
    else { _Pragma("unroll") for (int i = 0; i < I; ++i) c[i] = __ldg(&GF_COEFFS_LANCZOS4_DEV[(frac << 3) + i]); }
}

// The generic (float) sampler: any pixel format, any tap outside source_rect replaced by the background colour.
template <int I, class PIX>
static __device__ __noinline__ void sample_generic(int sx0, int sy0, const WarpArgs& A, float (&sum)[PIX::COUNT]) {
    const gf_kernel_params& P = A.p;
    constexpr int C = PIX::COUNT;
    const int sx = sx0 >> 5, sy = sy0 >> 5;
    float cx[I], cy[I];
    coeff_row<I>((uint32_t)sx0 & 31u, cx);
    coeff_row<I>((uint32_t)sy0 & 31u, cy);
    const int rx0 = A.src_rect[0], ry0 = A.src_rect[1], rx1 = A.src_rect[2], ry1 = A.src_rect[3];
    const bool vec = (A.feat & F_SRC_VEC) != 0;
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) sum[ch] = 0.0f;
    const long long row_base = (long long)sy * (long long)P.stride + (long long)sx * (long long)PIX::BYTES;
    #pragma unroll 1
    for (int yp = 0; yp < I; ++yp) {
        if (sy + yp >= ry0 && sy + yp < ry1) {
            float xsum[C];
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) xsum[ch] = 0.0f;
            #pragma unroll
            for (int xp = 0; xp < I; ++xp) {
                float px[C];
                if (sx + xp >= rx0 && sx + xp < rx1) {
                    const uint8_t* tap = A.src + (row_base + (long long)yp * P.stride + (long long)xp * PIX::BYTES);
                    if (vec) PIX::load_vec(tap, px); else PIX::load_bytes(tap, px);
                } else {
                    #pragma unroll
                    for (int ch = 0; ch < C; ++ch) px[ch] = A.bg[ch];
                }
                #pragma unroll
                for (int ch = 0; ch < C; ++ch) xsum[ch] += px[ch] * cx[xp];
            }
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) sum[ch] += xsum[ch] * cy[yp];
        } else {
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) sum[ch] += A.bg[ch] * cy[yp];
        }
    }
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) sum[ch] = rs_min(sum[ch], P.pixel_value_limit);
}

// Row window of the 16 / 64-tap samplers, integer formats of <= 4 bytes per pixel.  The I taps of one source row are I * BYTES
// contiguous bytes at pixel alignment; with F_SRC_VEC8 they are fetched as the aligned 8-byte words that cover them (2..3 LDG.64
// instead of I narrow loads) and re-aligned in registers: one select per 32-bit word for the 4-byte half, one funnel shift for
// the byte part.  Same bytes, same arithmetic.  Used for 1- and 2-byte pixels (GF_ROW_WINDOW_MAX_BYTES).
#ifndef GF_ROW_WINDOW
#define GF_ROW_WINDOW 1
#endif
#ifndef GF_ROW_WINDOW_MAX_BYTES
#define GF_ROW_WINDOW_MAX_BYTES 2    // measured: 8K Luma16 Lanczos4 +4 %, 4K RGBA8 (4 bytes: 5 LDG.64 + 8 SEL instead of 8 LDG.32) -4.5 %
#endif
#ifndef GF_HI_UNROLL
#define GF_HI_UNROLL 2               // rows of the 16 / 64-tap loop per iteration (full unrolling stalled on instruction fetch)
#endif
#ifndef GF_SHADE_MINB
#define GF_SHADE_MINB 5              // 48 registers: measured best of {none (57-64 regs), 4, 5} x unroll {1, 2}, profiles/README.md
#endif
#ifdef GF_SHADE_MINB
#define GF_SHADE_BOUNDS __launch_bounds__(GF_BLOCK_X * GF_BLOCK_Y, GF_SHADE_MINB)
#else
#define GF_SHADE_BOUNDS __launch_bounds__(GF_BLOCK_X * GF_BLOCK_Y)
#endif
#define GF_PRAGMA_(x) _Pragma(#x)
#define GF_PRAGMA_UNROLL(n) GF_PRAGMA_(unroll n)
template <int I, class PIX> struct RowWindow {
    static constexpr bool ENABLED = GF_ROW_WINDOW && (PIX::SCALAR == SC_U8 || PIX::SCALAR == SC_U16) && PIX::POW2 && PIX::BYTES <= GF_ROW_WINDOW_MAX_BYTES && (I == 4 || I == 8);
    static constexpr int SPAN = I * PIX::BYTES;                            // bytes of taps
    static constexpr int NT = SPAN / 4 > 0 ? SPAN / 4 : 1;                 // 32-bit words of taps
    static constexpr int NQ = (SPAN + 8 - PIX::BYTES + 7) / 8;             // aligned 8-byte words the taps can touch
    static GF_DEV void load(const uint8_t* __restrict__ p, uint32_t (&T)[NT]) {
        const uint32_t o = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 7u);
        const uint2* __restrict__ q = reinterpret_cast<const uint2*>(p - o);
        uint32_t W[2 * NQ];
        #pragma unroll
        for (int i = 0; i < NQ; ++i) {
            uint2 t = make_uint2(0u, 0u);
            if (i < NQ - 1 || o + (uint32_t)SPAN > 8u * (uint32_t)(NQ - 1)) t = __ldg(q + i);   // the last word only when a tap reaches it
            W[2 * i] = t.x; W[2 * i + 1] = t.y;
        }
        const bool hi = (o & 4u) != 0u;
        if (PIX::BYTES == 4) {
            #pragma unroll
            for (int j = 0; j < NT; ++j) T[j] = hi ? W[j + 1] : W[j];
        } else {
            const uint32_t sh = (o & 3u) * 8u;
            uint32_t U[NT + 1];
            #pragma unroll
            for (int j = 0; j <= NT; ++j) U[j] = hi ? W[j + 1] : W[j];
            #pragma unroll
            for (int j = 0; j < NT; ++j) T[j] = __funnelshift_r(U[j], U[j + 1], sh);
        }
    }
    // tap xp as COUNT "magic" floats 2^23 + raw (see Pix::load_magic)
    static GF_DEV void tap(const uint32_t (&T)[NT], int xp, float (&m)[PIX::COUNT]) {
        #pragma unroll
        for (int c = 0; c < PIX::COUNT; ++c) {
            if (PIX::SCALAR == SC_U8) { const int b = xp * PIX::BYTES + c; m[c] = __uint_as_float(__byte_perm(T[b >> 2], 0x4b000000u, 0x7540u + (uint32_t)(b & 3))); }
            else                      { const int h = xp * PIX::COUNT + c; m[c] = __uint_as_float(__byte_perm(T[h >> 1], 0x4b000000u, (h & 1) ? 0x7432u : 0x7410u)); }
        }
    }
};
// feature bit that makes sample_interior<I, PIX> legal
template <int I, class PIX> __host__ __device__ constexpr uint32_t interior_bit() { return RowWindow<I, PIX>::ENABLED ? F_SRC_VEC8 : F_SRC_VEC; }

// Interior fast path: all IxI taps inside source_rect, whole-pixel vector loads.  Same arithmetic, no per-tap tests.
template <int I, class PIX>
GF_DEV void sample_interior(int sx0, int sy0, const WarpArgs& A, float (&sum)[PIX::COUNT]) {
    const gf_kernel_params& P = A.p;
    constexpr int C = PIX::COUNT;
    const int sx = sx0 >> 5, sy = sy0 >> 5;
    const uint8_t* row = A.src + ((long long)sy * (long long)P.stride + (long long)sx * (long long)PIX::BYTES);
    if (I == 2) {
        float cx[I], cy[I];
        coeff_row<I>((uint32_t)sx0 & 31u, cx);
        coeff_row<I>((uint32_t)sy0 & 31u, cy);
        #pragma unroll
        for (int ch = 0; ch < C; ++ch) sum[ch] = 0.0f;
        #pragma unroll
        for (int yp = 0; yp < I; ++yp) {
            float xsum[C];
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) xsum[ch] = 0.0f;
            #pragma unroll
            for (int xp = 0; xp < I; ++xp) {
                float px[C];
                PIX::load_vec(row + xp * PIX::BYTES, px);
                #pragma unroll
                for (int ch = 0; ch < C; ++ch) xsum[ch] += px[ch] * cx[xp];
            }
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) sum[ch] += xsum[ch] * cy[yp];
            row += P.stride;
        }
    } else {
        // 16 / 64 taps.  Same operations in the same order (xsum += px * cx[xp] along a row, sum += xsum * cy[yp] down the rows);
        // the schedule differs: rows are a rolled loop (the fully unrolled 64-tap body stalled on instruction fetch) with cy[yp]
        // read from the table, and with an even channel count the multiply/add stream runs on register pairs (FFMA2), halving
        // its issue slots.  Integer taps are widened by PRMT into m = 2^23 + raw (exact), and the product is taken as
        // fma(m, cx, -2^23*cx): -2^23*cx is exact (a power-of-two scale), so the FMA rounds the exact real raw*cx once —
        // the same value as float(raw) * cx — and the separate subtraction of 2^23 disappears.  (A zero tap yields +0 where
        // the plain product yields sign(cx)*0; the running sum starts at +0 and x + (+-0) == x, so sums are identical; and since
        // the fused form never yields -0, the first tap's 0 + t is t itself and that addition is skipped.)
        constexpr bool INT_FMT = PIX::SCALAR == SC_U8 || PIX::SCALAR == SC_U16;
        constexpr bool PAIRS = (C % 2) == 0;
        constexpr int NP = PAIRS ? C / 2 : 1;
        using RW = RowWindow<I, PIX>;
        float cx[I];
        coeff_row<I>((uint32_t)sx0 & 31u, cx);
        float ncx[I];
        #pragma unroll
        for (int xp = 0; xp < I; ++xp) ncx[xp] = cx[xp] * -8388608.0f;
        const float* __restrict__ cyp = (I == 4 ? GF_COEFFS_BICUBIC_DEV : GF_COEFFS_LANCZOS4_DEV) + (((uint32_t)sy0 & 31u) * I);
        float2 s2[NP];
        #pragma unroll
        for (int k = 0; k < NP; ++k) s2[k] = make_float2(0.0f, 0.0f);
        #pragma unroll
        for (int ch = 0; ch < C; ++ch) sum[ch] = 0.0f;
        GF_PRAGMA_UNROLL(GF_HI_UNROLL)
        for (int yp = 0; yp < I; ++yp) {
            const float cy = __ldg(cyp + yp);
            if (PAIRS) {
                float2 x2[NP];
                #pragma unroll
                for (int k = 0; k < NP; ++k) x2[k] = make_float2(0.0f, 0.0f);
                uint32_t T[RW::NT];
                if (RW::ENABLED) RW::load(row, T);
                #pragma unroll
                for (int xp = 0; xp < I; ++xp) {
                    float v[C];
                    if (RW::ENABLED) RW::tap(T, xp, v); else if (INT_FMT) PIX::load_magic(row + xp * PIX::BYTES, v); else PIX::load_vec(row + xp * PIX::BYTES, v);
                    #pragma unroll
                    for (int k = 0; k < NP; ++k) {
                        const float2 px = make_float2(v[2 * k], v[2 * k + 1]);
                        const float2 t = INT_FMT ? p2::fma(px, p2::bc(cx[xp]), p2::bc(ncx[xp])) : p2::mul(px, p2::bc(cx[xp]));
                        x2[k] = (INT_FMT && xp == 0) ? t : p2::add(x2[k], t);      // integer taps: t is never -0, so 0 + t == t
                    }
                }
                #pragma unroll
                for (int k = 0; k < NP; ++k) s2[k] = p2::add(s2[k], p2::mul(x2[k], p2::bc(cy)));
            } else {
                float xsum[C];
                #pragma unroll
                for (int ch = 0; ch < C; ++ch) xsum[ch] = 0.0f;
                uint32_t T[RW::NT];
                if (RW::ENABLED) RW::load(row, T);
                #pragma unroll
                for (int xp = 0; xp < I; ++xp) {
                    float v[C];
                    if (RW::ENABLED) RW::tap(T, xp, v); else if (INT_FMT) PIX::load_magic(row + xp * PIX::BYTES, v); else PIX::load_vec(row + xp * PIX::BYTES, v);
                    #pragma unroll
                    for (int ch = 0; ch < C; ++ch) {
                        const float t = INT_FMT ? __fmaf_rn(v[ch], cx[xp], ncx[xp]) : v[ch] * cx[xp];
                        xsum[ch] = (INT_FMT && xp == 0) ? t : xsum[ch] + t;
                    }
                }
                #pragma unroll
                for (int ch = 0; ch < C; ++ch) sum[ch] += xsum[ch] * cy;
            }
            row += P.stride;
        }
        if (PAIRS) {
            #pragma unroll
            for (int k = 0; k < NP; ++k) { sum[2 * k] = s2[k].x; sum[2 * k + 1] = s2[k].y; }
        }
    }
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) sum[ch] = rs_min(sum[ch], P.pixel_value_limit);
}

// Integer bilinear for 8-bit formats (interior only).  For u8 taps and 5-bit weights every float operation of the
// reference is exact (8+5+5 = 18 bits < 24), so sum[ch] == N[ch] / 1024 with N = sum p * wx * wy (integers).
// Channels are processed two at a time in 16-bit lanes (max lane value 255*32 = 8160), the vertical pass is one dp2a.
template <class PIX>
GF_DEV void sample_u8_bilinear(int sx0, int sy0, const WarpArgs& A, uint32_t (&N)[PIX::COUNT]) {
    constexpr int C = PIX::COUNT;
    const int sx = sx0 >> 5, sy = sy0 >> 5;
    const uint32_t fx = (uint32_t)sx0 & 31u, fy = (uint32_t)sy0 & 31u;
    const uint32_t wx0 = 32u - fx, wx1 = fx;
    const uint32_t wy = (32u - fy) | (fy << 8);                 // dp2a byte operands: wy0, wy1
    const uint8_t* row0 = A.src + ((long long)sy * (long long)A.p.stride + (long long)sx * (long long)C);
    const uint8_t* row1 = row0 + A.p.stride;
    const uint32_t p00 = PIX::load_packed(row0), p01 = PIX::load_packed(row0 + C);
    const uint32_t p10 = PIX::load_packed(row1), p11 = PIX::load_packed(row1 + C);
    // even channels (bytes 0, 2) and odd channels (bytes 1, 3) in 16-bit lanes
    const uint32_t he0 = (p00 & 0x00ff00ffu) * wx0 + (p01 & 0x00ff00ffu) * wx1;      // row 0: ch0 | ch2 << 16
    const uint32_t he1 = (p10 & 0x00ff00ffu) * wx0 + (p11 & 0x00ff00ffu) * wx1;      // row 1
    N[0] = __dp2a_lo(__byte_perm(he0, he1, 0x5410), wy, 0u);                          // (he0.lo, he1.lo) . (wy0, wy1)
    if (C > 2) N[C > 2 ? 2 : 0] = __dp2a_lo(__byte_perm(he0, he1, 0x7632), wy, 0u);   // (he0.hi, he1.hi)
    if (C > 1) {
        const uint32_t ho0 = __byte_perm(p00, 0u, 0x4341) * wx0 + __byte_perm(p01, 0u, 0x4341) * wx1;   // ch1 | ch3 << 16
        const uint32_t ho1 = __byte_perm(p10, 0u, 0x4341) * wx0 + __byte_perm(p11, 0u, 0x4341) * wx1;
        N[1] = __dp2a_lo(__byte_perm(ho0, ho1, 0x5410), wy, 0u);
        if (C > 3) N[C > 3 ? 3 : 0] = __dp2a_lo(__byte_perm(ho0, ho1, 0x7632), wy, 0u);
    }
}

template <int C> GF_DEV void remap_colorrange(float (&px)[C], bool is_y) {      // cpu_undistort.rs:255-260
    const float s = is_y ? 0.85882352f : 0.87843137f;
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) px[ch] *= s;
    px[0] += 16.0f;
    if (C > 1) px[C > 1 ? 1 : 0] += 16.0f;
}

// sample_input_at at (u, v): picks the integer / interior / generic sampler.  Returns the clamped float sums
// (what the reference's `sum` holds after :413-418).
// Bicubic (I = 4) and Lanczos4 (I = 8) — cpu_undistort.rs:370-418 with offset 1 / 3 (:372-376).  Only the coordinate-map shading
// kernel reaches these (one instantiation per pixel format), through a uniform run-time branch on the resampler, and they are
// inlined into it: as an out-of-line function the sampler saw the kernel parameters through a generic pointer (LD.E + R2UR per
// access instead of constant-bank operands), which cost 12-18 % of the two-pass frame rate (profiles/README.md, r02n).
template <int I, class PIX>
GF_DEV void sample_input_at_hi(float uvx, float uvy, const WarpArgs& A, float (&sum)[PIX::COUNT]) {
    const float offset = I == 4 ? 1.0f : 3.0f;
    const int sx0 = as_i32(rs_round((uvx - offset) * 32.0f));
    const int sy0 = as_i32(rs_round((uvy - offset) * 32.0f));
    const int sx = sx0 >> 5, sy = sy0 >> 5;
    const bool interior = (A.feat & interior_bit<I, PIX>()) != 0 && sx >= A.src_rect[0] && sx + I <= A.src_rect[2] && sy >= A.src_rect[1] && sy + I <= A.src_rect[3];
    if (interior) sample_interior<I, PIX>(sx0, sy0, A, sum);
    else          sample_generic<I, PIX>(sx0, sy0, A, sum);
}
// EWA (Elliptical Weighted Average) CubicBC resampling, I = 10..13 — cpu_undistort.rs:271-327 (helpers), :331-369 (loop).
// jac = (du/dx, du/dy, dv/dx, dv/dy) by forward differences (:567-572).
GF_DEV float bc2(float x, const gf_kernel_params& P) {                                          // :316-326
    x = fabsf(x);
    const float x2 = x * x;
    if (x < 1.0f) return P.ewa_coeffs_p[0] + P.ewa_coeffs_p[1] * x + P.ewa_coeffs_p[2] * x2 + P.ewa_coeffs_p[3] * x2 * x;
    if (x < 2.0f) return P.ewa_coeffs_q[0] + P.ewa_coeffs_q[1] * x + P.ewa_coeffs_q[2] * x2 + P.ewa_coeffs_q[3] * x2 * x;
    return 0.0f;
}
template <class PIX>
GF_DEV void sample_ewa(float uvx, float uvy, float4 jac, const WarpArgs& A, float (&sum)[PIX::COUNT]) {
    const gf_kernel_params& P = A.p;
    constexpr int C = PIX::COUNT;
    // affine_bbox :272-277
    const float tsx = 2.0f * rs_max(rs_max(fabsf(jac.x + jac.y), fabsf(jac.x - jac.y)), 1.0f);
    const float tsy = 2.0f * rs_max(rs_max(fabsf(jac.z + jac.w), fabsf(jac.z - jac.w)), 1.0f);
    const int b0 = as_i32(floorf(uvx - tsx)), b1 = as_i32(ceilf(uvx + tsx));
    const int b2 = as_i32(floorf(uvy - tsy)), b3 = as_i32(ceilf(uvy + tsy));
    // clamped_ellipse :279-315
    const float f0 = fabsf(jac.x * jac.w - jac.y * jac.z);
    const float f = rs_max(f0 * f0, 0.1f);
    const float a = (jac.z * jac.z + jac.w * jac.w) / f;
    const float b = -2.0f * (jac.x * jac.z + jac.y * jac.w) / f;
    const float c = (jac.x * jac.x + jac.y * jac.y) / f;
    const float vx = c - a, vy = -b;
    const float lv = sqrtf(vx * vx + vy * vy);
    const float v0 = lv > 0.01f ? vx / lv : 1.0f;
    const float cc = sqrtf(rs_max(1.0f + v0, 0.0f) / 2.0f);
    float s = sqrtf(rs_max(1.0f - v0, 0.0f) / 2.0f);
    float a0 = a * cc * cc - b * cc * s + c * s * s;
    float c0 = a * s * s + b * cc * s + c * cc * cc;
    const float bt1 = b * (cc * cc - s * s);
    const float bt2 = 2.0f * (a - c) * cc * s;
    float b0v = bt1 + bt2;
    const float b0v2 = bt1 - bt2;
    if (fabsf(b0v) > fabsf(b0v2)) { s = -s; b0v = b0v2; }
    a0 = rs_min(a0, 1.0f);
    c0 = rs_min(c0, 1.0f);
    const float sn = -s;
    const float ea = a0 * cc * cc - b0v * cc * sn + c0 * sn * sn;
    const float eb = 2.0f * a0 * cc * sn + b0v * cc * cc - b0v * sn * sn - 2.0f * c0 * cc * sn;
    const float ec = a0 * sn * sn + b0v * cc * sn + c0 * cc * cc;

    const int rx0 = A.src_rect[0], ry0 = A.src_rect[1], rx1 = A.src_rect[2], ry1 = A.src_rect[3];
    const bool vec = (A.feat & F_SRC_VEC) != 0;
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) sum[ch] = 0.0f;
    float sum_div = 0.0f;
    // Footprint guard.  The bounding box comes straight from the Jacobian; where one probe coordinate is None (-> 0) next to a valid
    // centre the forward difference is ~1e5 and the box spans ~1e11 taps: the reference's CPU loop would grind through them for
    // hours, a GPU thread would hang the device.  A footprint of more than 2^22 taps (2048 x 2048; real minification ratios stay
    // below 16 x 16) is therefore rendered as background — the one documented divergence from the reference's (impractical) result.
    if (((long long)b1 - (long long)b0 + 1) * ((long long)b3 - (long long)b2 + 1) > (1ll << 22)) {
        #pragma unroll
        for (int ch = 0; ch < C; ++ch) sum[ch] = rs_min(A.bg[ch], P.pixel_value_limit);
        return;
    }
    // After the guard both spans fit an int; counting taps instead of comparing coordinates keeps the loops in 32-bit arithmetic
    // even when a bound is a saturated INT_MAX.  When the whole box lies inside source_rect the per-tap tests are skipped.
    const int nx = (int)((long long)b1 - (long long)b0 + 1), ny = (int)((long long)b3 - (long long)b2 + 1);
    const bool box_in = b0 >= rx0 && b1 < rx1 && b2 >= ry0 && b3 < ry1;
    const uint8_t* row = A.src + (long long)b2 * (long long)P.stride + (long long)b0 * (long long)PIX::BYTES;
    for (int iy = 0; iy < ny; ++iy, row += P.stride) {
        const int in_y = b2 + iy;
        const float in_fy = (float)in_y - uvy;
        const float in_fy2 = in_fy * eb;
        const float in_fy3 = in_fy * in_fy * ec;
        const bool row_in = box_in || (in_y >= ry0 && in_y < ry1);
        const uint8_t* tap = row;
        for (int ix = 0; ix < nx; ++ix, tap += PIX::BYTES) {
            const int in_x = b0 + ix;
            const float in_fx = (float)in_x - uvx;
            const float dr = in_fx * in_fx * ea + in_fx * in_fy2 + in_fy3;
            const float k = bc2(sqrtf(dr), P);                         // cylindrical filtering
            if (k == 0.0f) continue;
            float px[C];
            if (box_in || (row_in && in_x >= rx0 && in_x < rx1)) {
                if (vec) PIX::load_vec(tap, px); else PIX::load_bytes(tap, px);
            } else {
                #pragma unroll
                for (int ch = 0; ch < C; ++ch) px[ch] = A.bg[ch];
            }
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) sum[ch] += k * px[ch];
            sum_div += k;
        }
    }
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) sum[ch] = rs_min(sum[ch] / sum_div, P.pixel_value_limit);
}

template <class PIX>
GF_DEV void sample_high_order(float uvx, float uvy, float4 jac, const WarpArgs& A, float (&sum)[PIX::COUNT]) {
    if (A.p.interpolation == GF_INTERP_BICUBIC)       sample_input_at_hi<4, PIX>(uvx, uvy, A, sum);
    else if (A.p.interpolation == GF_INTERP_LANCZOS4) sample_input_at_hi<8, PIX>(uvx, uvy, A, sum);
    else                                              sample_ewa<PIX>(uvx, uvy, jac, A, sum);
}

// HI: may the resampler be anything but bilinear?  Only the coordinate-map shading kernel says yes; the fused warp kernels are
// bilinear-only (the host routes every other resampler through the two-pass path), which keeps the 64-tap / EWA code and
// its call out of all per-lens instantiations.
template <int I, class PIX, bool GEN, bool HI = false>
GF_DEV void sample_input_at(float uvx, float uvy, const WarpArgs& A, float (&sum)[PIX::COUNT], float4 jac = make_float4(1.0f, 0.0f, 0.0f, 1.0f)) {
    if (HI && I == 2 && A.p.interpolation != GF_INTERP_BILINEAR) { sample_high_order<PIX>(uvx, uvy, jac, A, sum); return; }
    const float offset = I == 2 ? 0.0f : (I == 4 ? 1.0f : 3.0f);
    const int sx0 = as_i32(rs_round((uvx - offset) * 32.0f));
    const int sy0 = as_i32(rs_round((uvy - offset) * 32.0f));
    const int sx = sx0 >> 5, sy = sy0 >> 5;
    const bool vec_ok = RowWindow<I, PIX>::ENABLED ? (A.feat & F_SRC_VEC8) != 0 : has<GEN>(A.feat, F_SRC_VEC);
    const bool interior = vec_ok && sx >= A.src_rect[0] && sx + I <= A.src_rect[2] && sy >= A.src_rect[1] && sy + I <= A.src_rect[3];
    if (interior) sample_interior<I, PIX>(sx0, sy0, A, sum);
    else          sample_generic<I, PIX>(sx0, sy0, A, sum);
}

// ------------------------------------------------------------------------------------------
// The kernel — main loop of undistort_image_cpu, cpu_undistort.rs:543-625
// ------------------------------------------------------------------------------------------
#define GF_BLOCK_X 32
#define GF_BLOCK_Y 8

// Coordinate-map entries of the multi-plane mode: (u, v) as raw bits, or one of three markers.  The marker's first word is a
// NaN with a payload no arithmetic instruction produces (results are canonical NaNs), so it cannot collide with a computed u.
#define GF_COORD_MARK 0x7fb0c0deu
enum { GF_COORD_NONE = 1, GF_COORD_SKIP = 2, GF_COORD_FILL = 3 };     // undistort_coord returned None / pixel not written / fill-with-background

// cpu_undistort.rs:576-622 — everything after undistort_coord for one output pixel: feather mode, sampling, range fix, store.
template <class PIX, bool GEN, bool HI>
GF_DEV void finish_pixel(bool have_uv, float u, float v, float4 jac, const WarpArgs& A, uint8_t* __restrict__ out) {
    const gf_kernel_params& P = A.p;
    constexpr int C = PIX::COUNT;
    constexpr int I = 2;
    const uint32_t feat = A.feat;
    const bool dvec = has<GEN>(feat, F_DST_VEC);
    float pixel[C];
    #pragma unroll
    for (int ch = 0; ch < C; ++ch) pixel[ch] = A.bg[ch];
    if (have_uv) {
        if (has<GEN>(feat, F_BG3)) {                                                                             // :576-613
            const float width_f = A.width_f, height_f = A.height_f;
            const float widthf = width_f - 1.0f, heightf = height_f - 1.0f;
            const float feather = rs_max(P.background_margin_feather * heightf, 0.0001f);
            float p2x = u, p2y = v, alpha = 1.0f;
            if ((u > widthf - feather) || (u < feather) || (v > heightf - feather) || (v < feather)) {
                alpha = rs_max(rs_min(rs_min(rs_min(rs_min(widthf - u, heightf - v), u), v) / feather, 1.0f), 0.0f);
                p2x = p2x / width_f; p2y = p2y / height_f;
                p2x = ((p2x - 0.5f) * (1.0f - P.background_margin)) + 0.5f;
                p2y = ((p2y - 0.5f) * (1.0f - P.background_margin)) + 0.5f;
                p2x = p2x * width_f; p2y = p2y * height_f;
            }
            u   = map_apply(u,   A.smap_x); v   = map_apply(v,   A.smap_y);
            p2x = map_apply(p2x, A.smap_x); p2y = map_apply(p2y, A.smap_y);
            float c1[C], c2[C];
            sample_input_at<I, PIX, GEN, HI>(u, v, A, c1, jac);
            sample_input_at<I, PIX, GEN, HI>(p2x, p2y, A, c2, jac);          // (the reference notes jac should be adjusted for pt2; it is not)
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) pixel[ch] = c1[ch] * alpha + c2[ch] * (1.0f - alpha);
        } else {
            if (PIX::SCALAR == SC_U8 && !has<GEN>(feat, F_FIXRANGE) && (!HI || P.interpolation == GF_INTERP_BILINEAR)) {
                // 8-bit bilinear interior: integer arithmetic, exact (see sample_u8_bilinear)
                const int sx0 = as_i32(rs_round(u * 32.0f)), sy0 = as_i32(rs_round(v * 32.0f));
                const int sx = sx0 >> 5, sy = sy0 >> 5;
                if (has<GEN>(feat, F_SRC_VEC) && sx >= A.src_rect[0] && sx + 2 <= A.src_rect[2] && sy >= A.src_rect[1] && sy + 2 <= A.src_rect[3]) {
                    uint32_t N[C];
                    sample_u8_bilinear<PIX>(sx0, sy0, A, N);
                    uint32_t s[C];
                    #pragma unroll
                    for (int ch = 0; ch < C; ++ch) s[ch] = (uint32_t)min((int)(N[ch] >> 10), A.u8_limit);   // trunc(min(N/1024, limit))
                    PIX::store_scalars(out, dvec, s);
                    return;
                }
                sample_generic<I, PIX>(sx0, sy0, A, pixel);
            } else {
                sample_input_at<I, PIX, GEN, HI>(u, v, A, pixel, jac);                                           // :615
            }
        }
    }
    if (has<GEN>(feat, F_FIXRANGE)) remap_colorrange<C>(pixel, (feat & F_IS_Y) != 0);                                     // :608-610 / :619-621
    PIX::store(out, dvec, pixel);                                                                                // :611 / :622
}

template <int LENS, int DIGITAL, class PIX, int I, bool GEN>
__global__ void __launch_bounds__(GF_BLOCK_X * GF_BLOCK_Y)
warp_kernel(const __grid_constant__ WarpArgs A) {
    const gf_kernel_params& P = A.p;
    constexpr int C = PIX::COUNT;
    const uint32_t feat = A.feat;
    const int x = blockIdx.x * GF_BLOCK_X + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= A.out_cols || y >= A.out_rows) return;
    uint2* const cmap = A.coord_out ? A.coord_out + ((size_t)y * (size_t)A.out_cols + (size_t)x) : nullptr;   // multi-plane mode, pass 1
    const unsigned long long off = (unsigned long long)y * (unsigned long long)P.output_stride + (unsigned long long)x * PIX::BYTES;
    if (off + PIX::BYTES > A.dst_len) { if (cmap) *cmap = make_uint2(GF_COORD_MARK, GF_COORD_SKIP); return; }   // trailing partial row (chunks_mut of a short last row)

    const float opx = map_apply_int((float)x, A.omap_x);          // :546-549 (and :422-423: same expression, same value)
    const float opy = map_apply_int((float)y, A.omap_y);
    if (!(opx >= 0.0f && opy >= 0.0f && as_i32(opx) < P.output_width && as_i32(opy) < P.output_height)) {            // :551
        if (cmap) *cmap = make_uint2(GF_COORD_MARK, GF_COORD_SKIP);
        return;
    }

    uint8_t* const out = A.dst + off;
    if (has<GEN>(feat, F_FILLBG)) {                                                                                  // :558-561
        if (cmap) { *cmap = make_uint2(GF_COORD_MARK, GF_COORD_FILL); return; }
        float pixel[C];
        #pragma unroll
        for (int ch = 0; ch < C; ++ch) pixel[ch] = A.bg[ch];
        PIX::store(out, has<GEN>(feat, F_DST_VEC), pixel);
        return;
    }

    // :565.  Pass 1 of the two-pass mode may ask for one of the EWA Jacobian probe positions (x + eps, y) / (x, y + eps), :567-572
    float u = 0.0f, v = 0.0f;
    const float qx = (cmap && A.coord_shift == 1) ? map_apply((float)x + 0.01f, A.omap_x) : opx;
    const float qy = (cmap && A.coord_shift == 2) ? map_apply((float)y + 0.01f, A.omap_y) : opy;
    const bool have_uv = undistort_coord<LENS, DIGITAL, GEN>(qx, qy, A, u, v);
    if (cmap) {      // pass 1 of the two-pass mode (multi-plane frames, non-bilinear resamplers, ST maps)
        *cmap = have_uv ? make_uint2(__float_as_uint(u), __float_as_uint(v)) : make_uint2(GF_COORD_MARK, GF_COORD_NONE);
        return;
    }
    finish_pixel<PIX, GEN, false>(have_uv, u, v, make_float4(1.0f, 0.0f, 0.0f, 1.0f), A, out);
}

// Pass 2 of the multi-plane mode: one launch per plane, coordinates from the map — sampling, conversion and store only.
template <class PIX>
__global__ void GF_SHADE_BOUNDS
shade_from_coords_kernel(const __grid_constant__ WarpArgs A) {
    const gf_kernel_params& P = A.p;
    constexpr int C = PIX::COUNT;
    const int x = blockIdx.x * GF_BLOCK_X + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= A.out_cols || y >= A.out_rows) return;
    const uint2 e = __ldg(A.coord_in + ((size_t)y * (size_t)A.out_cols + (size_t)x));
    const bool marked = e.x == GF_COORD_MARK;
    if (marked && e.y == GF_COORD_SKIP) return;
    uint8_t* const out = A.dst + ((unsigned long long)y * (unsigned long long)P.output_stride + (unsigned long long)x * PIX::BYTES);
    if (marked && e.y == GF_COORD_FILL) {
        float pixel[C];
        #pragma unroll
        for (int ch = 0; ch < C; ++ch) pixel[ch] = A.bg[ch];
        PIX::store(out, (A.feat & F_DST_VEC) != 0, pixel);
        return;
    }
    const float u = __uint_as_float(e.x), v = __uint_as_float(e.y);
    float4 jac = make_float4(1.0f, 0.0f, 0.0f, 1.0f);
    if (!marked && A.coord_maps == 3) {                        // :567-572: forward differences over eps = 0.01, None -> (0, 0)
        const size_t plane = (size_t)A.out_cols * (size_t)A.out_rows, i = (size_t)y * (size_t)A.out_cols + (size_t)x;
        const uint2 ex = __ldg(A.coord_in + plane + i), ey = __ldg(A.coord_in + 2 * plane + i);
        const float eps = 0.01f;
        const float xu = ex.x == GF_COORD_MARK ? 0.0f : __uint_as_float(ex.x), xv = ex.x == GF_COORD_MARK ? 0.0f : __uint_as_float(ex.y);
        const float yu = ey.x == GF_COORD_MARK ? 0.0f : __uint_as_float(ey.x), yv = ey.x == GF_COORD_MARK ? 0.0f : __uint_as_float(ey.y);
        jac = make_float4((xu - u) / eps, (yu - u) / eps, (xv - v) / eps, (yv - v) / eps);
    }
    finish_pixel<PIX, true, true>(!marked, u, v, jac, A, out);
}

} // namespace gf
