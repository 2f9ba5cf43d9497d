// kernel_registry.h — ahead-of-time kernel family: one instantiation per
// (lens model, digital lens, pixel layout, interpolation).  The reference selects its kernel by
// splicing lens-model source text into the OpenCL/WGSL program at run time (gpu/opencl.rs:184-211);
// here every valid combination is compiled for sm_100a up front and looked up by id.
#pragma once
#include <cstdlib>
#include "warp_kernel_x2.cuh"

#ifndef GF_X2_MINB
#define GF_X2_MINB 6      // resident 256-thread blocks per SM the packed kernel is compiled for (register cap 65536 / (256 * MINB))
#endif

namespace gf {

typedef void (*KernelFn)(const WarpArgs);

// pixel layouts: (COUNT, SCALAR) pairs that exist in pixel_formats.rs
enum {
    LAY_1U8 = 0, LAY_2U8, LAY_3U8, LAY_4U8,
    LAY_1U16, LAY_2U16, LAY_3U16, LAY_4U16,
    LAY_1F32, LAY_4F32, LAY_4F16,
    LAY_COUNT
};

struct KernelInfo { KernelFn fn; int bytes_per_pixel; };

// implemented once per lens model in inst_<model>.cu; returns nullptr for combinations that are not compiled
// `lean` selects the instantiation with the rare per-frame features compiled out (see F_GENERAL_ONLY)
KernelFn gf_kernel_opencv_fisheye(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_opencv_standard(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_poly3(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_poly5(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_ptlens(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_insta360(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_sony(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_generic_polynomial(int digital, int layout, int interp, int lean);
KernelFn gf_kernel_gopro(int digital, int layout, int interp, int lean);
KernelFn gf_shade_kernel(int layout);      // pass 2 of the multi-plane mode (shade_kernel.cu)

// lean == 5: the packed kernel's filtered instantiation (FILTERED in warp_kernel_x2.cuh), where the lens model has an approximate form
// lean == 4: the packed kernel in coordinate-output mode (pass 1 of the two-pass path); one instantiation per lens model serves
// every pixel layout
// lean == 2: the two-pixels-per-thread packed-f32x2 kernel (warp_kernel_x2.cuh), where the lens model has a packed form; it carries
// both the trusted-table and the guarded code path and picks one from the device word WarpArgs::table_flags
template <int LENS, int DIGITAL, class PIX>
static KernelFn pick_x2(int interp) {
    // packed digital lenses: superview, superview6, hyperview (fisheye pairs) and digital_stretch (every packed lens model)
    if constexpr (Lens2<LENS>::kHas && Digital2<DIGITAL>::kHas) {
        // 6 resident blocks per SM (40 registers): 5 (48 registers) measured 2 % slower on the filtered headline frames, 4 slower still,
        // 7 / 8 compile to the 6 code
        if (interp == GF_INTERP_BILINEAR) return warp_kernel_x2<LENS, DIGITAL, PIX, GF_X2_MINB>;
    }
    return nullptr;
}
template <int LENS, int DIGITAL, class PIX>
static KernelFn pick_interp(int interp, int lean) {
    if (lean == 5) {        // the packed kernel's main launch for filtered frames (fused bilinear sampling)
        if constexpr (LensApprox<LENS>::value && DIGITAL == GF_LENS_NONE)
            if (interp == GF_INTERP_BILINEAR) return warp_kernel_x2<LENS, DIGITAL, PIX, GF_X2_MINB, false, true>;
        return nullptr;
    }
    if (lean == 4) {
        if constexpr (Lens2<LENS>::kHas && Digital2<DIGITAL>::kHas)
            return warp_kernel_x2<LENS, DIGITAL, Pix<1, SC_U8>, GF_X2_MINB, true>;
        return nullptr;
    }
    if (lean == 2) return pick_x2<LENS, DIGITAL, PIX>(interp);
    switch (interp) {
    case GF_INTERP_BILINEAR: return lean ? warp_kernel<LENS, DIGITAL, PIX, 2, false> : warp_kernel<LENS, DIGITAL, PIX, 2, true>;
    // bicubic / Lanczos4: the same scalar kernels with their run-time high-order sampler (sample_high_order in warp_kernel.cuh)
    // EWA CubicBC (Robidoux sharp / Robidoux / Mitchell / Catmull-Rom): same, coefficients in KernelParams::ewa_coeffs_{p,q}
    case GF_INTERP_BICUBIC: case GF_INTERP_LANCZOS4:
    case GF_INTERP_ROBIDOUX_SHARP: case GF_INTERP_ROBIDOUX: case GF_INTERP_MITCHELL: case GF_INTERP_CATMULL_ROM:
        return lean ? warp_kernel<LENS, DIGITAL, PIX, 2, false> : warp_kernel<LENS, DIGITAL, PIX, 2, true>;
    default: return nullptr;
    }
}
template <int LENS, int DIGITAL>
static KernelFn pick_layout(int layout, int interp, int lean) {
    switch (layout) {
    case LAY_1U8:  return pick_interp<LENS, DIGITAL, Pix<1, SC_U8>>(interp, lean);
    case LAY_2U8:  return pick_interp<LENS, DIGITAL, Pix<2, SC_U8>>(interp, lean);
    case LAY_3U8:  return pick_interp<LENS, DIGITAL, Pix<3, SC_U8>>(interp, lean);
    case LAY_4U8:  return pick_interp<LENS, DIGITAL, Pix<4, SC_U8>>(interp, lean);
    case LAY_1U16: return pick_interp<LENS, DIGITAL, Pix<1, SC_U16>>(interp, lean);
    case LAY_2U16: return pick_interp<LENS, DIGITAL, Pix<2, SC_U16>>(interp, lean);
    case LAY_3U16: return pick_interp<LENS, DIGITAL, Pix<3, SC_U16>>(interp, lean);
    case LAY_4U16: return pick_interp<LENS, DIGITAL, Pix<4, SC_U16>>(interp, lean);
    case LAY_1F32: return pick_interp<LENS, DIGITAL, Pix<1, SC_F32>>(interp, lean);
    case LAY_4F32: return pick_interp<LENS, DIGITAL, Pix<4, SC_F32>>(interp, lean);
    case LAY_4F16: return pick_interp<LENS, DIGITAL, Pix<4, SC_F16>>(interp, lean);
    default: return nullptr;
    }
}

} // namespace gf
