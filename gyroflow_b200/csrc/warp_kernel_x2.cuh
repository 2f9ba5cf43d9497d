// warp_kernel_x2.cuh — the warp with two output pixels per thread on Blackwell's packed f32x2 pipe.
//
// Same arithmetic, same rounding, same results as warp_kernel.cuh (the scalar kernel remains the general
// implementation and the exact fallback).  What changes is the schedule:
//   * a thread owns the vertically adjacent pixels (x, y) and (x, y + 1); every FP32 multiply/add of the
//     undistort -> rotate -> redistort chain is issued once for both (FFMA2, see f32x2.cuh);
//   * the hot path is BRANCH-FREE: divisions, square roots and atanf run their exact fast sequences unconditionally
//     while a handful of integer tests accumulate one `bad` predicate (an operand outside the magnitude window in which
//     those sequences are the correctly rounded result, a scanline with IBIS data, ...).  Only if `bad` is set — in
//     practice never — the pair is re-evaluated with the scalar kernel's code (cold, out of line).  No convergence
//     barriers, no slow-path stubs inside the arithmetic, so the scheduler can overlap the two lens evaluations' loads,
//     MUFU ops and FFMA2 chains;
//   * `TRUSTED` tables: the producer of the table (host scan, gf_cuda_scan_tables_dev, or the on-device FrameTransform producer)
//     has established that every matrix entry is zero or of moderate magnitude and that no row carries IBIS data, and left that
//     verdict in a device word the kernel reads at entry; it removes the per-pixel numerator / IBIS tests.
// Only the "lean" feature set (F_GENERAL_ONLY in warp_kernel.cuh) is compiled here.
//
// Behavioural source: src/core/stabilization/cpu_undistort.rs:133-228, :421-517, :543-625 (as warp_kernel.cuh).
#pragma once
#include "warp_kernel.cuh"
#include "approx_atan_table.inc"

namespace gf {

using p2::f2;

// `a` in [2^-56, 2^48): then r = sqrt(a) lies in [2^-28, 2^24), strictly inside atanf's ordinary range [2^-29, 2^25)
GF_DEV bool in_window_r2(float a) {
    const uint32_t t = (__float_as_uint(a) << 1) - (71u << 24);
    return t < (104u << 24);
}
// zero, or 2^-60 <= |v| <= 2^60
GF_DEV bool zero_or_in_window(float v) {
    const uint32_t u = __float_as_uint(v) << 1;
    return u == 0u || (u - (67u << 24)) < (121u << 24);
}

// ------------------------------------------------------------------------------------------
// packed lens models: Lens2<M>::distort(x, y, z) for two pixels.  kHas = a packed implementation exists.
// `bad` is OR-ed with "some lane left the window in which the fast sequences are exact".
// All predicates are combined with & and | (never && / ||) so that no branch is generated for them.
// ------------------------------------------------------------------------------------------
template <int M> struct Lens2 { static constexpr bool kHas = false; };
// lens models with an approximate v evaluation for the filtered rolling-shutter pre-pass (Lens2<M>::approx_v)
template <int M> struct LensApprox { static constexpr bool value = false; };
template <> struct LensApprox<GF_LENS_OPENCV_FISHEYE> { static constexpr bool value = true; };

// opencv_fisheye.rs:72-93 (k != 0: the lean kernel is only chosen when F_LENS_NOOP is clear; |k| bounded by the host)
template <> struct Lens2<GF_LENS_OPENCV_FISHEYE> {
    static constexpr bool kHas = true;
    // FILTERED PRE-PASS.  The mid-row evaluation of cpu_undistort.rs:470-479 only decides which matrix row a pixel uses:
    // idx = clamp(round(v_mid), 0, H).  This is v_mid - c_y computed CHEAPLY — one MUFU.RCP instead of two refined divisions, no
    // square root, atan(r) / r from a cubic table in r^2 (approx_atan_table.inc), fused multiply-adds — together with a proven bound
    // on its distance from the reference's own float result (DESIGN.md §4 "filtered pre-pass"):
    //     |tv_approx - tv_exact| <= rho * |tv - c_y| + 2^-22 * |tv|,   rho = 2^-17,
    // valid while the divisor w is in the window of the exact sequences and r^2 < a_cap (the host derives a_cap from k so that the
    // polynomial 1 + k0 t^2 + ... stays within [3/4, 5/4], which bounds its cancellation).  (_x, _y, _w) are the reference's own
    // unfused products — bit-identical to the exact chain — so only relative perturbations enter after them.
    // Returns false outside that regime; tvc = (v - c_y) otherwise.
    static GF_DEV bool approx_v(float _x, float _y, float _w, const gf_kernel_params& P, float a_cap, float& tvc) {
        const bool ok_w = (_w >= 0x1p-56f) & (_w < 0x1p48f);
        const float iw = p2::rcp_approx(_w);
        const float x = _x * iw, y = _y * iw;
        const float a = __fmaf_rn(x, x, y * y);
        const uint32_t ab = __float_as_uint(a);
        const int idx = min(max((int)(ab >> 19) - (int)GF_APX_BASE, 0), GF_APX_ROWS - 1);
        const float a0 = __uint_as_float((ab & 0xfff80000u) | 0x00040000u);      // midpoint of a's 1/16-octave interval
        const float4 c = __ldg(&GF_APX_TAB[idx]);
        const float d = a - a0;
        const float T = __fmaf_rn(d, __fmaf_rn(d, __fmaf_rn(d, c.w, c.z), c.y), c.x);   // atan(r) / r
        const float t2 = (a * T) * T;                                                     // theta^2
        const float s = __fmaf_rn(t2, __fmaf_rn(t2, __fmaf_rn(t2, __fmaf_rn(t2, P.k[3], P.k[2]), P.k[1]), P.k[0]), 1.0f);
        tvc = ((y * T) * s) * P.f[1];
        return ok_w & (a < a_cap);              // NaN compares false
    }
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 a = add(mul(x, x), mul(y, y));
        // one window for the four quantities the fast sequences depend on: z (divisor; z <= 0 is the reference's `w > 0` test,
        // :138, and goes to the exact code as well) and a = r^2 (square root, r != 0, atanf's ordinary range), both in [2^-56, 2^48).
        if (TRUSTED) {      // no NaN can reach here (finite tame matrices and coordinates): fminf/fmaxf see every lane
            const float lo = fminf(fminf(z.x, z.y), fminf(a.x, a.y)), hi = fmaxf(fmaxf(z.x, z.y), fmaxf(a.x, a.y));
            bad |= !(lo >= 0x1p-56f) | !(hi < 0x1p48f);
        } else {
            bad |= !(z.x >= 0x1p-56f) | !(z.x < 0x1p48f) | !(z.y >= 0x1p-56f) | !(z.y < 0x1p48f) |
                   !in_window_r2(a.x) | !in_window_r2(a.y);
        }
        const f2 r = sqrt_seq(a);
        const f2 theta = atanf2_core(r, GF_ATAN_TAB);
        const f2 theta2 = mul(theta, theta), theta4 = mul(theta2, theta2), theta6 = mul(theta4, theta2), theta8 = mul(theta4, theta4);
        f2 s = add(bc(1.0f), mul(bc(P.k[0]), theta2));
        s = add(s, mul(bc(P.k[1]), theta4));
        s = add(s, mul(bc(P.k[2]), theta6));
        s = add(s, mul(bc(P.k[3]), theta8));
        const f2 theta_d = mul(theta, s);
        const f2 scale = div_seq(theta_d, r);           // r != 0 whenever !bad; theta_d is 0 or of moderate size (|k| <= 2^40, host-checked)
        ox = mul(x, scale); oy = mul(y, scale);
    }
};

// sony.rs:65-89 — the same shape as the fisheye model with a six-term polynomial in theta (all-zero k is F_LENS_NOOP -> scalar kernels)
template <> struct Lens2<GF_LENS_SONY> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 a = add(mul(x, x), mul(y, y));
        if (TRUSTED) {
            const float lo = fminf(fminf(z.x, z.y), fminf(a.x, a.y)), hi = fmaxf(fmaxf(z.x, z.y), fmaxf(a.x, a.y));
            bad |= !(lo >= 0x1p-56f) | !(hi < 0x1p48f);
        } else {
            bad |= !(z.x >= 0x1p-56f) | !(z.x < 0x1p48f) | !(z.y >= 0x1p-56f) | !(z.y < 0x1p48f) |
                   !in_window_r2(a.x) | !in_window_r2(a.y);
        }
        const f2 r = sqrt_seq(a);
        const f2 theta = atanf2_core(r, GF_ATAN_TAB);
        const f2 theta2 = mul(theta, theta), theta3 = mul(theta2, theta), theta4 = mul(theta2, theta2), theta5 = mul(theta2, theta3), theta6 = mul(theta3, theta3);
        f2 td = add(mul(theta, bc(P.k[0])), mul(theta2, bc(P.k[1])));
        td = add(td, mul(theta3, bc(P.k[2])));
        td = add(td, mul(theta4, bc(P.k[3])));
        td = add(td, mul(theta5, bc(P.k[4])));
        td = add(td, mul(theta6, bc(P.k[5])));
        const f2 scale = div_seq(td, r);
        ox = mul(x, scale); oy = mul(y, scale);
    }
};

// opencv_standard.rs:32-48 — rational radial term + tangential + thin-prism terms; the one division besides x/z, y/z is 1 / den
template <> struct Lens2<GF_LENS_OPENCV_STANDARD> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        const float* k = P.k;
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 r2 = add(mul(x, x), mul(y, y)), r4 = mul(r2, r2), r6 = mul(r4, r2);
        const f2 x2t = mul(bc(2.0f), x), y2t = mul(bc(2.0f), y);
        const f2 a1 = mul(x2t, y), a2 = add(r2, mul(x2t, x)), a3 = add(r2, mul(y2t, y));
        const f2 cdist = add(add(add(bc(1.0f), mul(bc(k[0]), r2)), mul(bc(k[1]), r4)), mul(bc(k[4]), r6));
        const f2 den = add(add(add(bc(1.0f), mul(bc(k[5]), r2)), mul(bc(k[6]), r4)), mul(bc(k[7]), r6));
        // z: divisor and the reference's `w > 0` test; den: divisor of 1 / den, any sign (NaN fails the integer window test)
        bad |= !(z.x >= 0x1p-56f) | !(z.x < 0x1p48f) | !(z.y >= 0x1p-56f) | !(z.y < 0x1p48f) | !in_window(den.x) | !in_window(den.y);
        const f2 icdist2 = div_seq(bc(1.0f), den);
        const f2 xr = mul(mul(x, cdist), icdist2), yr = mul(mul(y, cdist), icdist2);
        ox = add(add(add(add(xr, mul(bc(k[2]), a1)), mul(bc(k[3]), a2)), mul(bc(k[8]), r2)), mul(bc(k[9]), r4));
        oy = add(add(add(add(yr, mul(bc(k[2]), a3)), mul(bc(k[3]), a1)), mul(bc(k[10]), r2)), mul(bc(k[11]), r4));
    }
};

// z window shared by the models below: divisor of x / z, y / z and the reference's `w > 0` test (:138)
GF_DEV bool z_outside(f2 z) { return !(z.x >= 0x1p-56f) | !(z.x < 0x1p48f) | !(z.y >= 0x1p-56f) | !(z.y < 0x1p48f); }

// poly3.rs:54-63
template <> struct Lens2<GF_LENS_POLY3> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        bad |= z_outside(z);
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 poly2 = add(mul(bc(P.k[0]), add(mul(x, x), mul(y, y))), bc(1.0f));
        ox = mul(x, poly2); oy = mul(y, poly2);
    }
};
// poly5.rs:43-53
template <> struct Lens2<GF_LENS_POLY5> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        bad |= z_outside(z);
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 ru2 = add(mul(x, x), mul(y, y));
        const f2 poly4 = add(add(bc(1.0f), mul(bc(P.k[0]), ru2)), mul(mul(bc(P.k[1]), ru2), ru2));
        ox = mul(x, poly4); oy = mul(y, poly4);
    }
};
// ptlens.rs:42-53 — sqrt(ru2): ru2 == 0 is fine for the exact square-root sequence only inside its window, so ru2 is windowed too
template <> struct Lens2<GF_LENS_PTLENS> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        bad |= z_outside(z);
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 ru2 = add(mul(x, x), mul(y, y));
        bad |= !in_window(ru2.x) | !in_window(ru2.y);
        const f2 r = sqrt_seq(ru2);
        const f2 poly3 = add(add(add(mul(mul(bc(P.k[0]), ru2), r), mul(bc(P.k[1]), ru2)), mul(bc(P.k[2]), r)), bc(1.0f));
        ox = mul(x, poly3); oy = mul(y, poly3);
    }
};
// generic_polynomial.rs:83-122 — like sony with twelve terms (all-zero k is F_LENS_NOOP -> scalar kernels)
template <> struct Lens2<GF_LENS_GENERIC_POLYNOMIAL> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        const float* k = P.k;
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 a = add(mul(x, x), mul(y, y));
        bad |= z_outside(z) | !in_window_r2(a.x) | !in_window_r2(a.y);
        const f2 r = sqrt_seq(a);
        const f2 t = atanf2_core(r, GF_ATAN_TAB);
        const f2 t2 = mul(t, t), t3 = mul(t2, t), t4 = mul(t2, t2), t5 = mul(t2, t3), t6 = mul(t3, t3), t7 = mul(t3, t4), t8 = mul(t4, t4),
                 t9 = mul(t4, t5), t10 = mul(t5, t5), t11 = mul(t5, t6), t12 = mul(t6, t6);
        f2 td = add(mul(t, bc(k[0])), mul(t2, bc(k[1])));
        td = add(td, mul(t3, bc(k[2])));  td = add(td, mul(t4, bc(k[3])));  td = add(td, mul(t5, bc(k[4])));   td = add(td, mul(t6, bc(k[5])));
        td = add(td, mul(t7, bc(k[6])));  td = add(td, mul(t8, bc(k[7])));  td = add(td, mul(t9, bc(k[8])));   td = add(td, mul(t10, bc(k[9])));
        td = add(td, mul(t11, bc(k[10]))); td = add(td, mul(t12, bc(k[11])));
        const f2 scale = div_seq(td, r);
        ox = mul(x, scale); oy = mul(y, scale);
    }
};
// insta360.rs:27-48 — unified (Mei) model: len = |(x, y, z)|, x' = (x / len) / (z / len + xi)
template <> struct Lens2<GF_LENS_INSTA360> {
    static constexpr bool kHas = true;
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        const f2 k1 = bc(P.k[0]), k2 = bc(P.k[1]), k3 = bc(P.k[2]), p1 = bc(P.k[3]), p2v = bc(P.k[4]), xi = bc(P.k[5]);
        const f2 l2 = add(add(mul(x, x), mul(y, y)), mul(z, z));
        bad |= z_outside(z) | !in_window(l2.x) | !in_window(l2.y);       // z > 0 is the reference's test; l2 feeds the square root
        const f2 len = sqrt_seq(l2);                                       // in [2^-30, 2^30]: a valid divisor
        const f2 den = add(div_seq(z, len), xi);
        bad |= !in_window(den.x) | !in_window(den.y);
        const f2 xn = div_seq(x, len), yn = div_seq(y, len);
        // second-stage numerators can be far smaller than the matrix products (|x| / len): keep them zero or inside the window
        bad |= !zero_or_in_window(xn.x) | !zero_or_in_window(xn.y) | !zero_or_in_window(yn.x) | !zero_or_in_window(yn.y);
        x = div_seq(xn, den);
        y = div_seq(yn, den);
        const f2 r2 = add(mul(x, x), mul(y, y)), r4 = mul(r2, r2), r6 = mul(r4, r2);
        const f2 rad = add(add(add(bc(1.0f), mul(k1, r2)), mul(k2, r4)), mul(k3, r6));
        ox = add(add(mul(x, rad), mul(mul(mul(bc(2.0f), p1), x), y)), mul(p2v, add(r2, mul(mul(bc(2.0f), x), x))));
        oy = add(add(mul(y, rad), mul(mul(mul(bc(2.0f), p2v), x), y)), mul(p1, add(r2, mul(mul(bc(2.0f), y), y))));
    }
};

// gopro.rs:56-72 — angle from the radius (atan below tan(89 deg), the linear continuation above it goes to the exact code), then the
// Newton inversion of POLY(p) = theta (:26-36) with per-lane stop masks: a lane stops updating at the step where the scalar loop
// would `break` (|d| < 1e-12 before the update, |fix| < 1e-7 after it); the loop ends when both lanes have stopped or after 10 steps.
template <> struct Lens2<GF_LENS_GOPRO> {
    static constexpr bool kHas = true;
    static GF_DEV f2 peval(f2 p, const float* k) {          // k0 + p (k1 + p (k2 + p (k3 + p (k4 + p (k5 + p k6)))))
        using namespace p2;
        f2 v = mul(p, bc(k[6]));
        v = mul(p, add(bc(k[5]), v)); v = mul(p, add(bc(k[4]), v)); v = mul(p, add(bc(k[3]), v)); v = mul(p, add(bc(k[2]), v)); v = mul(p, add(bc(k[1]), v));
        return add(bc(k[0]), v);
    }
    static GF_DEV f2 pderiv(f2 p, const float* k) {         // k1 + p (2 k2 + p (3 k3 + p (4 k4 + p (5 k5 + p (6 k6)))))
        using namespace p2;
        f2 v = mul(p, bc(6.0f * k[6]));
        v = mul(p, add(bc(5.0f * k[5]), v)); v = mul(p, add(bc(4.0f * k[4]), v)); v = mul(p, add(bc(3.0f * k[3]), v)); v = mul(p, add(bc(2.0f * k[2]), v));
        return add(bc(k[1]), v);
    }
    template <bool TRUSTED>
    static GF_DEV void distort(f2 x, f2 y, f2 z, const gf_kernel_params& P, f2& ox, f2& oy, bool& bad) {
        using namespace p2;
        const float* k = P.k;
        x = div_seq(x, z); y = div_seq(y, z);
        const f2 a = add(mul(x, x), mul(y, y));
        bad |= z_outside(z) | !in_window_r2(a.x) | !in_window_r2(a.y);          // r in [2^-28, 2^24): above the 1e-9 special case (:69)
        const f2 r = sqrt_seq(a);
        const float tt = 0x1.c9315ap+5f;                                        // tanf(1.5533f) = 57.149097...; == gf_tanf(1.5533f), asserted on the host (fill_uniforms)
        bad |= !(r.x < tt) | !(r.y < tt);                                        // the continuation past ~89 degrees (:66): exact code
        const f2 theta = atanf2_core(r, GF_ATAN_TAB);
        // paraxial guess (theta - k0) / k1: k1 is frame-uniform and host-checked to be inside the division window
        const f2 n0 = sub(theta, bc(k[0]));
        bad |= !zero_or_in_window(n0.x) | !zero_or_in_window(n0.y);
        f2 p = div_seq(n0, bc(k[1]));
        bool da = false, db = false;
        #pragma unroll 1
        for (int i = 0; i < 10; ++i) {
            const f2 d = pderiv(p, k);
            da |= fabsf(d.x) < 1e-12f; db |= fabsf(d.y) < 1e-12f;               // `if d.abs() < 1e-12 { break; }`
            if (da & db) break;
            const f2 num = sub(peval(p, k), theta);
            // a stopped lane keeps dividing harmlessly (its result is discarded); active lanes must be inside the division windows
            bad |= (!da & (!in_window(d.x) | !zero_or_in_window(num.x))) | (!db & (!in_window(d.y) | !zero_or_in_window(num.y)));
            const f2 fix = div_seq(num, mk(da ? 1.0f : d.x, db ? 1.0f : d.y));
            const f2 np = sub(p, fix);
            p = mk(da ? p.x : np.x, db ? p.y : np.y);
            da |= fabsf(fix.x) < 1e-7f; db |= fabsf(fix.y) < 1e-7f;             // `if fix.abs() < 1e-7 { break; }` (after the update)
            if (da & db) break;
        }
        const f2 rn = mul(bc(k[1]), p);
        bad |= !zero_or_in_window(rn.x) | !zero_or_in_window(rn.y);
        const f2 scale = div_seq(rn, r);
        ox = mul(x, scale); oy = mul(y, scale);
    }
};

// ------------------------------------------------------------------------------------------
// packed digital lenses (the second, "digital" distortion of :216-220) for the pairs the fisheye model is compiled with
// ------------------------------------------------------------------------------------------
template <int D> struct Digital2 { static constexpr bool kHas = false; };
template <> struct Digital2<GF_LENS_NONE> { static constexpr bool kHas = true; static GF_DEV void distort(f2&, f2&, const gf_kernel_params&, bool&) {} };
// digital_stretch.rs:19-22
template <> struct Digital2<GF_LENS_DIGITAL_STRETCH> {
    static constexpr bool kHas = true;
    static GF_DEV void distort(f2& x, f2& y, const gf_kernel_params& P, bool&) {
        x = p2::mul(x, p2::bc(P.digital_lens_params[0])); y = p2::mul(y, p2::bc(P.digital_lens_params[1]));
    }
};
struct Superview2 {        // gopro_superview.rs:12-19, both lanes
    static GF_DEV void map(f2& ux, f2& uy) {
        using namespace p2;
        const f2 x2 = mul(ux, ux), y2 = mul(uy, uy);
        const f2 nx = mul(ux, add(bc(1.2100393f), mul(x2, add(bc(-1.2758402f), mul(x2, bc(1.7751845f))))));
        const f2 t1 = mul(sub(bc(0.4465308f), mul(bc(0.7683315f), y2)), y2);
        const f2 t2 = mul(add(add(bc(-0.3574087f), mul(bc(1.1584653f), y2)), mul(bc(0.3529348f), x2)), x2);
        const f2 ny = mul(uy, add(add(bc(0.9364505f), t1), t2));
        ux = nx; uy = ny;
    }
};
struct Superview62 {       // gopro6_superview.rs:12-17
    static GF_DEV f2 abs2(f2 v) { return make_float2(fabsf(v.x), fabsf(v.y)); }
    static GF_DEV void map(f2& ux, f2& uy) {
        using namespace p2;
        ux = mul(ux, sub(bc(1.0f), mul(bc(0.48f), abs2(ux))));
        ux = mul(ux, mul(bc(0.943396f), add(bc(1.0f), mul(bc(0.157895f), abs2(ux)))));
        uy = mul(uy, mul(bc(0.943396f), add(bc(1.0f), mul(bc(0.060000f), abs2(mul(uy, bc(2.0f)))))));
    }
};
struct Hyperview2 {        // gopro_hyperview.rs:10-17
    static GF_DEV void map(f2& ux, f2& uy) {
        using namespace p2;
        const f2 x2 = mul(ux, ux), y2 = mul(uy, uy);
        f2 h = add(bc(-2735.5422363f), mul(x2, bc(1923.1572266f)));
        h = add(bc(1551.2922363f), mul(x2, h));
        h = add(bc(-451.5002441f), mul(x2, h));
        h = add(bc(74.5198746f), mul(x2, h));
        h = add(bc(-8.1668825f), mul(x2, h));
        const f2 nx = mul(ux, add(add(bc(1.5805143f), mul(x2, h)), mul(y2, bc(-0.1086027f))));
        const f2 ny = mul(uy, add(add(bc(1.0238225f), mul(y2, bc(-0.1025671f))), mul(x2, add(bc(-0.2639930f), mul(x2, bc(0.2979266f))))));
        ux = nx; uy = ny;
    }
};
// the *_view.rs family (ViewLens::distort in lens_models.cuh): normalise, x-scale, <= 12 fixed-point steps, de-normalise.
// Each lane stops updating at the step where the scalar code would break; the loop ends when both have (or after 12 steps).
template <typename Fn, int XSCALE_KIND>
struct ViewDigital2 {
    static constexpr bool kHas = true;
    static GF_DEV void distort(f2& x, f2& y, const gf_kernel_params& P, bool& bad) {
        using namespace p2;
        const f2 sw = bc((float)P.width), sh = bc((float)P.height);
        // numerators: source coordinates, zero or of ordinary size (anything else goes to the exact code)
        bad |= !zero_or_in_window(x.x) | !zero_or_in_window(x.y) | !zero_or_in_window(y.x) | !zero_or_in_window(y.y);
        x = sub(div_seq(x, sw), bc(0.5f)); y = sub(div_seq(y, sh), bc(0.5f));
        if (XSCALE_KIND != 0) x = mul(x, bc(XSCALE_KIND == 1 ? 1.333333333f : 1.555555555f));
        f2 ppx = x, ppy = y;
        bool da = false, db = false;
        #pragma unroll 1
        for (int i = 0; i < 12; ++i) {
            f2 dx = ppx, dy = ppy;
            Fn::map(dx, dy);
            dx = sub(dx, x); dy = sub(dy, y);
            da |= (fabsf(dx.x) < 1e-6f) & (fabsf(dy.x) < 1e-6f);
            db |= (fabsf(dx.y) < 1e-6f) & (fabsf(dy.y) < 1e-6f);
            if (da & db) break;
            const f2 nx = sub(ppx, dx), ny = sub(ppy, dy);
            ppx = make_float2(da ? ppx.x : nx.x, db ? ppx.y : nx.y);
            ppy = make_float2(da ? ppy.x : ny.x, db ? ppy.y : ny.y);
        }
        x = mul(add(ppx, bc(0.5f)), sw); y = mul(add(ppy, bc(0.5f)), sh);
    }
};
// gopro_warp.rs:57-94 — the data-driven MAPX / MAPY warp of the `gopro` lens pair: 12-step fixed point towards (x * factor, y) from
// the un-stretched start, per-lane stop masks, then the off-frame sentinel when the iteration did not land on the target.
template <> struct Digital2<GF_LENS_GOPRO_WARP> {
    static constexpr bool kHas = true;
    static GF_DEV f2 clamp05(f2 v) { return make_float2(fminf(fmaxf(v.x, -0.5f), 0.5f), fminf(fmaxf(v.y, -0.5f), 0.5f)); }   // f32::clamp (NaN stays NaN: fmaxf(NaN, -0.5) = -0.5 differs, so NaN lanes are flagged below)
    static GF_DEV void map(f2& ux, f2& uy, const float* q) {                       // gopro_map :22-41
        using namespace p2;
        const f2 x = clamp05(ux), y = clamp05(uy);
        const f2 x2 = mul(x, x), y2 = mul(y, y);
        f2 px = mul(x2, bc(q[6]));
        px = mul(x2, add(bc(q[5]), px)); px = mul(x2, add(bc(q[4]), px)); px = mul(x2, add(bc(q[3]), px)); px = mul(x2, add(bc(q[2]), px)); px = mul(x2, add(bc(q[1]), px));
        px = add(bc(q[0]), px);
        const f2 nx = add(mul(x, add(px, mul(bc(q[7]), y2))), sub(ux, x));
        // y * (p8 + p9 y2 + p10 y2 y2 + x2 (p11 + p12 y2 + p13 x2)) + (uy - y), sums left to right
        const f2 inner = add(add(bc(q[11]), mul(bc(q[12]), y2)), mul(bc(q[13]), x2));
        const f2 sy = add(add(add(bc(q[8]), mul(bc(q[9]), y2)), mul(mul(bc(q[10]), y2), y2)), mul(x2, inner));
        const f2 ny = add(mul(y, sy), sub(uy, y));
        ux = nx; uy = ny;
    }
    static GF_DEV void distort(f2& x, f2& y, const gf_kernel_params& P, bool& bad) {
        using namespace p2;
        const float* q = P.digital_lens_params;
        const float factor = q[14] != 0.0f ? q[14] : 1.0f;
        const f2 sw = bc((float)P.width), sh = bc((float)P.height);
        bad |= !zero_or_in_window(x.x) | !zero_or_in_window(x.y) | !zero_or_in_window(y.x) | !zero_or_in_window(y.y);   // also NaN / Inf coordinates
        x = sub(div_seq(x, sw), bc(0.5f)); y = sub(div_seq(y, sh), bc(0.5f));
        const f2 tx = mul(x, bc(factor)), ty = y;
        f2 ppx = x, ppy = y;
        bool da = false, db = false;
        #pragma unroll 1
        for (int i = 0; i < 12; ++i) {
            f2 dx = ppx, dy = ppy;
            map(dx, dy, q);
            dx = sub(dx, tx); dy = sub(dy, ty);
            da |= (fabsf(dx.x) < 1e-6f) & (fabsf(dy.x) < 1e-6f);
            db |= (fabsf(dx.y) < 1e-6f) & (fabsf(dy.y) < 1e-6f);
            if (da & db) break;
            const f2 nx = sub(ppx, dx), ny = sub(ppy, dy);
            ppx = make_float2(da ? ppx.x : nx.x, db ? ppx.y : nx.y);
            ppy = make_float2(da ? ppy.x : ny.x, db ? ppy.y : ny.y);
        }
        f2 rx = ppx, ry = ppy;
        map(rx, ry, q);
        const f2 ex = sub(rx, tx), ey = sub(ry, ty);
        const bool offa = (fabsf(ex.x) > 0.02f) | (fabsf(ey.x) > 0.02f), offb = (fabsf(ex.y) > 0.02f) | (fabsf(ey.y) > 0.02f);
        bad |= (ppx.x != ppx.x) | (ppx.y != ppx.y) | (ppy.x != ppy.x) | (ppy.y != ppy.y);       // NaN: clamp semantics differ, exact code decides
        const f2 fx = mul(add(ppx, bc(0.5f)), sw), fy = mul(add(ppy, bc(0.5f)), sh);
        x = make_float2(offa ? -99999.0f : fx.x, offb ? -99999.0f : fx.y);
        y = make_float2(offa ? -99999.0f : fy.x, offb ? -99999.0f : fy.y);
    }
};
template <> struct Digital2<GF_LENS_GOPRO_SUPERVIEW>  : ViewDigital2<Superview2, 1>  {};
template <> struct Digital2<GF_LENS_GOPRO6_SUPERVIEW> : ViewDigital2<Superview62, 0> {};
template <> struct Digital2<GF_LENS_GOPRO_HYPERVIEW>  : ViewDigital2<Hyperview2, 2>  {};

// ------------------------------------------------------------------------------------------
// rotate_and_distort for two pixels — cpu_undistort.rs:133-228, lean feature set
// (no translation3d, r_limit, refraction, mesh, digital lens, input stretch).
// ------------------------------------------------------------------------------------------
struct MatRow9 { float2 m01, m23, m45, m67; float m8; };      // rows without the IBIS tail (TRUSTED tables have none)
GF_DEV MatRow9 load_row9(const float* __restrict__ matrices, uint32_t idx) {
    const float2* __restrict__ mp = reinterpret_cast<const float2*>(matrices + (size_t)idx * GF_MATRIX_STRIDE);
    MatRow9 r;
    r.m01 = __ldg(mp + 0); r.m23 = __ldg(mp + 1); r.m45 = __ldg(mp + 2); r.m67 = __ldg(mp + 3);
    r.m8 = __ldg(reinterpret_cast<const float*>(mp + 4));
    return r;
}
GF_DEV bool row_has_ibis(const float* __restrict__ matrices, uint32_t idx) {      // :157 — any of m[9..13] != 0.0
    const float* __restrict__ m = matrices + (size_t)idx * GF_MATRIX_STRIDE;
    return ((__float_as_uint(__ldg(m + 9)) | __float_as_uint(__ldg(m + 10)) | __float_as_uint(__ldg(m + 11)) |
             __float_as_uint(__ldg(m + 12)) | __float_as_uint(__ldg(m + 13))) << 1) != 0u;
}

// hot path: no branches.  Returns u, v for both lanes and ORs `bad`; a lane with w <= 0 (the reference's None, :138) counts as
// bad too — it is rare (rays more than 90 degrees off axis) and the exact code handles it.
template <int LENS, int DIGITAL, bool TRUSTED>
GF_DEV void rotate_and_distort_x2(f2 px, f2 py, uint32_t idx_a, uint32_t idx_b, const WarpArgs& A, f2& ou, f2& ov, bool& bad) {
    using namespace p2;
    const gf_kernel_params& P = A.p;
    // wide loads + pair-building moves measured faster than 18 scalar loads straight into register pairs (9.55k vs 9.39k frames/s)
    const MatRow9 ra = load_row9(A.matrices, idx_a), rb = load_row9(A.matrices, idx_b);
    const f2 _x = add(add(mul(px, mk(ra.m01.x, rb.m01.x)), mul(py, mk(ra.m01.y, rb.m01.y))), mk(ra.m23.x, rb.m23.x));
    const f2 _y = add(add(mul(px, mk(ra.m23.y, rb.m23.y)), mul(py, mk(ra.m45.x, rb.m45.x))), mk(ra.m45.y, rb.m45.y));
    const f2 _w = add(add(mul(px, mk(ra.m67.x, rb.m67.x)), mul(py, mk(ra.m67.y, rb.m67.y))), mk(ra.m8, rb.m8));
    if (!TRUSTED) {
        bad |= !zero_or_in_window(_x.x) | !zero_or_in_window(_y.x) | row_has_ibis(A.matrices, idx_a) |
               !zero_or_in_window(_x.y) | !zero_or_in_window(_y.y) | row_has_ibis(A.matrices, idx_b);
    }
    f2 ux, uy;
    Lens2<LENS>::template distort<TRUSTED>(_x, _y, _w, P, ux, uy, bad);                                // :154
    ux = mul(ux, bc(P.f[0])); uy = mul(uy, bc(P.f[1]));                                                // :155
    ou = add(ux, bc(P.c[0])); ov = add(uy, bc(P.c[1]));                                                // :167 (no IBIS rows on this path)
    Digital2<DIGITAL>::distort(ou, ov, P, bad);                                                        // :216-220 (the lean set has F_DIGITAL == (DIGITAL != none))
}

// cold path: the scalar kernel's exact code for both pixels of the pair, one call site per pass.
struct PairUV { float ua, va, ub, vb; int ok; };      // ok: bit 0/1 = lane a/b is Some(..); bit 2/3 = its coordinates are outside the
                                                       // domain of the hot path's rounding shortcut (|u| or |v| >= 2^16, or NaN)
GF_DEV bool outside_shortcut(float u, float v) { return !(fabsf(u) < 0x1p16f) | !(fabsf(v) < 0x1p16f); }
template <int LENS, int DIGITAL>
static __device__ __noinline__ PairUV rotate_and_distort_cold(float px, float pya, float pyb, uint32_t idx_a, uint32_t idx_b, const WarpArgs& A, int apply_smap) {
    PairUV o; o.ua = o.va = o.ub = o.vb = 0.0f; o.ok = 0;
    float cu, cv;
    if (rotate_and_distort<LENS, DIGITAL, false>(px, pya, idx_a, A, cu, cv)) {
        if (apply_smap) { cu = map_apply(cu, A.smap_x); cv = map_apply(cv, A.smap_y); }
        o.ua = cu; o.va = cv; o.ok |= 1 | (outside_shortcut(cu, cv) ? 4 : 0);
    }
    if (rotate_and_distort<LENS, DIGITAL, false>(px, pyb, idx_b, A, cu, cv)) {
        if (apply_smap) { cu = map_apply(cu, A.smap_x); cv = map_apply(cv, A.smap_y); }
        o.ub = cu; o.vb = cv; o.ok |= 2 | (outside_shortcut(cu, cv) ? 8 : 0);
    }
    return o;
}

// map_coord with a uniform divisor on a pair (see div_uniform in warp_kernel.cuh).  The two-step division is exact for a numerator
// that is +-0 or has 2^-80 < |a| < 2^60.  The host guarantees in_min == 0, 2^-40 <= |mul| and |c| >= 2^-10 (so a non-zero x is at
// least 2^-34 in magnitude and |a| >= 2^-74), and div <= 2^20 (so |a| >= 2^60 would give |result| >= 2^39): testing the RESULT
// against 2^16 therefore covers the numerator window, catches NaN/Inf, and bounds what the rounding shortcut has to handle.
GF_DEV f2 map_apply_x2(f2 x, const MapC& m, bool& bad) {
    using namespace p2;
    const f2 a = mul(sub(x, bc(m.in_min)), bc(m.mul));
    const f2 q0 = mul(a, bc(m.rcp));
    const f2 r0 = fma(bc(-m.div), q0, a);
    const f2 r = add(fma(r0, bc(m.rcp), q0), bc(m.add));
    bad |= !(fabsf(r.x) < 0x1p16f) | !(fabsf(r.y) < 0x1p16f);
    return r;
}
// map_coord of a pixel index; the host only selects this kernel when the map is the identity or has
// mul, div > 0 of moderate size (then (x - in_min) * mul is +0 or inside the window of the exact two-step division)
GF_DEV float map_apply_int_lean(float x, const MapC& m) {
    if (m.identity) return (x - m.in_min) + m.add;
    const float a = (x - m.in_min) * m.mul;
    const float q0 = a * m.rcp;
    const float r0 = __fmaf_rn(-m.div, q0, a);
    return __fmaf_rn(r0, m.rcp, q0) + m.add;
}

// (v * 32).round() as i32 — f32::round is half away from zero.  Exact version: (double)t + (+-0.5) is exact for every float t
// below 2^28 and truncation toward zero of that sum is round-half-away; above, t is an integer already.  cvt.rzi.s32.f64 saturates
// like Rust's `as i32`, but the hardware turns NaN into INT_MIN where Rust gives 0, hence the select.
GF_DEV int round_away_i32(float t) {
    const double h = __hiloint2double((int)((__float_as_uint(t) & 0x80000000u) | 0x3fe00000u), 0);     // copysign(0.5, t)
    const int r = __double2int_rz((double)t + h);
    return t == t ? r : 0;
}

// Hot-path rounding without conversions (no XU / FP64 pipe work).  Input a2 = 2 * t (exact: t is scaled by a power of two).
// max(a2, -4) tames large negative values and NaN (fmaxf(NaN, -4) == -4); s = RZ(a2 + 2^23) puts floor(a2) in the mantissa
// for 0 <= a2 < 2^23, so w = bits(s) - 0x4affffff == floor(2t) + 1 and w >> 1 == floor(t + 1/2) == round-half-away(t).
// Contract of w >> 1 (checked by the self-test):  -1/4 < t < 2^22: the exact result;  t <= -1/4 or NaN: some value <= 0, and < 0
// whenever the exact result is < 0 (it may also be -1 where the exact result is 0);  t >= 2^22 (or +inf): some value >= 2^22.
// Callers either clamp to [0, lim] with lim < 2^22 (then the result is exact for every input except NaN -> 0, which is also
// what the reference gives) or treat every negative / huge result as "not interior" and recompute exactly out of line.
template <bool BOUNDED = false>     // BOUNDED: the caller guarantees |a2| < 2^23 (no NaN), the max() is not needed
GF_DEV void round_half_away_w(f2 a2, int& wa, int& wb) {
    float sa, sb;
    asm("{ .reg .b64 t, m, r; mov.b64 t, {%2, %3}; mov.b64 m, {%4, %4}; add.rz.f32x2 r, t, m; mov.b64 {%0, %1}, r; }"
        : "=f"(sa), "=f"(sb) : "f"(BOUNDED ? a2.x : fmaxf(a2.x, -4.0f)), "f"(BOUNDED ? a2.y : fmaxf(a2.y, -4.0f)), "f"(8388608.0f));
    wa = __float_as_int(sa) - 0x4affffff; wb = __float_as_int(sb) - 0x4affffff;
}
// max(min(round(t) as i32, lim), 0) for both lanes, 0 <= lim < 2^22
GF_DEV void round_away_clamped_x2(f2 t, int lim, int& ra, int& rb) {
    int wa, wb;
    round_half_away_w(p2::mul(t, p2::bc(2.0f)), wa, wb);
    ra = max(min(wa >> 1, lim), 0); rb = max(min(wb >> 1, lim), 0);
}

// everything that is not "valid pixel with an interior 8-bit bilinear footprint": background fill or the generic sampler,
// from the exact coordinates
template <class PIX>
static __device__ __noinline__ void shade_cold(bool ok, float u, float v, const WarpArgs& A, uint8_t* __restrict__ out) {
    constexpr int C = PIX::COUNT;
    float pixel[C];
    if (ok) {
        sample_generic<2, PIX>(round_away_i32(u * 32.0f), round_away_i32(v * 32.0f), A, pixel);
    } else {
        #pragma unroll
        for (int ch = 0; ch < C; ++ch) pixel[ch] = A.bg[ch];
    }
    PIX::store(out, true, pixel);
}

// warp-aggregated atomicAdd(counter, 1) over the active lanes (one atomic per warp); returns this lane's slot.  blockDim.x == 32.
GF_DEV unsigned warp_append(unsigned* counter) {
    const unsigned m = __activemask();
    const unsigned lane = threadIdx.x & 31u;
    const int leader = __ffs((int)m) - 1;
    unsigned base = 0;
    if ((int)lane == leader) base = atomicAdd(counter, (unsigned)__popc(m));
    base = __shfl_sync(m, base, leader);
    return base + (unsigned)__popc(m & ((1u << lane) - 1u));
}
// append the pair (x, y0), y0 even, to the frame's deferred-pair queue; false when the queue is full
GF_DEV bool defer_pair(const WarpArgs& A, int x, int y0) {
    const unsigned slot = warp_append(A.flt.count + GF_FLT_PAIRS);
    if (slot >= A.flt.cap) return false;
    A.flt.q[slot] = (uint32_t)x | ((uint32_t)(y0 >> 1) << 16);
    return true;
}
// append pixel (x, y) with its exact source coordinates to the frame's deferred-pixel queue; a full queue marks the frame for the
// tail launch's whole-frame re-render
GF_DEV void defer_pixel(const WarpArgs& A, int x, int y, float u, float v) {
    const unsigned slot = warp_append(A.flt.count + GF_FLT_PIXELS);
    if (slot < A.flt.cap_px) A.flt.qpx[slot] = make_uint4((uint32_t)x, (uint32_t)y, __float_as_uint(u), __float_as_uint(v));
    else A.flt.count[GF_FLT_OVERFLOW] = 1u;
}

// sampling + conversion + store of one pixel (x, y), lean feature set (no fix_range, background mode 0, pixel_value_limit >= max).
// wu, wv: round_half_away_w of 64 * u, 64 * v (8-bit formats only).  DEFER (filtered body): a pixel without an interior 8-bit
// footprint goes to the deferred-pixel queue, which the tail launch finishes with shade_cold from the same u, v.
template <class PIX, bool DEFER = false>
GF_DEV void shade_lean(bool ok, bool far, float u, float v, int wu, int wv, const WarpArgs& A, uint8_t* __restrict__ out, int x, int y) {
    constexpr int C = PIX::COUNT;
    if (PIX::SCALAR == SC_U8) {
        const int sx0 = wu >> 1, sy0 = wv >> 1;
        const int sx = sx0 >> 5, sy = sy0 >> 5;
        // interior_span < 2^17 (host): negative and >= 2^22 results of the rounding shortcut can never pass
        const bool interior = ok & !far & ((unsigned)(sx - A.hot.rect[0]) <= (unsigned)A.hot.rect[2]) & ((unsigned)(sy - A.hot.rect[1]) <= (unsigned)A.hot.rect[3]);
        if (interior) {
            uint32_t N[C], s[C];
            sample_u8_bilinear<PIX>(sx0, sy0, A, N);
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) s[ch] = N[ch] >> 10;      // trunc(N / 1024); N / 1024 <= 255 <= pixel_value_limit
            PIX::store_scalars(out, true, s);
        } else if (DEFER) {
            defer_pixel(A, x, y, u, v);
        } else {
            shade_cold<PIX>(ok, u, v, A, out);
        }
    } else {
        float pixel[C];
        if (ok) {
            sample_input_at<2, PIX, false>(u, v, A, pixel);
        } else {
            #pragma unroll
            for (int ch = 0; ch < C; ++ch) pixel[ch] = A.bg[ch];
        }
        PIX::store(out, true, pixel);
    }
}

#define GF_X2_ROWS_PER_BLOCK (2 * GF_BLOCK_Y)

// COORD: pass 1 of the two-pass mode — write the coordinates to A.coord_out instead of sampling (pixel-format independent: the
// pixel size then comes from KernelParams, PIX is a placeholder).
// exact_prepass: evaluate the mid-row transform with the reference's own arithmetic (always true unless the frame runs the filtered
// pre-pass; true as well for the pairs the tail launch re-renders)
// FILTERED: the main launch of a filtered frame (trusted tables, fused sampling).  Everything rare leaves the launch instead of running
// inline, so the body holds no call: an uncertified row or a `bad` pair goes to the deferred-pair queue (neither pixel written), a
// pixel without an interior 8-bit footprint to the deferred-pixel queue, and a full queue to the tail's whole-frame re-render.
template <int LENS, int DIGITAL, class PIX, bool TRUSTED, bool COORD, bool FILTERED = false>
GF_DEV void warp_x2_body(const WarpArgs& A, const int x, const int y0, const bool exact_prepass) {
    using namespace p2;
    static_assert(!FILTERED || (TRUSTED && !COORD && LensApprox<LENS>::value && DIGITAL == GF_LENS_NONE), "filtered body: trusted fused fisheye only");
    const gf_kernel_params& P = A.p;
    if (x >= A.out_cols || y0 >= A.out_rows) return;
    const unsigned long long BYTES = COORD ? (unsigned long long)P.bytes_per_pixel : (unsigned long long)PIX::BYTES;
    const unsigned long long ostride = (unsigned long long)P.output_stride;
    const unsigned long long off_a = (unsigned long long)y0 * ostride + (unsigned long long)x * BYTES;
    const unsigned long long off_b = off_a + ostride;
    // lane validity: row exists, pixel fits in the buffer (short last row), bounds test of :551
    float opx, opy_a, opy_b;
    bool wr_a, wr_b;
    if (A.feat & F_INTPRO) {                                 // identity rect maps: the same tests on integers (host: fill_uniforms)
        const bool in_x = (x >= A.hot.x0) & (x < A.hot.x1);
        const int y1 = y0 + 1;
        wr_a = in_x & (y0 >= A.hot.y0) & (y0 < A.hot.y1) & ((y0 < A.hot.full_rows) | ((y0 == A.hot.full_rows) & (x < A.hot.last_cols)));
        wr_b = in_x & (y1 >= A.hot.y0) & (y1 < A.hot.y1) & ((y1 < A.hot.full_rows) | ((y1 == A.hot.full_rows) & (x < A.hot.last_cols)));
        opx = (float)(x + A.hot.x_off); opy_a = (float)(y0 + A.hot.y_off); opy_b = (float)(y1 + A.hot.y_off);
    } else {
        opx = map_apply_int_lean((float)x, A.omap_x);
        opy_a = map_apply_int_lean((float)y0, A.omap_y);
        opy_b = map_apply_int_lean((float)(y0 + 1), A.omap_y);
        const bool in_x = (opx >= 0.0f) & (as_i32(opx) < P.output_width);
        wr_a = in_x & (off_a + BYTES <= A.dst_len) & (opy_a >= 0.0f) & (as_i32(opy_a) < P.output_height);
        wr_b = in_x & ((y0 + 1) < A.out_rows) & (off_b + BYTES <= A.dst_len) & (opy_b >= 0.0f) & (as_i32(opy_b) < P.output_height);
    }
    uint2* const cm_a = COORD ? A.coord_out + ((size_t)y0 * (size_t)A.out_cols + (size_t)x) : nullptr;
    const bool row_b = (y0 + 1) < A.out_rows;
    if (!(wr_a | wr_b)) {
        if (COORD) { *cm_a = make_uint2(GF_COORD_MARK, GF_COORD_SKIP); if (row_b) cm_a[A.out_cols] = make_uint2(GF_COORD_MARK, GF_COORD_SKIP); }
        return;
    }

    // undistort_coord, :421-517
    const float pxs = opx + P.translation2d[0];
    const f2 px = bc(pxs);
    const f2 py = mk(opy_a + P.translation2d[1], opy_b + P.translation2d[1]);
    const int lim = A.rs_lim;
    int sy_a, sy_b;
    round_away_clamped_x2(py, lim, sy_a, sy_b);                                                         // :465-469
    bool have_row = false;
    if constexpr (TRUSTED && LensApprox<LENS>::value && DIGITAL == GF_LENS_NONE) if (FILTERED || !exact_prepass) {  // F_FILTER & F_RS (host)
        // :470-479, filtered: certify round(v_mid) from the approximate evaluation, defer the pair when it cannot be
        const MatRow9 rm = load_row9(A.matrices, (uint32_t)P.matrix_count / 2u);
        const float bx = pxs * rm.m01.x, by = pxs * rm.m23.y, bw = pxs * rm.m67.x;                      // the reference's products and sums, unfused
        const float xa = (bx + py.x * rm.m01.y) + rm.m23.x, xb = (bx + py.y * rm.m01.y) + rm.m23.x;
        const float ya = (by + py.x * rm.m45.x) + rm.m45.y, yb = (by + py.y * rm.m45.x) + rm.m45.y;
        const float wa = (bw + py.x * rm.m67.y) + rm.m8,    wb = (bw + py.y * rm.m67.y) + rm.m8;
        float ca, cb;
        const bool ra = Lens2<LENS>::approx_v(xa, ya, wa, P, A.flt.a_cap, ca);
        const bool rb = Lens2<LENS>::approx_v(xb, yb, wb, P, A.flt.a_cap, cb);
        const float ta = ca + P.c[1], tb = cb + P.c[1];
        // distance of t to the nearest rounding boundary n + 1/2 (|t| < 2^20: the magic-number rounding is exact)
        const float za = ta - 0.5f, zb = tb - 0.5f;
        const float da = fabsf(za - ((za + 12582912.0f) - 12582912.0f)), db = fabsf(zb - ((zb + 12582912.0f) - 12582912.0f));
        const float ea = __fmaf_rn(fabsf(ca), A.flt.rho, fabsf(ta) * 0x1p-22f), eb = __fmaf_rn(fabsf(cb), A.flt.rho, fabsf(tb) * 0x1p-22f);
        const bool sure = ra & rb & (da > ea) & (db > eb) & (fabsf(ta) < 0x1p20f) & (fabsf(tb) < 0x1p20f);
        if (sure) {
            round_away_clamped_x2(mk(ta, tb), lim, sy_a, sy_b);
            have_row = true;
        } else {                                         // append the pair to the frame's queue, rendered by the tail launch
            if (defer_pair(A, x, y0)) return;
            if (FILTERED) { A.flt.count[GF_FLT_OVERFLOW] = 1u; return; }
            // queue full: this thread evaluates the exact pre-pass itself
        }
    }
    if (!FILTERED && (A.feat & F_RS) && !have_row) {                                                    // :470-479
        const uint32_t mid = (uint32_t)P.matrix_count / 2u;
        f2 tu, tv; bool oa = true, ob = true, bad = false;
        rotate_and_distort_x2<LENS, DIGITAL, TRUSTED>(px, py, mid, mid, A, tu, tv, bad);
        if (bad) {                                       // cold: exact scalar code for both pixels
            const PairUV c = rotate_and_distort_cold<LENS, DIGITAL>(pxs, py.x, py.y, mid, mid, A, 0);
            oa = (c.ok & 1) != 0; ob = (c.ok & 2) != 0; tv = mk(c.va, c.vb);
        }
        int ra, rb;
        round_away_clamped_x2(tv, lim, ra, rb);
        sy_a = oa ? ra : sy_a; sy_b = ob ? rb : sy_b;
    }
    const uint32_t last = (uint32_t)(P.matrix_count - 1);
    const uint32_t idx_a = min((uint32_t)sy_a, last), idx_b = min((uint32_t)sy_b, last);               // :482
    f2 u, v; bool ok_a = true, ok_b = true, far_a = false, far_b = false, bad = false;
    rotate_and_distort_x2<LENS, DIGITAL, TRUSTED>(px, py, idx_a, idx_b, A, u, v, bad);                           // :483
    u = map_apply_x2(u, A.smap_x, bad);                                                                 // :510-515
    v = map_apply_x2(v, A.smap_y, bad);
    if (FILTERED && bad) {                               // the tail renders the pair from scratch
        warp_append(A.flt.count + GF_FLT_BAD);
        if (!defer_pair(A, x, y0)) A.flt.count[GF_FLT_OVERFLOW] = 1u;
        return;
    }
    if (!FILTERED && bad) {
        const PairUV c = rotate_and_distort_cold<LENS, DIGITAL>(pxs, py.x, py.y, idx_a, idx_b, A, 1);
        ok_a = (c.ok & 1) != 0; ok_b = (c.ok & 2) != 0; far_a = (c.ok & 4) != 0; far_b = (c.ok & 8) != 0;
        u = mk(c.ua, c.ub); v = mk(c.va, c.vb);
    }

    if (COORD) {      // the exact coordinates (hot or cold path alike); None / not-written pixels as markers
        *cm_a = !wr_a ? make_uint2(GF_COORD_MARK, GF_COORD_SKIP) : (ok_a ? make_uint2(__float_as_uint(u.x), __float_as_uint(v.x)) : make_uint2(GF_COORD_MARK, GF_COORD_NONE));
        if (row_b) cm_a[A.out_cols] = !wr_b ? make_uint2(GF_COORD_MARK, GF_COORD_SKIP) : (ok_b ? make_uint2(__float_as_uint(u.y), __float_as_uint(v.y)) : make_uint2(GF_COORD_MARK, GF_COORD_NONE));
        return;
    }
    int wu_a = 0, wu_b = 0, wv_a = 0, wv_b = 0;
    if (PIX::SCALAR == SC_U8) {                          // (u * 32).round() for both pixels: 64 * u == 2 * (32 * u) exactly.
        // |u|, |v| < 2^16 here unless far_* is set (then the result is not used), so the unguarded form of the shortcut applies;
        // a garbage value for a far lane is harmless because `interior` below is false for it
        round_half_away_w<true>(mul(u, bc(64.0f)), wu_a, wu_b);
        round_half_away_w<true>(mul(v, bc(64.0f)), wv_a, wv_b);
    }
    if constexpr (FILTERED) {
        // the offsets are recomputed here (the empty asm keeps the compiler from reusing the prologue's): kept live from the prologue,
        // the two 64-bit values were spilled across the whole evaluation under the register cap
        int xs = x, ys = y0;
        asm("" : "+r"(xs), "+r"(ys));
        const unsigned long long o = (unsigned long long)ys * ostride + (unsigned long long)xs * BYTES;
        if (wr_a) shade_lean<PIX, true>(true, false, u.x, v.x, wu_a, wv_a, A, A.dst + o, xs, ys);       // :615-622
        if (wr_b) shade_lean<PIX, true>(true, false, u.y, v.y, wu_b, wv_b, A, A.dst + o + ostride, xs, ys + 1);
    } else {
        if (wr_a) shade_lean<PIX>(ok_a, far_a, u.x, v.x, wu_a, wv_a, A, A.dst + off_a, x, y0);           // :615-622
        if (wr_b) shade_lean<PIX>(ok_b, far_b, u.y, v.y, wu_b, wv_b, A, A.dst + off_b, x, y0 + 1);
    }
}

// The kernel: both table-trust variants in one launch, selected by a DEVICE word.  `A.table_flags` points to the verdict on the
// matrix table this frame reads — written on the same stream by whoever produced the table (the host scan of host tables via a
// context-owned constant, gf_cuda_scan_tables_dev for caller-owned device tables, or the on-device producer
// gf_cuda_frame_transform_dev itself): 0 = every entry zero or 2^-40..2^40 and no IBIS rows.  Trust is therefore a property of
// the bytes the kernel is about to read, ordered by the stream — not of a host-side pointer cache.  The branch is uniform.
//
// Filtered frames (F_FILTER, host-selected: trusted-capable lens with an approximate form, rolling shutter on) launch two kernels.  The
// main launch (FILTERED instantiation; COORD: this one) certifies each pair's matrix row from the approximate mid-row evaluation and
// sends what it cannot finish cheaply to the frame's queues: uncertified and `bad` pairs, and pixels whose 8-bit footprint is not
// interior.  The tail launch (A.flt.tail, a small grid-stride grid, always this unfiltered instantiation) renders the deferred pairs with
// the exact pre-pass and finishes the deferred pixels with shade_cold; if a queue overflowed it re-renders the whole frame instead.
template <int LENS, int DIGITAL, class PIX, int MINB, bool COORD = false, bool FILTERED = false>
__global__ void __launch_bounds__(GF_BLOCK_X * GF_BLOCK_Y, MINB)
warp_kernel_x2(const __grid_constant__ WarpArgs A) {
    constexpr bool kFilter = LensApprox<LENS>::value && DIGITAL == GF_LENS_NONE;
    // launched with programmatic stream serialization (c_abi.cu: launch_pdl): nothing of the previous kernel on the stream — the matrix
    // table and its verdict word, the deferred queues and their counters, the previous frame's output — may be read or written before this
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const bool trusted = __ldg(A.table_flags) == 0u;
    if constexpr (kFilter && !FILTERED) if (A.flt.tail) {
        const unsigned tid = (blockIdx.y * gridDim.x + blockIdx.x) * (blockDim.x * blockDim.y) + threadIdx.y * blockDim.x + threadIdx.x;
        if (tid == 0u) {                                              // re-arm the counters the NEXT frame's main launch will use
            #pragma unroll
            for (int i = 0; i < GF_FLT_WORDS; ++i) A.flt.count_next[i] = 0u;
        }
        if (!trusted) return;                                         // the main launch deferred nothing on the guarded path
        const unsigned stride = gridDim.x * gridDim.y * blockDim.x * blockDim.y;
        // a full queue left pixels missing anywhere in the frame: then every pair is rendered, else the deferred pairs, then the pixels
        const bool all = A.flt.count[GF_FLT_OVERFLOW] != 0u;
        const unsigned long long cols = (unsigned long long)A.out_cols;
        const unsigned long long np = all ? cols * (unsigned long long)((A.out_rows + 1) / 2) : min(A.flt.count[GF_FLT_PAIRS], A.flt.cap);
        const unsigned long long n = np + ((all || COORD) ? 0u : min(A.flt.count[GF_FLT_PIXELS], A.flt.cap_px));
        for (unsigned long long i = tid; i < n; i += stride) {
            if (i < np) {
                int px, py0;
                if (all) { px = (int)(i % cols); py0 = (int)(i / cols) * 2; }
                else     { const uint32_t e = A.flt.q[i]; px = (int)(e & 0xffffu); py0 = (int)(e >> 16) * 2; }
                warp_x2_body<LENS, DIGITAL, PIX, true, COORD>(A, px, py0, true);
            } else if constexpr (!COORD && PIX::SCALAR == SC_U8) {
                const uint4 e = A.flt.qpx[i - np];
                const unsigned long long off = (unsigned long long)e.y * (unsigned long long)A.p.output_stride + (unsigned long long)e.x * PIX::BYTES;
                shade_cold<PIX>(true, __uint_as_float(e.z), __uint_as_float(e.w), A, A.dst + off);
            }
        }
        return;
    }
    const int x = blockIdx.x * GF_BLOCK_X + threadIdx.x;
    const int y0 = (blockIdx.y * blockDim.y + threadIdx.y) * 2;          // blockDim.y: the host may launch flatter blocks (GF_X2_BLOCK_Y)
    if (trusted) {
        if constexpr (FILTERED) warp_x2_body<LENS, DIGITAL, PIX, true, false, true>(A, x, y0, false);
        else warp_x2_body<LENS, DIGITAL, PIX, true, COORD>(A, x, y0, !(COORD && kFilter && (A.feat & F_FILTER)));
    } else {
        warp_x2_body<LENS, DIGITAL, PIX, false, COORD>(A, x, y0, true);
    }
}

} // namespace gf
