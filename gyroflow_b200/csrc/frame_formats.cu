// frame_formats.cu — the decoder-frame plane table of rendering/mod.rs:563-651 and PixelType::from_rgb_color (pixel_formats.rs:23-48
// plus the per-type impls), host only.  The render queue's frame mode (render_queue.cu) builds every plane's KernelParams from these.
// This TU is built with -ffp-contract=off: rgb_to_yuv must round every f32 product and sum on its own, like the Rust code.
#include <cstring>
#include <cmath>
#include "../../include/gyroflow_cuda.h"

namespace {

struct PlaneRow { int pix; int size_plane; int n_ind; int ind[4]; float max_value; };
struct FormatRow { int log2_cw, log2_ch; int n_planes; PlaneRow planes[GF_FRAME_MAX_PLANES]; };

// (type, $ind, $yuvi, $max_val) per plane, rows in the order of the match at rendering/mod.rs:563-651
#define P1(t, i, v, m)          { t, i, 1, { v, 0, 0, 0 }, m }
#define LUMA_UV(t1, t2, u, v, m) { P1(t1, 0, 0, m), { t2, 1, 2, { u, v, 0, 0 }, m } }
#define YUV3(t, m)              { P1(t, 0, 0, m), P1(t, 1, 1, m), P1(t, 2, 2, m) }
#define YUV4(t, m)              { P1(t, 0, 0, m), P1(t, 1, 1, m), P1(t, 2, 2, m), P1(t, 3, 3, m) }
#define PACKED(t, m)            { { t, 0, 0, { 0, 0, 0, 0 }, m } }
const FormatRow kFormats[GF_FRAME_COUNT] = {
    { 1, 1, 2, LUMA_UV(GF_PIX_LUMA8, GF_PIX_UV8, 1, 2, 255.0f) },            // NV12                  :564-569
    { 1, 1, 2, LUMA_UV(GF_PIX_LUMA8, GF_PIX_UV8, 2, 1, 255.0f) },            // NV21                  :570-575
    { 1, 1, 2, LUMA_UV(GF_PIX_LUMA16, GF_PIX_UV16, 1, 2, 65535.0f) },        // P010LE                :576-588 (65535 for every P0xx)
    { 1, 1, 2, LUMA_UV(GF_PIX_LUMA16, GF_PIX_UV16, 1, 2, 65535.0f) },        // P016LE
    { 1, 0, 2, LUMA_UV(GF_PIX_LUMA16, GF_PIX_UV16, 1, 2, 65535.0f) },        // P210LE
    { 1, 0, 2, LUMA_UV(GF_PIX_LUMA16, GF_PIX_UV16, 1, 2, 65535.0f) },        // P216LE
    { 0, 0, 2, LUMA_UV(GF_PIX_LUMA16, GF_PIX_UV16, 1, 2, 65535.0f) },        // P410LE
    { 0, 0, 2, LUMA_UV(GF_PIX_LUMA16, GF_PIX_UV16, 1, 2, 65535.0f) },        // P416LE
    { 1, 1, 3, YUV3(GF_PIX_LUMA8, 255.0f) },                                  // YUV420P               :589-595
    { 1, 1, 3, YUV3(GF_PIX_LUMA8, 255.0f) },                                  // YUVJ420P
    { 1, 1, 3, YUV3(GF_PIX_LUMA16, 1023.0f) },                                // YUV420P10LE           :596-610
    { 1, 1, 3, YUV3(GF_PIX_LUMA16, 4095.0f) },                                // YUV420P12LE
    { 1, 1, 3, YUV3(GF_PIX_LUMA16, 16383.0f) },                               // YUV420P14LE
    { 1, 1, 3, YUV3(GF_PIX_LUMA16, 65535.0f) },                               // YUV420P16LE
    { 1, 0, 3, YUV3(GF_PIX_LUMA16, 1023.0f) },                                // YUV422P10LE
    { 1, 0, 3, YUV3(GF_PIX_LUMA16, 4095.0f) },                                // YUV422P12LE
    { 1, 0, 3, YUV3(GF_PIX_LUMA16, 16383.0f) },                               // YUV422P14LE
    { 1, 0, 3, YUV3(GF_PIX_LUMA16, 65535.0f) },                               // YUV422P16LE
    { 0, 0, 3, YUV3(GF_PIX_LUMA16, 1023.0f) },                                // YUV444P10LE
    { 0, 0, 3, YUV3(GF_PIX_LUMA16, 4095.0f) },                                // YUV444P12LE
    { 0, 0, 3, YUV3(GF_PIX_LUMA16, 16383.0f) },                               // YUV444P14LE
    { 0, 0, 3, YUV3(GF_PIX_LUMA16, 65535.0f) },                               // YUV444P16LE
    { 0, 0, 4, YUV4(GF_PIX_LUMA16, 1023.0f) },                                // YUVA444P10LE          :611-623
    { 0, 0, 4, YUV4(GF_PIX_LUMA16, 4095.0f) },                                // YUVA444P12LE
    { 0, 0, 4, YUV4(GF_PIX_LUMA16, 65535.0f) },                               // YUVA444P16LE
    { 0, 0, 4, { P1(GF_PIX_R32F, 0, 2, 255.0f), P1(GF_PIX_R32F, 0, 0, 255.0f), P1(GF_PIX_R32F, 0, 1, 255.0f), P1(GF_PIX_R32F, 0, 3, 255.0f) } },  // GBRAPF32LE :624-629
    { 0, 0, 3, { P1(GF_PIX_R32F, 0, 2, 255.0f), P1(GF_PIX_R32F, 0, 0, 255.0f), P1(GF_PIX_R32F, 0, 1, 255.0f) } },                               // GBRPF32LE  :630-634
    { 0, 0, 1, { { GF_PIX_AYUV16, 0, 4, { 3, 0, 1, 2 }, 65535.0f } } },     // AYUV64LE              :635
    { 0, 0, 1, PACKED(GF_PIX_RGB8, 255.0f) },                                 // RGB24                 :636
    { 0, 0, 1, PACKED(GF_PIX_RGBA8, 255.0f) },                                // RGBA                  :637
    { 0, 0, 1, PACKED(GF_PIX_RGB16, 65535.0f) },                              // RGB48BE               :638
    { 0, 0, 1, PACKED(GF_PIX_RGBA16, 65535.0f) },                             // RGBA64BE              :639
};
#undef P1
#undef LUMA_UV
#undef YUV3
#undef YUV4
#undef PACKED

// rgb_to_yuv, pixel_formats.rs:23-48.  The constants are f32 constant expressions in Rust, evaluated in f32.
void rgb_to_yuv(const float v[4], bool is_limited, float out[4]) {
    const float KR = 0.2126f, KB = 0.0722f;
    const float KG = 1.0f - KR - KB;
    const float US = 1.0f / (2.0f - 2.0f * KB);
    const float VS = 1.0f / (2.0f - 2.0f * KR);
    auto clamp01 = [](float x) { return fminf(fmaxf(x, 0.0f), 1.0f); };      // f32::max / f32::min: a NaN operand yields the other one
    out[0] = clamp01(KR * v[0] + KG * v[1] + KB * v[2]);
    out[1] = clamp01((-KR * US) * v[0] + (-KG * US) * v[1] + ((1.0f - KB) * US) * v[2] + 0.5f);
    out[2] = clamp01(((1.0f - KR) * VS) * v[0] + (-KG * VS) * v[1] + (-KB * VS) * v[2] + 0.5f);
    out[3] = clamp01(v[3]);
    if (is_limited) {                                                          // remap_to_limited
        out[0] = (16.0f / 255.0f) + (out[0] * ((235.0f - 16.0f) / 255.0f));
        out[1] = (16.0f / 255.0f) + (out[1] * ((240.0f - 16.0f) / 255.0f));
        out[2] = (16.0f / 255.0f) + (out[2] * ((240.0f - 16.0f) / 255.0f));
    }
}

} // namespace

extern "C" {

GF_API int gf_frame_layout(int format, int32_t width, int32_t height, gf_plane_spec* out, size_t* n) {
    if (format < 0 || format >= GF_FRAME_COUNT || width < 1 || height < 1 || !out || !n) return GF_ERR_BAD_PARAMS;
    const FormatRow& f = kFormats[format];
    for (int i = 0; i < f.n_planes; ++i) {
        const PlaneRow& r = f.planes[i];
        gf_plane_spec& s = out[i];
        memset(&s, 0, sizeof(s));
        s.pixel_type = r.pix;
        const bool chroma = r.size_plane == 1 || r.size_plane == 2;           // av_image plane_width: planes 1 and 2 carry the chroma shift
        s.width  = chroma ? -((-width)  >> f.log2_cw) : width;
        s.height = chroma ? -((-height) >> f.log2_ch) : height;
        s.n_ind = r.n_ind;
        for (int k = 0; k < 4; ++k) s.ind[k] = r.ind[k];
        s.max_value = r.max_value;
    }
    *n = (size_t)f.n_planes;
    return GF_OK;
}

GF_API int gf_background_for_plane(int pixel_type, const float rgb[4], const int32_t* ind, size_t n_ind, int is_limited, float out[4]) {
    if (!rgb || !out || (n_ind && !ind)) return GF_ERR_BAD_PARAMS;
    size_t need = 0;
    switch (pixel_type) {
    case GF_PIX_LUMA8: case GF_PIX_LUMA16: case GF_PIX_R32F: need = 1; break;
    case GF_PIX_UV8: case GF_PIX_UV16: need = 2; break;
    case GF_PIX_AYUV16: need = 4; break;
    case GF_PIX_RGB8: case GF_PIX_RGBA8: case GF_PIX_BGRA8: case GF_PIX_RGB16: case GF_PIX_RGBA16: case GF_PIX_RGBAF: case GF_PIX_RGBAF16: break;
    default: return GF_ERR_BAD_PARAMS;
    }
    if (n_ind < need) return GF_ERR_BAD_PARAMS;
    for (size_t i = 0; i < need; ++i) if (ind[i] < 0 || ind[i] > 3) return GF_ERR_BAD_PARAMS;
    float yuv[4];
    rgb_to_yuv(rgb, is_limited != 0, yuv);
    switch (pixel_type) {
    case GF_PIX_LUMA8: case GF_PIX_LUMA16:                                     // :77, :95
        out[0] = yuv[ind[0]]; out[1] = out[2] = out[3] = 0.0f; break;
    case GF_PIX_UV8: case GF_PIX_UV16:                                         // :280, :298
        out[0] = yuv[ind[0]]; out[1] = yuv[ind[1]]; out[2] = out[3] = 0.0f; break;
    case GF_PIX_AYUV16:                                                        // :203
        for (int i = 0; i < 4; ++i) out[i] = yuv[ind[i]];
        break;
    case GF_PIX_R32F:                                                          // :262 — no YUV conversion, the RGB component itself
        out[0] = rgb[ind[0]]; out[1] = out[2] = out[3] = 0.0f; break;
    case GF_PIX_BGRA8:                                                         // :149
        out[0] = rgb[2]; out[1] = rgb[1]; out[2] = rgb[0]; out[3] = rgb[3]; break;
    default:                                                                   // RGB8, RGBA8, RGB16, RGBA16, RGBAf, RGBAf16: unchanged
        for (int i = 0; i < 4; ++i) out[i] = rgb[i];
        break;
    }
    return GF_OK;
}

} // extern "C"
