// c_abi_internal.h — entry points shared between the translation units of libgyroflow_cuda.so, NOT exported
// (the library is built with -fvisibility=hidden; only GF_API symbols leave it).
#pragma once
#include <cstddef>
#include <cstdint>
#include "../../include/gyroflow_cuda.h"

// One frame through the warp with a DEVICE matrix table + verdict word, never synchronising: HOST image buffers (page-locked) are
// copied on `cu_stream` before / after the kernel.  `checksum_dev` (nullable): the output buffer's checksum is accumulated into it
// on the same stream, between the kernel and the device-to-host copy.  Used by the render queue.
int gf_internal_run_frame(gf_cuda_ctx* ctx, const gf_buffer_desc* in, const gf_buffer_desc* out, const gf_kernel_params* params,
                          const float* matrices_dev, size_t matrix_rows, const float* mesh_dev, size_t mesh_len,
                          const uint32_t* table_flags_dev, void* cu_stream, uint64_t* checksum_dev);

// Can two planes of one frame share one coordinate pass (gf_cuda_undistort_planes_dev_flagged fuses planes for which this holds)?
bool gf_internal_same_plane_geometry(const gf_kernel_params* pa, const gf_buffer_desc* ia, const gf_buffer_desc* oa,
                                     const gf_kernel_params* pb, const gf_buffer_desc* ib, const gf_buffer_desc* ob);

// Preview overlays (overlay.cu): draw_pixel + draw_safe_area of opencl_undistort.cl:109-154 as a pass over a DEVICE buffer.
// count / scalar: channels and scalar kind (0 u8, 1 u16, 2 f32, 3 f16) of the pixel type.
int gf_internal_draw_overlays(void* cu_stream, uint8_t* buf_dev, size_t len, int width, int height, int stride, const gf_kernel_params* p,
                              int count, int scalar, int is_input, const uint8_t* drawing_dev, size_t drawing_len);
