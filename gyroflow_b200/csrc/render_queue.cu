// render_queue.cu — the frame-sharded render queue of one GPU (SURVEY §8e, §7.9).
//
// What the reference does per frame on the render path (rendering/mod.rs:451,531-542,657-661): the ffmpeg frame callback calls
// `Stabilization::get_frame_transform_at` (FrameTransform::at_timestamp + the per-buffer fields) and then `process_pixels`,
// strictly one frame after another on one device; `render_queue.rs:550-612` only runs whole jobs side by side.  Frames are
// independent units (at_timestamp depends on immutable ComputeParams + the timestamp, frame_transform.rs:165), so this queue keeps
// `depth` of them in flight on one GPU and lets a box shard `i -> GPU (i mod G)` across processes with no data-path collective.
//
// One slot = one stream + one warp context (its own device staging when the buffers are HOST) + a device matrix table with its
// trust verdict word.  Per submitted frame, all enqueued on the slot's stream, nothing synchronous:
//     producer kernel (gf_cuda_frame_transform_dev_flagged: table + verdict)  ->  [mesh H2D]  ->  [frame H2D]  ->  warp kernel
//     ->  [checksum kernel]  ->  [frame D2H]  ->  event
// Slots are used round-robin; submit() waits for a slot's previous frame only when it comes round again, wait() hands finished
// frames back in submission order (output order restored by frame index on the host, as §8e asks).
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <sched.h>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <vector>
#include <deque>
#include <algorithm>
#include "../../include/gyroflow_cuda.h"
#include "c_abi_internal.h"

namespace {

struct QSlot {
    gf_cuda_ctx* ctx = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    float* d_mat = nullptr;
    uint32_t* d_flags = nullptr;
    float* h_mesh = nullptr; float* d_mesh = nullptr;      // per-frame mesh staging (pinned / device)
    uint64_t* d_sum = nullptr; uint64_t* h_sum = nullptr;  // checksums, one per plane (device words, pinned host copies)
    // frame mode: one warp context per distinct pixel type of the format, device staging per HOST plane
    std::vector<gf_cuda_ctx*> pix_ctx;
    std::vector<uint8_t*> d_in, d_out;
    bool busy = false;
    size_t frame = 0;
};

// sum(word[i] * (2 i + 1)) mod 2^64: order-independent, so blocks may add their partial sums in any order
__global__ void checksum_kernel(const uint32_t* __restrict__ w, size_t n, unsigned long long* __restrict__ out) {
    unsigned long long s = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        s += (unsigned long long)w[i] * (2ull * (unsigned long long)i + 1ull);
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31u) == 0u && s) atomicAdd(out, s);
}

// One launch for every plane of a frame: blockIdx.y picks the plane, out[plane] = sum(word[i] * (2 i + 1)) over that plane's words
struct PlaneWords { const uint32_t* w[GF_FRAME_MAX_PLANES]; size_t n[GF_FRAME_MAX_PLANES]; };
__global__ void checksum_planes_kernel(const __grid_constant__ PlaneWords p, unsigned long long* __restrict__ out) {   // grid constant: indexed in place, no local copy
    const uint32_t* __restrict__ w = p.w[blockIdx.y];
    const size_t n = p.n[blockIdx.y];
    unsigned long long s = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        s += (unsigned long long)w[i] * (2ull * (unsigned long long)i + 1ull);
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31u) == 0u && s) atomicAdd(out + blockIdx.y, s);
}

} // namespace

struct gf_cuda_queue {
    gf_queue_config cfg;
    gf_compute_params cp;                 // shallow copy: the arrays it points to stay owned by the caller for the queue's lifetime
    gf_cuda_gyro* gyro = nullptr;
    std::vector<QSlot> slots;
    std::deque<int> fifo;                 // slots in submission order
    int next = 0;
    size_t max_rows = 0;
    unsigned long long launches = 0;
    std::string last_error;
    // frame mode (gf_cuda_queue_create_frame); empty for a single-buffer queue
    std::vector<gf_plane_spec> planes, out_planes;       // input / output layout
    std::vector<gf_stab_config> plane_stab;              // cfg.stab with the plane's pixel type and converted background
    std::vector<int> plane_ctx;                          // index into QSlot::pix_ctx
    std::vector<int> plane_kind_in, plane_kind_out;      // GF_BUF_* of the prototypes
    std::vector<size_t> plane_len_in, plane_len_out;     // staging sizes (HOST planes)
};

namespace {
int qfail(gf_cuda_queue* q, int code, const std::string& msg) { if (q) q->last_error = msg; return code; }
int qcuda(gf_cuda_queue* q, cudaError_t e, const char* what) {
    return qfail(q, GF_ERR_CUDA, std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}
#define QCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return qcuda(q, e_, #call); } while (0)

// stream, event, device table + verdict word, mesh staging, checksum words: what every slot has in both modes
int alloc_slot(gf_cuda_queue* q, QSlot& s) {
    QCK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    QCK(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    QCK(cudaMalloc(&s.d_mat, q->max_rows * GF_MATRIX_STRIDE * sizeof(float)));
    QCK(cudaMalloc(&s.d_flags, sizeof(uint32_t)));
    QCK(cudaMallocHost(&s.h_mesh, GF_MESH_MAX_LEN * sizeof(float)));
    QCK(cudaMalloc(&s.d_mesh, GF_MESH_MAX_LEN * sizeof(float)));
    QCK(cudaMalloc(&s.d_sum, GF_FRAME_MAX_PLANES * sizeof(uint64_t)));
    QCK(cudaMallocHost(&s.h_sum, GF_FRAME_MAX_PLANES * sizeof(uint64_t)));
    memset(s.h_sum, 0, GF_FRAME_MAX_PLANES * sizeof(uint64_t));
    return GF_OK;
}

int finish_slot(gf_cuda_queue* q, QSlot& s) {
    if (!s.busy) return GF_OK;
    QCK(cudaEventSynchronize(s.done));
    s.busy = false;
    return GF_OK;
}
} // namespace

extern "C" {

GF_API int gf_cuda_bind_thread_to_device(int device) {
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) { (void)cudaGetLastError(); return GF_ERR_CUDA; }
    for (char* c = bdf; *c; ++c) if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');      // sysfs uses lower-case hex
    char path[128];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", bdf);
    FILE* f = fopen(path, "r");
    if (!f) return 0;
    char line[1024] = {0};
    const bool got = fgets(line, sizeof(line), f) != nullptr;
    fclose(f);
    if (!got) return 0;
    cpu_set_t want, have;
    CPU_ZERO(&want);
    int n = 0;
    for (char* tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {                  // "32-63,96-127"
        int a = 0, b = 0;
        const int k = sscanf(tok, "%d-%d", &a, &b);
        if (k == 1) b = a;
        if (k < 1 || a < 0 || b < a) continue;
        for (int c = a; c <= b && c < CPU_SETSIZE; ++c) CPU_SET(c, &want);
    }
    // stay inside what the process is allowed to use (cgroup / taskset): intersect, and keep the old mask if the intersection is empty
    if (sched_getaffinity(0, sizeof(have), &have) == 0) {
        cpu_set_t both; CPU_AND(&both, &want, &have);
        if (CPU_COUNT(&both) == 0) return 0;
        want = both;
    }
    n = CPU_COUNT(&want);
    if (n == 0) return 0;
    if (sched_setaffinity(0, sizeof(want), &want) != 0) return GF_ERR_BAD_PARAMS;
    return n;
}

// Page-lock an existing host allocation (the decoder's frame pool, a long-lived Vec<u8>) so that HOST-buffer calls copy at the link's rate
// instead of through the driver's bounce buffers (bench: 742 vs 262 sequential 4K frames/s).  Thin wrappers over cudaHostRegister /
// cudaHostUnregister: the caller owns the lifetime — unregister before the memory is freed.
GF_API int gf_cuda_host_register(void* ptr, size_t len) {
    if (!ptr || !len) return GF_ERR_BAD_PARAMS;
    const cudaError_t e = cudaHostRegister(ptr, len, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { (void)cudaGetLastError(); return GF_OK; }
    if (e != cudaSuccess) { (void)cudaGetLastError(); return GF_ERR_CUDA; }
    return GF_OK;
}
GF_API int gf_cuda_host_unregister(void* ptr) {
    if (!ptr) return GF_ERR_BAD_PARAMS;
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return GF_ERR_CUDA; }
    return GF_OK;
}

GF_API int gf_cuda_checksum_dev(const void* ptr_dev, size_t len, uint64_t* out_dev, void* cu_stream) {
    if (!ptr_dev || !out_dev) return GF_ERR_BAD_PARAMS;
    cudaStream_t st = (cudaStream_t)cu_stream;
    if (cudaMemsetAsync(out_dev, 0, sizeof(uint64_t), st) != cudaSuccess) { (void)cudaGetLastError(); return GF_ERR_CUDA; }
    const size_t n = len / 4;
    if (n) checksum_kernel<<<148 * 4, 256, 0, st>>>(reinterpret_cast<const uint32_t*>(ptr_dev), n, reinterpret_cast<unsigned long long*>(out_dev));
    if (cudaGetLastError() != cudaSuccess) return GF_ERR_CUDA;
    return GF_OK;
}

GF_API int gf_cuda_queue_create(gf_cuda_queue** out, const gf_queue_config* cfg, const gf_compute_params* cp,
                                const gf_buffer_desc* in_proto, const gf_buffer_desc* out_proto) {
    if (!out || !cfg || !cp || !in_proto || !out_proto) return GF_ERR_BAD_PARAMS;
    *out = nullptr;
    if (cfg->depth < 1 || cfg->depth > 16) return GF_ERR_BAD_PARAMS;
    gf_cuda_queue* q = new gf_cuda_queue();
    q->cfg = *cfg; q->cp = *cp;
    auto bail = [&](int rc) { gf_cuda_queue_destroy(q); return rc; };
    if (cudaSetDevice(cfg->device) != cudaSuccess) { (void)cudaGetLastError(); return bail(GF_ERR_CUDA); }
    if (cfg->pin_numa) (void)gf_cuda_bind_thread_to_device(cfg->device);      // before any page-locked staging is allocated
    int rc = gf_cuda_gyro_upload(&q->gyro, cfg->device, cp);
    if (rc != GF_OK) return bail(rc);
    // a template KernelParams good enough for gf_cuda_create's validation (sizes, strides, interpolation, pixel size)
    gf_kernel_params kp; memset(&kp, 0, sizeof(kp));
    kp.matrix_count = 1;
    rc = gf_get_frame_transform_at(&cfg->stab, cp, in_proto, out_proto, nullptr, 0, 0.0, 0, 1.0, &kp);
    if (rc != GF_OK) return bail(rc);
    q->max_rows = (size_t)(cp->width > cp->height ? cp->width : cp->height);
    q->slots.resize((size_t)cfg->depth);
    for (QSlot& s : q->slots) {
        rc = gf_cuda_create(&s.ctx, cfg->device, &kp, cfg->stab.pixel_type, cfg->distortion_model, cfg->digital_lens, in_proto, out_proto, 0);
        if (rc != GF_OK) { q->last_error = gf_cuda_last_error(nullptr); return bail(rc); }
        rc = alloc_slot(q, s);
        if (rc != GF_OK) return bail(rc);
    }
    *out = q;
    return GF_OK;
}

GF_API int gf_cuda_queue_submit(gf_cuda_queue* q, size_t frame, double timestamp_ms, const gf_buffer_desc* in, const gf_buffer_desc* out,
                                const float* mesh, size_t mesh_len) {
    if (!q || !in || !out) return qfail(q, GF_ERR_BAD_PARAMS, "null argument");
    if (!q->planes.empty()) return qfail(q, GF_ERR_BAD_PARAMS, "a frame queue takes gf_cuda_queue_submit_frame");
    if (mesh_len > GF_MESH_MAX_LEN) return qfail(q, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch buf_mesh_data");
    QCK(cudaSetDevice(q->cfg.device));
    QSlot& s = q->slots[(size_t)q->next];
    if (s.busy) return qfail(q, GF_ERR_BAD_PARAMS, "queue full: gf_cuda_queue_wait for the oldest frame first");
    nvtxRangePushA("gf_queue_submit");
    // FrameTransform::at_timestamp on the device: rows x 14 table + its trust verdict, then the per-buffer half of KernelParams
    gf_kernel_params kp; size_t rows = 0; double fov = 1.0, minimal_fov = 1.0;
    int rc = gf_cuda_frame_transform_dev_flagged(q->gyro, &q->cp, timestamp_ms, frame, &kp, s.d_mat, q->max_rows, s.d_flags,
                                                 &rows, &fov, &minimal_fov, (void*)s.stream);
    if (rc != GF_OK) { nvtxRangePop(); return qfail(q, rc, "gf_cuda_frame_transform_dev_flagged failed"); }
    q->launches++;
    rc = gf_get_frame_transform_at(&q->cfg.stab, &q->cp, in, out, mesh, mesh_len, timestamp_ms, frame, minimal_fov, &kp);
    if (rc != GF_OK) { nvtxRangePop(); return qfail(q, rc, "gf_get_frame_transform_at failed"); }
    const float* mesh_dev = nullptr;
    if (mesh && mesh_len) {
        memcpy(s.h_mesh, mesh, mesh_len * sizeof(float));
        cudaError_t e = cudaMemcpyAsync(s.d_mesh, s.h_mesh, mesh_len * sizeof(float), cudaMemcpyHostToDevice, s.stream);
        if (e != cudaSuccess) { nvtxRangePop(); return qcuda(q, e, "mesh upload"); }
        mesh_dev = s.d_mesh;
    }
    const unsigned long long l0 = gf_cuda_launch_count(s.ctx);
    rc = gf_internal_run_frame(s.ctx, in, out, &kp, s.d_mat, rows, mesh_dev, mesh_dev ? mesh_len : 0, s.d_flags, (void*)s.stream,
                               q->cfg.checksum ? s.d_sum : nullptr);
    if (rc != GF_OK) { q->last_error = gf_cuda_last_error(s.ctx); nvtxRangePop(); return rc; }
    q->launches += gf_cuda_launch_count(s.ctx) - l0 + (q->cfg.checksum ? 1 : 0);
    if (q->cfg.checksum) {
        cudaError_t e = cudaMemcpyAsync(s.h_sum, s.d_sum, sizeof(uint64_t), cudaMemcpyDeviceToHost, s.stream);
        if (e != cudaSuccess) { nvtxRangePop(); return qcuda(q, e, "checksum download"); }
    }
    cudaError_t e = cudaEventRecord(s.done, s.stream);
    nvtxRangePop();
    if (e != cudaSuccess) return qcuda(q, e, "cudaEventRecord");
    s.busy = true; s.frame = frame;
    q->fifo.push_back(q->next);
    q->next = (q->next + 1) % (int)q->slots.size();
    return GF_OK;
}

GF_API int gf_cuda_queue_wait(gf_cuda_queue* q, size_t* out_frame, uint64_t* out_checksum) {
    if (!q) return GF_ERR_BAD_PARAMS;
    if (q->fifo.empty()) return qfail(q, GF_ERR_NO_DATA, "nothing in flight");
    QSlot& s = q->slots[(size_t)q->fifo.front()];
    q->fifo.pop_front();
    int rc = finish_slot(q, s);
    if (rc != GF_OK) return rc;
    if (out_frame) *out_frame = s.frame;
    if (out_checksum) *out_checksum = *s.h_sum;
    return GF_OK;
}

// ---- frame mode: every plane of a decoder frame in one submission --------------------------------------------------------------

// The plane's KernelParams exactly as the reference's per-plane closure hands it to process_pixels (rendering/mod.rs:531-541):
// get_frame_transform_at with the plane's buffers, then the format's value limit, plane_index and the per-frame fill flag.
// `kp` holds the at_timestamp half on entry.
static int plane_params(const gf_cuda_queue* q, size_t i, const gf_buffer_desc* in, const gf_buffer_desc* out, const float* mesh, size_t mesh_len,
                        double timestamp_ms, size_t frame, double minimal_fov, int fill_with_background, gf_kernel_params* kp) {
    const int rc = gf_get_frame_transform_at(&q->plane_stab[i], &q->cp, in, out, mesh, mesh_len, timestamp_ms, frame, minimal_fov, kp);
    if (rc != GF_OK) return rc;
    kp->pixel_value_limit = q->planes[i].max_value;                                  // :532-533
    kp->max_pixel_value = q->planes[i].max_value;
    kp->plane_index = (int32_t)i;                                                     // :538
    if (fill_with_background) kp->flags |= GF_FLAG_FILL_WITH_BACKGROUND;              // :539-541
    return GF_OK;
}

GF_API int gf_cuda_queue_create_frame(gf_cuda_queue** out, const gf_queue_config* cfg, const gf_compute_params* cp, int format,
                                      int is_limited_range, size_t n_planes, const gf_buffer_desc* in_protos, const gf_buffer_desc* out_protos) {
    if (!out || !cfg || !cp || !in_protos || !out_protos) return GF_ERR_BAD_PARAMS;
    *out = nullptr;
    if (cfg->depth < 1 || cfg->depth > 16) return GF_ERR_BAD_PARAMS;
    gf_plane_spec in_spec[GF_FRAME_MAX_PLANES], out_spec[GF_FRAME_MAX_PLANES];
    size_t n_in = 0, n_out = 0;
    int rc = gf_frame_layout(format, cfg->stab.width, cfg->stab.height, in_spec, &n_in);
    if (rc != GF_OK) return rc;
    rc = gf_frame_layout(format, cfg->stab.output_width, cfg->stab.output_height, out_spec, &n_out);
    if (rc != GF_OK) return rc;
    if (n_planes != n_in) return GF_ERR_BAD_PARAMS;
    for (size_t i = 0; i < n_planes; ++i)
        if (in_protos[i].width != in_spec[i].width || in_protos[i].height != in_spec[i].height ||
            out_protos[i].width != out_spec[i].width || out_protos[i].height != out_spec[i].height) return GF_ERR_SIZE_MISMATCH;
    gf_cuda_queue* q = new gf_cuda_queue();
    q->cfg = *cfg; q->cp = *cp;
    auto bail = [&](int code) { gf_cuda_queue_destroy(q); return code; };
    if (cudaSetDevice(cfg->device) != cudaSuccess) { (void)cudaGetLastError(); return bail(GF_ERR_CUDA); }
    if (cfg->pin_numa) (void)gf_cuda_bind_thread_to_device(cfg->device);
    rc = gf_cuda_gyro_upload(&q->gyro, cfg->device, cp);
    if (rc != GF_OK) return bail(rc);
    q->planes.assign(in_spec, in_spec + n_planes);
    q->out_planes.assign(out_spec, out_spec + n_planes);
    // per distinct pixel type: the first plane of that type is the context's validation template
    std::vector<int> ctx_pix; std::vector<gf_kernel_params> ctx_kp; std::vector<size_t> ctx_plane;
    for (size_t i = 0; i < n_planes; ++i) {
        gf_stab_config st = cfg->stab;                                                // :504-507, :514
        st.pixel_type = in_spec[i].pixel_type;
        rc = gf_background_for_plane(st.pixel_type, cfg->stab.background, in_spec[i].ind, (size_t)in_spec[i].n_ind, is_limited_range, st.background);
        if (rc != GF_OK) return bail(rc);
        q->plane_stab.push_back(st);
        q->plane_kind_in.push_back(in_protos[i].kind); q->plane_kind_out.push_back(out_protos[i].kind);
        q->plane_len_in.push_back(in_protos[i].len);   q->plane_len_out.push_back(out_protos[i].len);
        size_t c = 0;
        while (c < ctx_pix.size() && ctx_pix[c] != st.pixel_type) ++c;
        if (c == ctx_pix.size()) {
            gf_kernel_params kp; memset(&kp, 0, sizeof(kp));
            kp.matrix_count = 1;
            rc = plane_params(q, i, &in_protos[i], &out_protos[i], nullptr, 0, 0.0, 0, 1.0, 0, &kp);
            if (rc != GF_OK) return bail(rc);
            ctx_pix.push_back(st.pixel_type); ctx_kp.push_back(kp); ctx_plane.push_back(i);
        }
        q->plane_ctx.push_back((int)c);
    }
    q->max_rows = (size_t)(cp->width > cp->height ? cp->width : cp->height);
    q->slots.resize((size_t)cfg->depth);
    for (QSlot& s : q->slots) {
        for (size_t c = 0; c < ctx_pix.size(); ++c) {
            // the contexts only ever see DEVICE buffers (the slot stages HOST planes itself), so they allocate no staging of their own
            gf_buffer_desc i = in_protos[ctx_plane[c]], o = out_protos[ctx_plane[c]];
            i.kind = GF_BUF_DEVICE; o.kind = GF_BUF_DEVICE;
            gf_cuda_ctx* ctx = nullptr;
            rc = gf_cuda_create(&ctx, cfg->device, &ctx_kp[c], ctx_pix[c], cfg->distortion_model, cfg->digital_lens, &i, &o, 0);
            if (rc != GF_OK) { q->last_error = gf_cuda_last_error(nullptr); return bail(rc); }
            s.pix_ctx.push_back(ctx);
        }
        s.d_in.assign(n_planes, nullptr); s.d_out.assign(n_planes, nullptr);
        for (size_t i = 0; i < n_planes; ++i) {
            cudaError_t e = cudaSuccess;
            if (in_protos[i].kind == GF_BUF_HOST) e = cudaMalloc(&s.d_in[i], in_protos[i].len);
            if (e == cudaSuccess && out_protos[i].kind == GF_BUF_HOST) e = cudaMalloc(&s.d_out[i], out_protos[i].len);
            if (e == cudaSuccess && s.d_out[i]) e = cudaMemset(s.d_out[i], 0, out_protos[i].len);   // row padding the warp never writes: defined checksums
            if (e != cudaSuccess) { qcuda(q, e, "plane staging allocation"); return bail(GF_ERR_CUDA); }
        }
        rc = alloc_slot(q, s);
        if (rc != GF_OK) return bail(rc);
    }
    *out = q;
    return GF_OK;
}

GF_API int gf_cuda_queue_submit_frame(gf_cuda_queue* q, size_t frame, double timestamp_ms, size_t n_planes, const gf_buffer_desc* in,
                                      const gf_buffer_desc* out, const float* mesh, size_t mesh_len, int fill_with_background) {
    if (!q || !in || !out) return qfail(q, GF_ERR_BAD_PARAMS, "null argument");
    if (q->planes.empty()) return qfail(q, GF_ERR_BAD_PARAMS, "a single-buffer queue takes gf_cuda_queue_submit");
    if (n_planes != q->planes.size()) return qfail(q, GF_ERR_BAD_PARAMS, "plane count differs from the format's layout");
    if (mesh_len > GF_MESH_MAX_LEN) return qfail(q, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch buf_mesh_data");
    for (size_t i = 0; i < n_planes; ++i) {
        if (in[i].width != q->planes[i].width || in[i].height != q->planes[i].height ||
            out[i].width != q->out_planes[i].width || out[i].height != q->out_planes[i].height)
            return qfail(q, GF_ERR_SIZE_MISMATCH, "SizeMismatch: plane " + std::to_string(i) + " differs from the format's layout");
        if (in[i].kind != q->plane_kind_in[i] || out[i].kind != q->plane_kind_out[i])
            return qfail(q, GF_ERR_BAD_PARAMS, "plane " + std::to_string(i) + ": buffer kind differs from the prototype's");
        if ((in[i].kind == GF_BUF_HOST && in[i].len > q->plane_len_in[i]) || (out[i].kind == GF_BUF_HOST && out[i].len > q->plane_len_out[i]))
            return qfail(q, GF_ERR_BUFFER_TOO_SMALL, "Buffer size mismatch: plane " + std::to_string(i) + " exceeds its prototype's staging");
    }
    QCK(cudaSetDevice(q->cfg.device));
    QSlot& s = q->slots[(size_t)q->next];
    if (s.busy) return qfail(q, GF_ERR_BAD_PARAMS, "queue full: gf_cuda_queue_wait_frame for the oldest frame first");
    nvtxRangePushA("gf_queue_submit_frame");
    struct NvtxPop { ~NvtxPop() { nvtxRangePop(); } } nvtx_pop_;
    // one at_timestamp for every plane: the planes differ only in their background, which at_timestamp does not read
    gf_kernel_params kp0; size_t rows = 0; double fov = 1.0, minimal_fov = 1.0;
    int rc = gf_cuda_frame_transform_dev_flagged(q->gyro, &q->cp, timestamp_ms, frame, &kp0, s.d_mat, q->max_rows, s.d_flags,
                                                 &rows, &fov, &minimal_fov, (void*)s.stream);
    if (rc != GF_OK) return qfail(q, rc, "gf_cuda_frame_transform_dev_flagged failed");
    q->launches++;
    gf_kernel_params kp[GF_FRAME_MAX_PLANES];
    gf_buffer_desc din[GF_FRAME_MAX_PLANES], dout[GF_FRAME_MAX_PLANES];
    for (size_t i = 0; i < n_planes; ++i) {
        kp[i] = kp0;
        rc = plane_params(q, i, &in[i], &out[i], mesh, mesh_len, timestamp_ms, frame, minimal_fov, fill_with_background, &kp[i]);
        if (rc != GF_OK) return qfail(q, rc, "gf_get_frame_transform_at failed for plane " + std::to_string(i));
    }
    const float* mesh_dev = nullptr;
    if (mesh && mesh_len) {
        memcpy(s.h_mesh, mesh, mesh_len * sizeof(float));
        QCK(cudaMemcpyAsync(s.d_mesh, s.h_mesh, mesh_len * sizeof(float), cudaMemcpyHostToDevice, s.stream));
        mesh_dev = s.d_mesh;
    }
    bool full_cover[GF_FRAME_MAX_PLANES] = {false, false, false, false};
    for (size_t i = 0; i < n_planes; ++i) {
        din[i] = in[i]; dout[i] = out[i];
        if (in[i].kind == GF_BUF_HOST) {
            QCK(cudaMemcpyAsync(s.d_in[i], in[i].ptr, in[i].len, cudaMemcpyHostToDevice, s.stream));
            din[i].kind = GF_BUF_DEVICE; din[i].ptr = s.d_in[i];
        }
        if (out[i].kind == GF_BUF_HOST) {
            // Pixels the warp does not write keep the buffer's previous content, like on the CPU path.  When the output rect is the whole
            // plane every pixel of its width x height is written (the rect maps onto [0, output size)), so only those bytes travel back;
            // otherwise the plane is uploaded first and returned whole.
            const gf_kernel_params& k = kp[i];
            full_cover[i] = k.output_rect[0] == 0 && k.output_rect[1] == 0 && k.output_rect[2] == out[i].width && k.output_rect[3] == out[i].height &&
                            (k.flags & GF_FLAG_FILL_WITH_BACKGROUND) == 0 &&
                            (size_t)out[i].height * (size_t)k.output_stride <= out[i].len + (size_t)(k.output_stride - out[i].width * k.bytes_per_pixel);
            if (!full_cover[i]) QCK(cudaMemcpyAsync(s.d_out[i], out[i].ptr, out[i].len, cudaMemcpyHostToDevice, s.stream));
            dout[i].kind = GF_BUF_DEVICE; dout[i].ptr = s.d_out[i];
        }
    }
    // warp: planes of one pixel type and equal geometry go through one call of the planes path (one coordinate pass)
    bool done[GF_FRAME_MAX_PLANES] = {false, false, false, false};
    for (size_t i = 0; i < n_planes; ++i) {
        if (done[i]) continue;
        gf_buffer_desc gin[GF_FRAME_MAX_PLANES], gout[GF_FRAME_MAX_PLANES]; gf_kernel_params gkp[GF_FRAME_MAX_PLANES];
        size_t ng = 0;
        for (size_t j = i; j < n_planes; ++j) {
            if (done[j] || q->plane_ctx[j] != q->plane_ctx[i]) continue;
            if (j != i && !gf_internal_same_plane_geometry(&kp[i], &din[i], &dout[i], &kp[j], &din[j], &dout[j])) continue;
            gin[ng] = din[j]; gout[ng] = dout[j]; gkp[ng] = kp[j]; ++ng; done[j] = true;
        }
        gf_cuda_ctx* ctx = s.pix_ctx[(size_t)q->plane_ctx[i]];
        const unsigned long long l0 = gf_cuda_launch_count(ctx);
        rc = gf_cuda_undistort_planes_dev_flagged(ctx, ng, gin, gout, gkp, s.d_mat, rows, mesh_dev, mesh_dev ? mesh_len : 0, s.d_flags, (void*)s.stream);
        if (rc != GF_OK) { q->last_error = gf_cuda_last_error(ctx); return rc; }
        q->launches += gf_cuda_launch_count(ctx) - l0;
    }
    if (q->cfg.checksum) {
        PlaneWords pw; memset(&pw, 0, sizeof(pw));
        for (size_t i = 0; i < n_planes; ++i) {
            pw.w[i] = reinterpret_cast<const uint32_t*>(dout[i].ptr);
            pw.n[i] = std::min<size_t>(out[i].len, (size_t)out[i].height * (size_t)kp[i].output_stride) / 4;
        }
        QCK(cudaMemsetAsync(s.d_sum, 0, n_planes * sizeof(uint64_t), s.stream));
        checksum_planes_kernel<<<dim3(148 * 2, (unsigned)n_planes), 256, 0, s.stream>>>(pw, reinterpret_cast<unsigned long long*>(s.d_sum));
        QCK(cudaGetLastError());
        q->launches++;
        QCK(cudaMemcpyAsync(s.h_sum, s.d_sum, n_planes * sizeof(uint64_t), cudaMemcpyDeviceToHost, s.stream));
    }
    for (size_t i = 0; i < n_planes; ++i) {
        if (out[i].kind != GF_BUF_HOST) continue;
        if (full_cover[i]) QCK(cudaMemcpy2DAsync(out[i].ptr, (size_t)kp[i].output_stride, s.d_out[i], (size_t)kp[i].output_stride,
                                                 (size_t)out[i].width * (size_t)kp[i].bytes_per_pixel, (size_t)out[i].height, cudaMemcpyDeviceToHost, s.stream));
        else               QCK(cudaMemcpyAsync(out[i].ptr, s.d_out[i], out[i].len, cudaMemcpyDeviceToHost, s.stream));
    }
    QCK(cudaEventRecord(s.done, s.stream));
    s.busy = true; s.frame = frame;
    q->fifo.push_back(q->next);
    q->next = (q->next + 1) % (int)q->slots.size();
    return GF_OK;
}

GF_API int gf_cuda_queue_wait_frame(gf_cuda_queue* q, size_t* out_frame, uint64_t* out_checksums, size_t n_checksums) {
    if (!q) return GF_ERR_BAD_PARAMS;
    if (q->fifo.empty()) return qfail(q, GF_ERR_NO_DATA, "nothing in flight");
    QSlot& s = q->slots[(size_t)q->fifo.front()];
    q->fifo.pop_front();
    int rc = finish_slot(q, s);
    if (rc != GF_OK) return rc;
    if (out_frame) *out_frame = s.frame;
    const size_t n = std::min<size_t>(n_checksums, q->planes.empty() ? 1 : q->planes.size());
    for (size_t i = 0; out_checksums && i < n; ++i) out_checksums[i] = q->cfg.checksum ? s.h_sum[i] : 0;
    return GF_OK;
}

GF_API int gf_cuda_queue_drain(gf_cuda_queue* q) {
    if (!q) return GF_ERR_BAD_PARAMS;
    while (!q->fifo.empty()) { int rc = gf_cuda_queue_wait(q, nullptr, nullptr); if (rc != GF_OK) return rc; }
    return GF_OK;
}

GF_API uint64_t gf_cuda_queue_launches(gf_cuda_queue* q) { return q ? q->launches : 0; }
GF_API const char* gf_cuda_queue_last_error(gf_cuda_queue* q) { return q ? q->last_error.c_str() : ""; }

GF_API void gf_cuda_queue_destroy(gf_cuda_queue* q) {
    if (!q) return;
    cudaSetDevice(q->cfg.device);
    for (QSlot& s : q->slots) {
        if (s.stream) cudaStreamSynchronize(s.stream);
        if (s.ctx) gf_cuda_destroy(s.ctx);
        if (s.d_mat) cudaFree(s.d_mat);
        if (s.d_flags) cudaFree(s.d_flags);
        if (s.h_mesh) cudaFreeHost(s.h_mesh);
        if (s.d_mesh) cudaFree(s.d_mesh);
        if (s.d_sum) cudaFree(s.d_sum);
        if (s.h_sum) cudaFreeHost(s.h_sum);
        for (gf_cuda_ctx* c : s.pix_ctx) if (c) gf_cuda_destroy(c);
        for (uint8_t* b : s.d_in) if (b) cudaFree(b);
        for (uint8_t* b : s.d_out) if (b) cudaFree(b);
        if (s.done) cudaEventDestroy(s.done);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    if (q->gyro) gf_cuda_gyro_free(q->gyro);
    (void)cudaGetLastError();
    delete q;
}

} // extern "C"
