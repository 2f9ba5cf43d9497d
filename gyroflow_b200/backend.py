"""Host-side mirror of the reference's backend-wrapper convention, over the C ABI.

Names follow the reference so the parity tests read like its call sites:

  BufferDescription / Buffers      src/core/gpu/mod.rs:17-29
  FrameTransform                   src/core/stabilization/frame_transform.rs:11-19
  CudaWrapper.new / undistort_image   <- OclWrapper::new / undistort_image  src/core/gpu/opencl.rs:178,330
  GyroflowCoreError                src/core/lib.rs:2098-2141

This module only marshals arguments; all pixel work happens in libgyroflow_cuda.so.
"""
import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Tuple

import numpy as np

from . import abi


class GyroflowCoreError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("%s: %s" % (abi.ERRORS.get(code, str(code)), message))
        self.code = code
        self.kind = abi.ERRORS.get(code, "Unknown")


@dataclass
class BufferDescription:
    """size = (width, height, stride_bytes); data is a C-contiguous uint8 numpy array (BufferSource::Cpu) or an
    integer device pointer with `length` bytes (BufferSource::CUDABuffer)."""
    size: Tuple[int, int, int]
    data: object = None
    rect: Optional[Tuple[int, int, int, int]] = None
    rotation: Optional[float] = None
    length: Optional[int] = None          # bytes, required for device pointers

    def to_c(self):
        d = abi.BufferDesc()
        d.width, d.height, d.stride = self.size
        if self.rect is not None:
            d.has_rect = 1
            d.rect[:] = list(self.rect)
        if self.rotation is not None:
            d.has_rotation = 1
            d.rotation = self.rotation
        if isinstance(self.data, np.ndarray):
            assert self.data.dtype == np.uint8 and self.data.flags["C_CONTIGUOUS"]
            d.kind = abi.BUF_HOST
            d.ptr = self.data.ctypes.data
            d.len = self.data.nbytes
        elif isinstance(self.data, int):
            d.kind = abi.BUF_DEVICE
            d.ptr = self.data
            d.len = int(self.length)
        else:
            d.kind = abi.BUF_NONE
        return d

    def get_rect(self):
        """Stabilization::get_rect — stabilization/mod.rs:209-224 (stretch to the buffer by default)."""
        if self.rect is not None:
            return [int(v) for v in self.rect]
        return [0, 0, int(self.size[0]), int(self.size[1])]


@dataclass
class Buffers:
    input: BufferDescription
    output: BufferDescription


@dataclass
class FrameTransform:
    matrices: np.ndarray                      # (rows, 14) float32
    kernel_params: abi.KernelParams
    fov: float = 1.0
    minimal_fov: float = 1.0
    focal_length: Optional[float] = None
    mesh_data: np.ndarray = field(default_factory=lambda: np.zeros(0, np.float32))


@dataclass
class ProcessedInfo:
    fov: float
    minimal_fov: float
    focal_length: Optional[float]
    backend: str


def list_devices():
    """`"[CUDA] <name>"` entries, like the `[OpenCL]`/`[wgpu]` lists of stabilization/mod.rs:399-410."""
    lib = abi.load_library()
    out = []
    for i in range(lib.gf_cuda_device_count()):
        buf = C.create_string_buffer(256)
        if lib.gf_cuda_device_name(i, buf, 256) == 0:
            out.append(buf.value.decode())
    return out


class CudaWrapper:
    """One pre-compiled kernel instantiation + its device staging; not thread-safe (one per host thread/stream)."""

    def __init__(self, handle, lib, pixel_type):
        self._h = handle
        self._lib = lib
        self.pixel_type = pixel_type

    @classmethod
    def new(cls, params: abi.KernelParams, pixel_type: str, distortion_model: str, digital_lens: Optional[str],
            buffers: Buffers, drawing_len: int = 0, device: int = 0):
        lib = abi.load_library()
        h = C.c_void_p()
        i, o = buffers.input.to_c(), buffers.output.to_c()
        rc = lib.gf_cuda_create(C.byref(h), device, C.byref(params), abi.PIXEL_TYPES[pixel_type][0],
                                abi.LENS[distortion_model], abi.LENS[digital_lens] if digital_lens else 0,
                                C.byref(i), C.byref(o), drawing_len)
        if rc != 0:
            raise GyroflowCoreError(rc, (lib.gf_cuda_last_error(None) or b"").decode())
        return cls(h, lib, pixel_type)

    def _err(self, rc):
        return GyroflowCoreError(rc, (self._lib.gf_cuda_last_error(self._h) or b"").decode())

    def set_overlays(self, enabled: bool):
        """Preview overlays (draw_pixel / draw_safe_area of the reference's GPU kernels); off by default like the CPU path."""
        rc = self._lib.gf_cuda_set_overlays(self._h, int(enabled))
        if rc != 0:
            raise self._err(rc)

    def undistort_image(self, buffers: Buffers, itm: FrameTransform, drawing_buffer=None, stream: int = 0):
        i, o = buffers.input.to_c(), buffers.output.to_c()
        m = np.ascontiguousarray(itm.matrices, dtype=np.float32)
        mesh = np.ascontiguousarray(itm.mesh_data, dtype=np.float32)
        d = None if drawing_buffer is None else np.ascontiguousarray(drawing_buffer, dtype=np.uint8)
        rc = self._lib.gf_cuda_undistort_image(
            self._h, C.byref(i), C.byref(o), C.byref(itm.kernel_params),
            m.ctypes.data, m.shape[0], mesh.ctypes.data if mesh.size else None, mesh.size,
            d.ctypes.data if d is not None and d.size else None, d.size if d is not None else 0, stream or None)
        if rc != 0:
            raise self._err(rc)

    def undistort_image_async(self, buffers: Buffers, itm: FrameTransform, stream: int = 0):
        """Enqueue only (HOST buffers must be pinned and outlive the call); pair with synchronize()."""
        i, o = buffers.input.to_c(), buffers.output.to_c()
        m = np.ascontiguousarray(itm.matrices, dtype=np.float32)
        mesh = np.ascontiguousarray(itm.mesh_data, dtype=np.float32)
        rc = self._lib.gf_cuda_undistort_image_async(
            self._h, C.byref(i), C.byref(o), C.byref(itm.kernel_params),
            m.ctypes.data, m.shape[0], mesh.ctypes.data if mesh.size else None, mesh.size, stream or None)
        if rc != 0:
            raise self._err(rc)

    def undistort_image_dev(self, buffers: Buffers, params: abi.KernelParams, matrices_dev: int, matrix_rows: int,
                            mesh_dev: int = 0, mesh_len: int = 0, stream: int = 0, table_flags_dev: int = 0):
        """Device-resident tables.  table_flags_dev: device address of the table's trust verdict word (written by scan_tables_dev or by
        DeviceGyro.frame_transform); 0 = none, the guarded code path runs."""
        i, o = buffers.input.to_c(), buffers.output.to_c()
        if table_flags_dev:
            rc = self._lib.gf_cuda_undistort_image_dev_flagged(self._h, C.byref(i), C.byref(o), C.byref(params), matrices_dev, matrix_rows,
                                                               mesh_dev or None, mesh_len, table_flags_dev, stream or None)
        else:
            rc = self._lib.gf_cuda_undistort_image_dev(self._h, C.byref(i), C.byref(o), C.byref(params),
                                                       matrices_dev, matrix_rows, mesh_dev or None, mesh_len, stream or None)
        if rc != 0:
            raise self._err(rc)

    def undistort_planes_dev(self, buffers, params, matrices_dev: int, matrix_rows: int, mesh_dev: int = 0, mesh_len: int = 0, stream: int = 0,
                             table_flags_dev: int = 0):
        """buffers: list of Buffers (DEVICE), params: list of KernelParams — the planes of one frame (gf_cuda_undistort_planes_dev)."""
        n = len(buffers)
        ins = (abi.BufferDesc * n)(*[b.input.to_c() for b in buffers])
        outs = (abi.BufferDesc * n)(*[b.output.to_c() for b in buffers])
        ps = (abi.KernelParams * n)(*params)
        rc = self._lib.gf_cuda_undistort_planes_dev_flagged(self._h, n, ins, outs, ps, matrices_dev, matrix_rows, mesh_dev or None, mesh_len,
                                                            table_flags_dev or None, stream or None)
        if rc != 0:
            raise self._err(rc)

    def undistort_planes(self, buffers, params, itm: FrameTransform, stream: int = 0):
        """The planes of one frame in HOST memory (gf_cuda_undistort_planes): buffers = list of Buffers with numpy data, params = list of
        KernelParams; tables from `itm` (host).  Synchronous."""
        n = len(buffers)
        ins = (abi.BufferDesc * n)(*[b.input.to_c() for b in buffers])
        outs = (abi.BufferDesc * n)(*[b.output.to_c() for b in buffers])
        ps = (abi.KernelParams * n)(*params)
        m = np.ascontiguousarray(itm.matrices, dtype=np.float32)
        mesh = np.ascontiguousarray(itm.mesh_data, dtype=np.float32)
        rc = self._lib.gf_cuda_undistort_planes(self._h, n, ins, outs, ps, m.ctypes.data, m.shape[0], mesh.ctypes.data if mesh.size else None, mesh.size, stream or None)
        if rc != 0:
            raise self._err(rc)

    def validate_tables_dev(self, matrices_dev: int, matrix_rows: int):
        """Synchronous query of a device table's verdict: 0 tame and IBIS-free, bit 0 wild entry, bit 1 IBIS rows.  Nothing is cached."""
        rc = self._lib.gf_cuda_validate_tables_dev(self._h, matrices_dev, matrix_rows)
        if rc < 0:
            raise self._err(rc)
        return rc

    def synchronize(self):
        rc = self._lib.gf_cuda_synchronize(self._h)
        if rc != 0:
            raise self._err(rc)

    @property
    def launch_count(self):
        return int(self._lib.gf_cuda_launch_count(self._h))

    def filter_counts(self):
        """Counters of the latest frame on the filtered rolling-shutter pre-pass (waits for the work queued so far): pairs and pixels
        sent to the tail launch, whether a queue was full, and how many of the pairs the final pass deferred (gf_cuda_filter_counts)."""
        out = (C.c_uint32 * 4)()
        rc = self._lib.gf_cuda_filter_counts(self._h, out)
        if rc != 0:
            raise self._err(rc)
        return dict(pairs=int(out[0]), pixels=int(out[1]), overflow=bool(out[2]), bad_pairs=int(out[3]))

    def close(self):
        if self._h:
            self._lib.gf_cuda_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ------------------------------------------------------------------------------------------ per-frame transform producer


class ComputeParams:
    """Owns a gf_compute_params plus the numpy arrays it points to (quaternion tracks, fovs)."""

    def __init__(self, kernel_params: abi.KernelParams, org, smoothed, frame_readout_time_ms=16.0, fovs=None, video_rotation=0.0,
                 horizontal=False, inverted=False, framebuffer_inverted=False, fov_scale=1.0, sync_offsets=None,
                 per_frame_time_offsets=None, focal_lengths=None, smoothed_focal_lengths=None, readout_time_scale=0.0, camera_stab=None,
                 gyro_offset_ms=0.0, keyframes=None, keyframe_timestamp_scale=0.0, lens_per_frame=None, distorting_meshes=None):
        """sync_offsets: {timestamp_us: offset_ms} (GyroSource::offsets_adjusted); camera_stab: list (one per frame) of dicts with
        offset, sensor_size, crop_area, pixel_pitch, ibis=(pos[n], xyz[n,3]), ois=(pos[n], xyz[n,3]) (CameraStabData);
        keyframes: {KeyframeType name: [(timestamp_us, value, easing name), ...]} for the types at_timestamp reads (abi.KEYFRAME_TYPES)."""
        p = kernel_params
        c = abi.ComputeParams()
        c.width, c.height, c.output_width, c.output_height = p.width, p.height, p.output_width, p.output_height
        c.camera_matrix[:] = [float(p.f[0]), 0.0, float(p.c[0]), 0.0, float(p.f[1]), float(p.c[1]), 0.0, 0.0, 1.0]
        c.distortion_coeffs[:] = [float(v) for v in p.k]
        c.radial_distortion_limit = float(p.r_limit)
        c.input_horizontal_stretch = float(p.input_horizontal_stretch)
        c.input_vertical_stretch = float(p.input_vertical_stretch)
        c.fov_scale = fov_scale
        self._fovs = np.ascontiguousarray(fovs if fovs is not None else [], dtype=np.float64)
        if self._fovs.size:
            c.fovs = self._fovs.ctypes.data_as(C.POINTER(C.c_double)); c.n_fovs = self._fovs.size
        c.frame_readout_time = frame_readout_time_ms
        c.readout_horizontal, c.readout_inverted = int(horizontal), int(inverted)
        c.framebuffer_inverted = int(framebuffer_inverted)
        c.video_rotation = video_rotation
        c.lens_correction_amount = float(p.lens_correction_amount)
        c.light_refraction_coefficient = float(p.light_refraction_coefficient)
        c.background_mode = p.background_mode
        c.digital_lens_params[:] = [float(v) for v in p.digital_lens_params]
        c.n_digital_lens_params = 16
        self._ots = np.ascontiguousarray(org.ts, dtype=np.int64); self._oq = np.ascontiguousarray(org.q, dtype=np.float64)
        self._sts = np.ascontiguousarray(smoothed.ts, dtype=np.int64); self._sq = np.ascontiguousarray(smoothed.q, dtype=np.float64)
        c.org = abi.QuatTrack(self._ots.ctypes.data_as(C.POINTER(C.c_int64)), self._oq.ctypes.data_as(C.POINTER(C.c_double)), len(self._ots))
        c.smoothed = abi.QuatTrack(self._sts.ctypes.data_as(C.POINTER(C.c_int64)), self._sq.ctypes.data_as(C.POINTER(C.c_double)), len(self._sts))
        c.duration_ms = float(self._ots[-1] - self._ots[0]) / 1000.0
        c.gyro_offset_ms = gyro_offset_ms
        if sync_offsets:
            ks = sorted(sync_offsets)
            self._so_ts = np.asarray(ks, dtype=np.int64); self._so_ms = np.asarray([sync_offsets[k] for k in ks], dtype=np.float64)
            c.sync_offset_ts_us = self._so_ts.ctypes.data_as(C.POINTER(C.c_int64)); c.sync_offset_ms = self._so_ms.ctypes.data_as(C.POINTER(C.c_double))
            c.n_sync_offsets = len(ks)
        if per_frame_time_offsets is not None:
            self._pfo = np.ascontiguousarray(per_frame_time_offsets, dtype=np.float64)
            c.per_frame_time_offsets = self._pfo.ctypes.data_as(C.POINTER(C.c_double)); c.n_per_frame_time_offsets = self._pfo.size
        if focal_lengths is not None and smoothed_focal_lengths is not None:
            self._fl = np.ascontiguousarray(focal_lengths, dtype=np.float64); self._sfl = np.ascontiguousarray(smoothed_focal_lengths, dtype=np.float64)
            assert self._fl.size == self._sfl.size
            c.focal_length_smoothing_enabled = 1
            c.focal_lengths = self._fl.ctypes.data_as(C.POINTER(C.c_double)); c.smoothed_focal_lengths = self._sfl.ctypes.data_as(C.POINTER(C.c_double))
            c.n_focal_lengths = self._fl.size
        c.readout_time_scale = readout_time_scale
        c.keyframe_timestamp_scale = keyframe_timestamp_scale
        if lens_per_frame:        # list of dicts: camera_matrix[9], distortion_coeffs[12], radial_distortion_limit, input_horizontal_stretch, input_vertical_stretch
            arr = (abi.LensData * len(lens_per_frame))()
            for i, d in enumerate(lens_per_frame):
                arr[i].camera_matrix[:] = [float(v) for v in d["camera_matrix"]]
                arr[i].distortion_coeffs[:] = [float(v) for v in d["distortion_coeffs"]]
                arr[i].radial_distortion_limit = float(d.get("radial_distortion_limit", 0.0))
                arr[i].input_horizontal_stretch = float(d.get("input_horizontal_stretch", 1.0)); arr[i].input_vertical_stretch = float(d.get("input_vertical_stretch", 1.0))
            self._lens = arr
            c.lens_per_frame = C.cast(arr, C.c_void_p); c.n_lens_per_frame = len(lens_per_frame)
        self._kf_arrays = []
        for name, keys in (keyframes or {}).items():
            keys = sorted(keys)
            ts = np.asarray([k[0] for k in keys], dtype=np.int64); val = np.asarray([k[1] for k in keys], dtype=np.float64)
            ea = np.asarray([abi.EASING[k[2]] if len(k) > 2 else abi.EASING["EaseInOut"] for k in keys], dtype=np.uint8)
            self._kf_arrays += [ts, val, ea]
            t = c.keyframes[abi.KEYFRAME_TYPES[name]]
            t.ts_us = ts.ctypes.data_as(C.POINTER(C.c_int64)); t.value = val.ctypes.data_as(C.POINTER(C.c_double))
            t.easing = ea.ctypes.data_as(C.POINTER(C.c_uint8)); t.n = len(keys)
        if distorting_meshes:     # one f64 mesh (or None) per frame: file_metadata.mesh_correction[frame].0
            arr = (abi.MeshF64 * len(distorting_meshes))()
            self._dmesh_arrays = []
            for i, mesh in enumerate(distorting_meshes):
                if mesh is None:
                    continue
                a = np.ascontiguousarray(mesh, dtype=np.float64); self._dmesh_arrays.append(a)
                arr[i].data = a.ctypes.data_as(C.POINTER(C.c_double)); arr[i].len = a.size
            self._dmesh = arr
            c.distorting_mesh = C.cast(arr, C.c_void_p); c.n_distorting_mesh = len(distorting_meshes)
        if camera_stab:
            self._stab_arrays = []
            arr = (abi.CameraStab * len(camera_stab))()
            dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
            for i, d in enumerate(camera_stab):
                cs = arr[i]
                cs.offset = float(d.get("offset", 0.0))
                cs.sensor_size[:] = [int(v) for v in d["sensor_size"]]
                cs.crop_area[:] = [float(v) for v in d["crop_area"]]
                cs.pixel_pitch[:] = [int(v) for v in d["pixel_pitch"]]
                for name in ("ibis", "ois"):
                    pos, xyz = d.get(name, (np.zeros(0), np.zeros((0, 3))))
                    pos = np.ascontiguousarray(pos, dtype=np.float64); xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
                    assert pos.size == xyz.shape[0]
                    self._stab_arrays += [pos, xyz]
                    setattr(cs, name + "_pos", dp(pos)); setattr(cs, name + "_xyz", dp(xyz)); setattr(cs, "n_" + name, pos.size)
            self._stab = arr
            c.camera_stab = C.cast(arr, C.c_void_p); c.n_camera_stab = len(camera_stab)
        self.c = c

    def at_timestamp(self, timestamp_ms, frame=0):
        """FrameTransform::at_timestamp on the host (f64): returns (KernelParams fields it sets, matrices[rows,14], fov, minimal_fov)."""
        lib = abi.load_library()
        rows_max = max(self.c.width, self.c.height)
        m = np.zeros((rows_max, 14), np.float32)
        kp = abi.KernelParams(); rows = C.c_size_t(); fov = C.c_double(); mfov = C.c_double()
        rc = lib.gf_frame_transform_at_timestamp(C.byref(self.c), timestamp_ms, frame, C.byref(kp), m.ctypes.data, rows_max,
                                                 C.byref(rows), C.byref(fov), C.byref(mfov))
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_frame_transform_at_timestamp")
        return kp, m[: rows.value].copy(), fov.value, mfov.value


class DeviceGyro:
    """Quaternion tracks resident in HBM + the per-frame matrix kernel (gf_cuda_frame_transform_dev)."""

    def __init__(self, cp: ComputeParams, device=0):
        self._lib = abi.load_library()
        self.cp = cp
        h = C.c_void_p()
        rc = self._lib.gf_cuda_gyro_upload(C.byref(h), device, C.byref(cp.c))
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_gyro_upload")
        self._h = h

    def frame_transform(self, timestamp_ms, matrices_dev: int, max_rows: int, frame=0, stream=0, table_flags_dev: int = 0):
        """FrameTransform::at_timestamp on the device.  table_flags_dev: device word that receives the table's trust verdict.
        stream = 0: the call waits for the kernel before returning; otherwise it only enqueues (give the warp the same stream)."""
        kp = abi.KernelParams(); rows = C.c_size_t(); fov = C.c_double(); mfov = C.c_double()
        rc = self._lib.gf_cuda_frame_transform_dev_flagged(self._h, C.byref(self.cp.c), timestamp_ms, frame, C.byref(kp), matrices_dev, max_rows,
                                                           table_flags_dev or None, C.byref(rows), C.byref(fov), C.byref(mfov), stream or None)
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_frame_transform_dev")
        return kp, rows.value

    def find_fovs(self, distortion_model: str, digital_lens, timestamps_ms, margin=2.0, stream=0):
        """FovIterative::compute on the device: per-frame minimal FOV (zooming/fov_iterative.rs:31-134)."""
        ts = np.ascontiguousarray(timestamps_ms, dtype=np.float64)
        out = np.zeros(ts.size, np.float64)
        rc = self._lib.gf_cuda_find_fovs(self._h, C.byref(self.cp.c), abi.LENS[distortion_model], abi.LENS[digital_lens] if digital_lens else 0,
                                         ts.ctypes.data, ts.size, margin, out.ctypes.data, stream or None)
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_find_fovs")
        return out

    def undistort_points(self, distortion_model: str, digital_lens, points_xy, timestamp_ms, frame=0, use_fovs=False, lens_correction_amount=1.0):
        """undistort_points_with_rolling_shutter (cpu_undistort.rs:636-641) on the device; points_xy: (n, 2) float32."""
        pts = np.ascontiguousarray(points_xy, dtype=np.float32).reshape(-1, 2)
        out = np.zeros_like(pts)
        rc = self._lib.gf_cuda_undistort_points(self._h, C.byref(self.cp.c), abi.LENS[distortion_model], abi.LENS[digital_lens] if digital_lens else 0,
                                                timestamp_ms, frame, int(use_fovs), lens_correction_amount, pts.ctypes.data, pts.shape[0], out.ctypes.data, None)
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_undistort_points")
        return out

    def generate_stmap(self, distortion_model: str, digital_lens, timestamp_ms, frame=0, per_frame=True):
        """generate_stmaps for one frame (stmap.rs:6-146): returns (dist[h, w, 3], undist[new_h, new_w, 3]) float32 RGB maps."""
        import torch
        m, d = abi.LENS[distortion_model], abi.LENS[digital_lens] if digital_lens else 0
        nw, nh = C.c_int32(), C.c_int32()
        rc = self._lib.gf_cuda_generate_stmap(self._h, C.byref(self.cp.c), m, d, int(per_frame), frame, timestamp_ms, C.byref(nw), C.byref(nh), None, 0, None, 0, None)
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_generate_stmap (size query)")
        w, h = self.cp.c.width, self.cp.c.height
        dist = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        und = torch.empty((nh.value, nw.value, 3), dtype=torch.float32, device="cuda")
        rc = self._lib.gf_cuda_generate_stmap(self._h, C.byref(self.cp.c), m, d, int(per_frame), frame, timestamp_ms, C.byref(nw), C.byref(nh),
                                              dist.data_ptr(), dist.numel(), und.data_ptr(), und.numel(), None)
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_generate_stmap")
        torch.cuda.synchronize()
        return dist.cpu().numpy(), und.cpu().numpy()

    def close(self):
        if self._h:
            self._lib.gf_cuda_gyro_free(self._h); self._h = None

    def __del__(self):
        try: self.close()
        except Exception: pass


def zoom_dynamic(fov_minimal, window_s, fps, method=1):
    """zoom_dynamic::compute, static-window branch (zoom_dynamic.rs:56-76) — host."""
    lib = abi.load_library()
    a = np.ascontiguousarray(fov_minimal, dtype=np.float64)
    out = np.zeros_like(a)
    rc = lib.gf_zoom_dynamic_compute(a.ctypes.data, a.size, window_s, fps, method, out.ctypes.data)
    if rc != 0:
        raise GyroflowCoreError(rc, "gf_zoom_dynamic_compute")
    return out


def scan_tables_dev(matrices_dev: int, matrix_rows: int, table_flags_dev: int, stream: int = 0):
    """Asynchronous: one small kernel on `stream` writes the table's trust verdict (0 = tame, IBIS-free) to the device word."""
    rc = abi.load_library().gf_cuda_scan_tables_dev(matrices_dev, matrix_rows, table_flags_dev, stream or None)
    if rc != 0:
        raise GyroflowCoreError(rc, "gf_cuda_scan_tables_dev")


def bind_thread_to_device(device: int) -> int:
    """Pin the calling thread to the CPUs of the GPU's NUMA node (call before allocating page-locked buffers).  Returns the CPU count."""
    return int(abi.load_library().gf_cuda_bind_thread_to_device(device))


def host_register(arr: np.ndarray):
    """Page-lock a host array in place (gf_cuda_host_register); pair with host_unregister before the array is freed."""
    rc = abi.load_library().gf_cuda_host_register(arr.ctypes.data, arr.nbytes)
    if rc != 0:
        raise GyroflowCoreError(rc, "gf_cuda_host_register")


def host_unregister(arr: np.ndarray):
    rc = abi.load_library().gf_cuda_host_unregister(arr.ctypes.data)
    if rc != 0:
        raise GyroflowCoreError(rc, "gf_cuda_host_unregister")


def stab_config(params: abi.KernelParams, pixel_type: str, digital_lens=None, base_flags=0, background=(0.0, 0.0, 0.0, 0.0),
                canvas_scale=1.0, show_safe_area=False, adaptive_zoom_window=0.0):
    """gf_stab_config from the per-buffer half of a KernelParams (what `Stabilization` holds: size, output_size, interpolation, ...)."""
    st = abi.StabConfig()
    st.width, st.height, st.output_width, st.output_height = params.width, params.height, params.output_width, params.output_height
    st.interpolation = params.interpolation
    st.pixel_type = abi.PIXEL_TYPES[pixel_type][0]
    st.base_flags = base_flags
    st.has_digital_lens = 1 if digital_lens else 0
    st.background[:] = [float(v) for v in background]
    st.canvas_scale = canvas_scale
    st.show_safe_area = int(show_safe_area)
    st.adaptive_zoom_window = adaptive_zoom_window
    return st


def get_frame_transform_at(stab: abi.StabConfig, cp: ComputeParams, buffers: Buffers, kernel_params: abi.KernelParams, mesh=None, frame=0, minimal_fov=1.0, timestamp_ms=0.0):
    """Stabilization::get_frame_transform_at (stabilization/mod.rs:253-326): completes `kernel_params` (as produced by at_timestamp) in place."""
    i, o = buffers.input.to_c(), buffers.output.to_c()
    m = None if mesh is None else np.ascontiguousarray(mesh, dtype=np.float32)
    rc = abi.load_library().gf_get_frame_transform_at(C.byref(stab), C.byref(cp.c), C.byref(i), C.byref(o), m.ctypes.data if m is not None and m.size else None,
                                                      m.size if m is not None else 0, float(timestamp_ms), frame, minimal_fov, C.byref(kernel_params))
    if rc != 0:
        raise GyroflowCoreError(rc, "gf_get_frame_transform_at")
    return kernel_params
