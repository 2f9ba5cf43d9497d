"""Frame-sharded render queue: the multi-GPU shape of the path (SURVEY.md §8e).

Frames are independent units (FrameTransform::at_timestamp depends only on immutable params + the timestamp,
src/core/stabilization/frame_transform.rs:165), so frame i goes to rank i % world and there is NO data-path collective.
The only communication is one broadcast, at job start, of the tables every rank needs (KernelParams template,
lens coefficients, per-frame matrix tables / quaternion tracks) from rank 0 — NCCL over NVLink on GPUs, gloo in the CPU
tests.  The reference has no counterpart: its render queue runs whole jobs in parallel (rendering/render_queue.rs:550-612)
but each job is a sequential decode -> warp -> encode loop on one device (rendering/mod.rs:451).
"""
import ctypes as C

import numpy as np

from . import abi
from .backend import GyroflowCoreError


class RenderQueue:
    """One GPU's render queue (gf_cuda_queue, csrc/render_queue.cu): `depth` frames in flight, each
    producer kernel -> [H2D] -> warp -> [checksum] -> [D2H] on its own stream; results come back in submission order.

    bench.py and the multi-GPU tests drive this class: rank r of a world of G submits frames r, r + G, r + 2G, ...
    (shard_frames) and the per-frame checksums are gathered in frame order (gather_results)."""

    def __init__(self, compute_params, stab: abi.StabConfig, distortion_model: str, digital_lens, in_proto, out_proto,
                 device=0, depth=4, pin_numa=True, checksum=False):
        self._lib = abi.load_library()
        self.cp = compute_params                      # keeps the arrays alive
        cfg = abi.QueueConfig()
        cfg.device = device
        cfg.distortion_model = abi.LENS[distortion_model]
        cfg.digital_lens = abi.LENS[digital_lens] if digital_lens else 0
        cfg.depth, cfg.pin_numa, cfg.checksum = depth, int(pin_numa), int(checksum)
        cfg.stab = stab
        self.depth = depth
        self.in_flight = 0
        h = C.c_void_p()
        i, o = in_proto.to_c(), out_proto.to_c()
        rc = self._lib.gf_cuda_queue_create(C.byref(h), C.byref(cfg), C.byref(compute_params.c), C.byref(i), C.byref(o))
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_queue_create: " + (self._lib.gf_cuda_last_error(None) or b"").decode())
        self._h = h

    def _err(self, rc, what):
        return GyroflowCoreError(rc, what + ": " + (self._lib.gf_cuda_queue_last_error(self._h) or b"").decode())

    def submit(self, frame: int, timestamp_ms: float, buffers, mesh=None):
        """Enqueue one frame.  The queue must have a free slot (in_flight < depth): call wait() first otherwise."""
        i, o = buffers.input.to_c(), buffers.output.to_c()
        m = None if mesh is None else np.ascontiguousarray(mesh, dtype=np.float32)
        rc = self._lib.gf_cuda_queue_submit(self._h, frame, timestamp_ms, C.byref(i), C.byref(o),
                                            m.ctypes.data if m is not None and m.size else None, m.size if m is not None else 0)
        if rc != 0:
            raise self._err(rc, "gf_cuda_queue_submit")
        self.in_flight += 1

    def wait(self):
        """Block until the oldest in-flight frame is finished; returns (frame, checksum)."""
        f = C.c_size_t(); s = C.c_uint64()
        rc = self._lib.gf_cuda_queue_wait(self._h, C.byref(f), C.byref(s))
        if rc != 0:
            raise self._err(rc, "gf_cuda_queue_wait")
        self.in_flight -= 1
        return int(f.value), int(s.value)

    def render(self, frames, timestamp_of, buffers_of, mesh_of=None):
        """Run `frames` (an iterable of frame indices) through the queue keeping it full; returns {frame: checksum} in frame order."""
        out = {}
        for f in frames:
            if self.in_flight == self.depth:
                k, v = self.wait(); out[k] = v
            self.submit(f, timestamp_of(f), buffers_of(f), mesh_of(f) if mesh_of else None)
        while self.in_flight:
            k, v = self.wait(); out[k] = v
        return dict(sorted(out.items()))

    def drain(self):
        rc = self._lib.gf_cuda_queue_drain(self._h)
        if rc != 0:
            raise self._err(rc, "gf_cuda_queue_drain")
        self.in_flight = 0

    @property
    def launch_count(self):
        return int(self._lib.gf_cuda_queue_launches(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gf_cuda_queue_destroy(self._h); self._h = None

    def __del__(self):
        try: self.close()
        except Exception: pass


class FrameRenderQueue:
    """A render queue over whole decoder frames (gf_cuda_queue_create_frame): every submission is all planes of one frame of `format`
    (NV12, P010LE, YUV420P, ... — abi.FRAME_FORMATS), with one producer launch per frame and each plane's KernelParams set the way the
    reference's per-plane closures set them (rendering/mod.rs:483-548): value limit, background converted for the plane, plane_index,
    per-frame FILL_WITH_BACKGROUND.  `stab` describes the whole frame; its pixel_type is ignored.  in_protos / out_protos: one
    BufferDescription per plane in the order of frame_layout(format, ...)."""

    def __init__(self, compute_params, stab: abi.StabConfig, format: str, distortion_model: str, digital_lens, in_protos, out_protos,
                 limited_range=False, device=0, depth=4, pin_numa=True, checksum=False):
        self._lib = abi.load_library()
        self.cp = compute_params
        cfg = abi.QueueConfig()
        cfg.device = device
        cfg.distortion_model = abi.LENS[distortion_model]
        cfg.digital_lens = abi.LENS[digital_lens] if digital_lens else 0
        cfg.depth, cfg.pin_numa, cfg.checksum = depth, int(pin_numa), int(checksum)
        cfg.stab = stab
        self.depth = depth
        self.in_flight = 0
        self.n_planes = len(in_protos)
        h = C.c_void_p()
        i = (abi.BufferDesc * self.n_planes)(*[b.to_c() for b in in_protos])
        o = (abi.BufferDesc * len(out_protos))(*[b.to_c() for b in out_protos])
        rc = self._lib.gf_cuda_queue_create_frame(C.byref(h), C.byref(cfg), C.byref(compute_params.c), abi.FRAME_FORMATS[format],
                                                  int(limited_range), self.n_planes, i, o)
        if rc != 0:
            raise GyroflowCoreError(rc, "gf_cuda_queue_create_frame: " + (self._lib.gf_cuda_last_error(None) or b"").decode())
        self._h = h

    def _err(self, rc, what):
        return GyroflowCoreError(rc, what + ": " + (self._lib.gf_cuda_queue_last_error(self._h) or b"").decode())

    def submit(self, frame: int, timestamp_ms: float, planes, mesh=None, fill_with_background=False):
        """Enqueue one frame; `planes` is a list of Buffers, one per plane.  The queue must have a free slot."""
        n = len(planes)
        i = (abi.BufferDesc * max(n, 1))(*[b.input.to_c() for b in planes])
        o = (abi.BufferDesc * max(n, 1))(*[b.output.to_c() for b in planes])
        m = None if mesh is None else np.ascontiguousarray(mesh, dtype=np.float32)
        rc = self._lib.gf_cuda_queue_submit_frame(self._h, frame, timestamp_ms, n, i, o, m.ctypes.data if m is not None and m.size else None,
                                                  m.size if m is not None else 0, int(bool(fill_with_background)))
        if rc != 0:
            raise self._err(rc, "gf_cuda_queue_submit_frame")
        self.in_flight += 1

    def wait(self):
        """Block until the oldest in-flight frame is finished; returns (frame, (checksum per plane))."""
        f = C.c_size_t(); s = (C.c_uint64 * self.n_planes)()
        rc = self._lib.gf_cuda_queue_wait_frame(self._h, C.byref(f), s, self.n_planes)
        if rc != 0:
            raise self._err(rc, "gf_cuda_queue_wait_frame")
        self.in_flight -= 1
        return int(f.value), tuple(int(v) for v in s)

    def render(self, frames, timestamp_of, planes_of, mesh_of=None, fill_of=None):
        """Run `frames` through the queue keeping it full; returns {frame: (checksum per plane)} in frame order."""
        out = {}
        for f in frames:
            if self.in_flight == self.depth:
                k, v = self.wait(); out[k] = v
            self.submit(f, timestamp_of(f), planes_of(f), mesh_of(f) if mesh_of else None, fill_of(f) if fill_of else False)
        while self.in_flight:
            k, v = self.wait(); out[k] = v
        return dict(sorted(out.items()))

    @property
    def launch_count(self):
        return int(self._lib.gf_cuda_queue_launches(self._h))

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gf_cuda_queue_destroy(self._h); self._h = None

    def __del__(self):
        try: self.close()
        except Exception: pass


def checksum_host(buf: np.ndarray) -> int:
    """The queue's per-frame checksum on the host: sum(word[i] * (2 i + 1)) mod 2^64 over the buffer's 32-bit words."""
    w = np.ascontiguousarray(buf).view(np.uint8).reshape(-1)
    w = w[: w.size // 4 * 4].view(np.uint32).astype(np.uint64)
    k = np.arange(w.size, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    with np.errstate(over="ignore"):
        return int((w * k).sum(dtype=np.uint64))


def shard_frames(n_frames, world, rank):
    """Frame indices owned by `rank`: round-robin, so every rank sees the same mix of timestamps."""
    return list(range(rank, n_frames, world))


def frame_owner(frame, world):
    return frame % world


def params_to_tensor(p, torch):
    """KernelParams (368 B) as a uint8 tensor (for the broadcast)."""
    raw = C.string_at(C.byref(p), C.sizeof(abi.KernelParams))
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).clone()


def params_from_tensor(t):
    p = abi.KernelParams()
    raw = bytes(t.cpu().numpy().tobytes())
    C.memmove(C.byref(p), raw, C.sizeof(abi.KernelParams))
    return p


def broadcast_tables(params, matrices, dist, torch, device, src=0):
    """One-time broadcast of the job's tables from `src`.  `params`/`matrices` are only read on the source rank;
    every rank passes the expected matrices shape.  Returns (KernelParams, matrices tensor on `device`)."""
    rank = dist.get_rank()
    pt = params_to_tensor(params, torch).to(device) if rank == src else torch.empty(C.sizeof(abi.KernelParams), dtype=torch.uint8, device=device)
    shape = torch.tensor(list(matrices.shape) if rank == src else [0, 0, 0], dtype=torch.int64, device=device)
    dist.broadcast(shape, src=src)
    mt = (torch.as_tensor(np.ascontiguousarray(matrices, dtype=np.float32)).to(device) if rank == src
          else torch.empty(tuple(int(v) for v in shape.tolist()), dtype=torch.float32, device=device))
    dist.broadcast(pt, src=src)
    dist.broadcast(mt, src=src)
    return params_from_tensor(pt), mt


def _as_i64(v):
    v &= (1 << 64) - 1
    return v - (1 << 64) if v >= (1 << 63) else v


def gather_results(local, dist, torch, device, dst=0):
    """Collect {frame: value} dicts (small per-frame results such as 64-bit checksums) on every rank, restoring frame order."""
    local = {k: _as_i64(int(v)) for k, v in local.items()}
    world = dist.get_world_size()
    keys = torch.tensor(sorted(local), dtype=torch.int64, device=device)
    vals = torch.tensor([local[k] for k in sorted(local)], dtype=torch.int64, device=device)
    n = torch.tensor([keys.numel()], dtype=torch.int64, device=device)
    ns = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(ns, n)
    m = int(max(int(v.item()) for v in ns))
    pad = lambda t: torch.cat([t, torch.full((m - t.numel(),), -1, dtype=torch.int64, device=device)])
    ks = [torch.empty(m, dtype=torch.int64, device=device) for _ in range(world)]
    vs = [torch.empty(m, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(ks, pad(keys)); dist.all_gather(vs, pad(vals))
    out = {}
    for k, v in zip(ks, vs):
        for a, b in zip(k.tolist(), v.tolist()):
            if a >= 0: out[a] = b & ((1 << 64) - 1)
    return dict(sorted(out.items()))
