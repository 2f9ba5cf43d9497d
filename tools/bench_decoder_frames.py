#!/usr/bin/env python3
"""Decoder-frame throughput of the render queue: whole 4K NV12, P010LE and YUV420P frames (opencv_fisheye, rolling shutter, bilinear)
through FrameRenderQueue, with DEVICE frames (4 in flight, an input ring larger than the 126 MB L2) and with page-locked HOST frames
(5 in flight).  For each it reports frames/s, kernel launches per frame, bytes per frame each way over the host link, and the same
frames through the reference-shaped chain (host at_timestamp, then one synchronous gf_cuda_undistort_image per plane, like the
per-plane closures of rendering/mod.rs:517-545 called in turn at :657-661).  A few timed frames' per-plane checksums are checked
against the CPU oracle in the same run.  Prints one JSON line.

    python tools/bench_decoder_frames.py [--frames 2000] [--warmup 24]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import gyroflow_b200 as g
from gyroflow_b200 import abi, render_queue, synth
from tests import oracle_lib

W, H = 3840, 2160
FPS = 30.0
LENS = "opencv_fisheye"
L2_BYTES = 126 << 20


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    f = [x.strip() for x in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return dict(name=f[0], power_limit_w=float(f[1]), sm_clock_mhz=float(f[2]), sm_clock_max_mhz=float(f[3])) if len(f) == 4 else dict(name=None)


def ts_of(f):
    return 100.0 + f * (1000.0 / FPS)


class Workload:
    def __init__(self, fmt, kind, n_total):
        self.fmt, self.kind = fmt, kind
        self.layout = g.frame_layout(fmt, W, H)
        self.p = synth.base_kernel_params(W, H, lens=LENS)
        org, sm = synth.synthetic_gyro(n_total / FPS + 2.0)
        self.cp = g.ComputeParams(self.p, org, sm)                       # 16 ms readout: rolling shutter on
        self.st = g.stab_config(self.p, "Luma8")
        self.strides = []
        for pl in self.layout:
            _, count, sdt = abi.PIXEL_TYPES[pl["pixel_type"]]
            self.strides.append(pl["width"] * count * np.dtype(sdt).itemsize)
        self.frame_bytes = sum(s * pl["height"] for s, pl in zip(self.strides, self.layout))
        self.depth = 4 if kind == "device" else 5
        n_in = max(4, -(-2 * L2_BYTES // self.frame_bytes)) if kind == "device" else 8
        n_out = self.depth + 4
        self.srcs = [[self._plane(pl, s, 3 * f + i, True) for i, (pl, s) in enumerate(zip(self.layout, self.strides))] for f in range(n_in)]
        self.outs = [[self._plane(pl, s, 0, False) for pl, s in zip(self.layout, self.strides)] for _ in range(n_out)]

    def _plane(self, pl, stride, seed, src):
        a = synth.synthetic_frame(pl["width"], pl["height"], pl["pixel_type"], frame=seed, stride=stride) if src else \
            np.zeros((pl["height"], stride), np.uint8)
        t = torch.from_numpy(a)
        return t.cuda() if self.kind == "device" else t.pin_memory()

    def _desc(self, t, pl, stride):
        if self.kind == "device":
            return g.BufferDescription((pl["width"], pl["height"], stride), t.data_ptr(), length=t.numel())
        return g.BufferDescription((pl["width"], pl["height"], stride), t.numpy())

    def planes(self, f):
        s, o = self.srcs[f % len(self.srcs)], self.outs[f % len(self.outs)]
        return [g.Buffers(self._desc(a, pl, st), self._desc(b, pl, st)) for a, b, pl, st in zip(s, o, self.layout, self.strides)]

    def queue(self):
        b = self.planes(0)
        return g.FrameRenderQueue(self.cp, self.st, self.fmt, LENS, None, [x.input for x in b], [x.output for x in b], depth=self.depth, checksum=True)

    def plane_params(self, kp, f, i, bufs):
        pl = self.layout[i]
        k = kp.copy()
        st = g.stab_config(self.p, pl["pixel_type"], background=g.background_for_plane(pl["pixel_type"], (0, 0, 0, 0), pl["ind"], False))
        g.get_frame_transform_at(st, self.cp, bufs[i], k, frame=f)
        k.pixel_value_limit = pl["max_value"]; k.max_pixel_value = pl["max_value"]; k.plane_index = i
        return k


def run_queue(wl, warmup, frames):
    q = wl.queue()
    q.render(range(warmup), ts_of, wl.planes)
    l0 = q.launch_count
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    sums = q.render(range(warmup, warmup + frames), ts_of, wl.planes)     # ends with a wait for every frame
    dt = time.perf_counter() - t0
    launches = (q.launch_count - l0) / frames
    q.close()
    return frames / dt, launches, sums


def run_reference_chain(wl, frames, first):
    """Host at_timestamp, then per plane get_frame_transform_at + the plane's settings and one synchronous gf_cuda_undistort_image."""
    ctxs = {}
    for i, pl in enumerate(wl.layout):
        if pl["pixel_type"] not in ctxs:
            b = wl.planes(0)
            kp, _, _, _ = wl.cp.at_timestamp(ts_of(0), 0)
            ctxs[pl["pixel_type"]] = g.CudaWrapper.new(wl.plane_params(kp, 0, i, b), pl["pixel_type"], LENS, None, b[i])
    t0 = None
    for f in range(first - 1, first + frames):                            # the first frame is warm-up
        if f == first:
            torch.cuda.synchronize(); t0 = time.perf_counter()
        bufs = wl.planes(f)
        kp, m, _, _ = wl.cp.at_timestamp(ts_of(f), f)
        for i, pl in enumerate(wl.layout):
            w = ctxs[pl["pixel_type"]]
            w.undistort_image(bufs[i], g.FrameTransform(matrices=m, kernel_params=wl.plane_params(kp, f, i, bufs)))
            w.synchronize()
    dt = time.perf_counter() - t0
    for w in ctxs.values():
        w.close()
    return frames / dt


def oracle_check(wl, frames_to_check, sums):
    """Per-plane checksums of finished frames (still in the output ring) against the oracle on the table the device producer writes."""
    dg = g.DeviceGyro(wl.cp)
    mats = torch.zeros((max(W, H), 14), dtype=torch.float32, device="cuda")
    ok = True
    for f in frames_to_check:
        kp, rows = dg.frame_transform(ts_of(f), mats.data_ptr(), max(W, H), frame=f)
        table = mats.cpu().numpy()[:rows].copy()
        bufs = wl.planes(f)
        for i, pl in enumerate(wl.layout):
            k = wl.plane_params(kp, f, i, bufs)
            want = np.zeros((pl["height"], wl.strides[i]), np.uint8)
            src = wl.srcs[f % len(wl.srcs)][i].cpu().numpy()
            assert oracle_lib.undistort_image(src, want, k, pl["pixel_type"], LENS, None, table, None) == 0
            ok &= sums[f][i] == render_queue.checksum_host(want)
    dg.close()
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=24)
    ap.add_argument("--reference-frames", type=int, default=24)
    ap.add_argument("--formats", default="NV12,P010LE,YUV420P")
    args = ap.parse_args()
    assert g.load_library().gf_cuda_device_count() > 0, "no CUDA device: nothing to measure"
    out = dict(metric="decoder_frames_per_s", size=[W, H], lens=LENS, rolling_shutter=True, interpolation="Bilinear",
               card=card(), workloads={})
    for fmt in args.formats.split(","):
        for kind in ("device", "host"):
            wl = Workload(fmt, kind, args.warmup + args.frames + args.reference_frames)
            fps, launches, sums = run_queue(wl, args.warmup, args.frames)
            last = args.warmup + args.frames
            checked = [f for f in range(last - 2, last)]                      # still in the output ring
            ok = oracle_check(wl, checked, sums)
            ref = run_reference_chain(wl, args.reference_frames, last)
            bytes_in = sum(pl["height"] * s for pl, s in zip(wl.layout, wl.strides))
            out["workloads"]["%s_%s" % (fmt, kind)] = dict(
                frames_per_s=round(fps, 1), launches_per_frame=launches, depth=wl.depth, input_ring_frames=len(wl.srcs),
                bytes_h2d_per_frame=bytes_in if kind == "host" else 0, bytes_d2h_per_frame=bytes_in if kind == "host" else 0,
                reference_chain_frames_per_s=round(ref, 1), oracle_frames_checked=checked, oracle_checksums_match=bool(ok))
            del wl
            torch.cuda.empty_cache()
    out["card_after"] = card()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
