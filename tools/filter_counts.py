"""Per-frame counts of the packed fisheye kernel's filtered rolling-shutter pre-pass: how many pairs and pixels its main launch
leaves to the tail launch, and whether a queue overflowed (then the tail re-renders the whole frame).

  uncertain   pairs whose mid-row row index the approximate evaluation could not certify
  bad         pairs whose final pass left the window of the exact fast sequences (w <= 0, far coordinates, ...)
  px          pixels whose 8-bit bilinear footprint is not interior (background, source rect edges)

These numbers size the queues (c_abi.cu: defer_cap, defer_cap_px) and explain the tail launch's share of the frame time.

    python tools/filter_counts.py [--frames N] [--cases]

Default: N frames shaped like bench.py's headline (3840x2160 RGBA8, opencv_fisheye, 16 ms rolling shutter, 60 fps timestamps of
the synthetic gyro).  --cases adds filtered frames like those of the parity tests: strong roll, zoomed-out views (background,
rays past 90 degrees), a source rect smaller than the frame, a lens at its conditioning cap.  Needs a GPU.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import gyroflow_b200 as g  # noqa: E402
from gyroflow_b200 import synth  # noqa: E402

W, H, PIX, LENS = 3840, 2160, "RGBA8", "opencv_fisheye"

CASES = [
    dict(w=1920, h=1080, video_rotation=33.0), dict(w=1920, h=1080, fov=3.5, ts=1234.0),
    dict(w=1280, h=720, params=dict(k=[-0.21, 0.0, 0.0, 0.0] + [0.0] * 8), fov=1.7), dict(w=3840, h=2160, ts=3456.7, pix="Luma8"),
    dict(w=1280, h=720, fov=1.6, in_rect=(160, 90, 960, 540)), dict(w=1280, h=720, fov=3.0, ts=777.0, readout=33.0),
    dict(w=1031, h=577, fov=8.0, ts=1999.0, readout=33.0),
]


def render(wrapper_args, bufs, itm):
    w = g.CudaWrapper.new(*wrapper_args, bufs)
    try:
        w.undistort_image(bufs, itm)
        return w.filter_counts()
    finally:
        w.close()


def row(label, c):
    return dict(frame=label, uncertain=c["pairs"] - c["bad_pairs"], bad=c["bad_pairs"], px=c["pixels"], overflow=c["overflow"])


def bench_frames(n):
    p = synth.base_kernel_params(W, H, pixel_type=PIX, lens=LENS, fov=1.0, interpolation="Bilinear")
    org, sm = synth.synthetic_gyro(n / 60.0 + 2.0)
    cp = g.ComputeParams(p, org, sm, frame_readout_time_ms=16.0)
    st = g.stab_config(p, PIX)
    src = synth.synthetic_frame(W, H, PIX, stride=p.stride)
    dst = np.zeros((H, p.output_stride), np.uint8)
    bufs = g.Buffers(g.BufferDescription((W, H, p.stride), src), g.BufferDescription((W, H, p.output_stride), dst))
    for f in range(n):
        kp, mats, _, _ = cp.at_timestamp(500.0 + f * (1000.0 / 60.0), f)
        g.get_frame_transform_at(st, cp, bufs, kp, frame=f)          # the per-buffer half: sizes, strides, rects, interpolation
        yield row(f, render((kp, PIX, LENS, None), bufs, g.FrameTransform(matrices=mats, kernel_params=kp)))


def case_frames():
    from tests import cases
    for c in CASES:
        p, src, m, mesh, dst, pix, lens, digital = cases.build(c)
        bw, bh = c.get("in_size", (c["w"], c["h"]))
        bufs = g.Buffers(g.BufferDescription((bw, bh, p.stride), src), g.BufferDescription((c["w"], c["h"], p.output_stride), dst))
        yield row(json.dumps(c), render((p, pix, lens, digital), bufs, g.FrameTransform(matrices=m, kernel_params=p)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--cases", action="store_true")
    args = ap.parse_args()
    g.load_library()
    print("device:", g.list_devices()[0])
    rows = list(bench_frames(args.frames))
    for r in rows:
        print(json.dumps(r))
    pairs, pixels = W * H // 2, W * H
    print("bench frames: max uncertain %.3f %% of pairs, max bad %d, max px %.3f %% of pixels, overflow in %d of %d" % (
        100.0 * max(r["uncertain"] for r in rows) / pairs, max(r["bad"] for r in rows), 100.0 * max(r["px"] for r in rows) / pixels,
        sum(r["overflow"] for r in rows), len(rows)))
    if args.cases:
        for r in case_frames():
            print(json.dumps(r))


if __name__ == "__main__":
    main()
