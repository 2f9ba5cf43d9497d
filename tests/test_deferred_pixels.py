"""The filtered main launch of the packed fisheye kernel keeps its rare cases out of line: pairs whose final pass leaves the exact fast
sequences' window (`bad`) and pixels whose 8-bit footprint is not interior go to queues that the tail launch renders, and a full queue
makes the tail launch re-render the whole frame.  Every route against the CPU oracle, bit for bit, with the frame's counters
(gf_cuda_filter_counts) showing that the route was taken."""
import numpy as np
import pytest

import gyroflow_b200 as g
from gyroflow_b200 import render_queue, synth
from tests import cases, oracle_lib
from tests.test_render_queue import _expected

pytestmark = pytest.mark.gpu


def _render(case, frames=1):
    """Render `case` `frames` times through one context; returns (mismatching bytes, counters of the last frame, launches)."""
    p, src, m, mesh, dst0, pix, lens, digital = cases.build(case)
    want = dst0.copy()
    assert oracle_lib.undistort_image(src, want, p, pix, lens, digital, m, mesh) == 0
    got = dst0.copy()
    bufs = g.Buffers(g.BufferDescription((case["w"], case["h"], p.stride), src), g.BufferDescription((case["w"], case["h"], p.output_stride), got))
    w = g.CudaWrapper.new(p, pix, lens, digital, bufs)
    try:
        for _ in range(frames):
            got[:] = dst0
            w.undistort_image(bufs, g.FrameTransform(matrices=m, kernel_params=p))
        return int((want != got).sum()), w.filter_counts(), w.launch_count
    finally:
        w.close()


# many outputs map outside the source: zoomed-out views, a source rect smaller than the frame
NON_INTERIOR = [dict(w=1280, h=720, fov=1.6), dict(w=1280, h=720, fov=1.3, in_rect=(160, 90, 960, 540)),
                dict(w=1280, h=720, fov=1.2, ts=2345.6, pix="Luma8"), dict(w=640, h=360, fov=1.5, pix="RGB8", in_rect=(1, 2, 600, 301))]


def _on_axis(rows):
    """Zero the rows' x and y terms: every pixel whose final row is one of them lands exactly on the optical axis (r == 0), which the
    final pass's operand window sends to the exact code.  The mid row stays ordinary unless it is zeroed too."""
    def hook(m):
        sel = rows(m.shape[0])
        m[sel, 0:6] = 0.0
        return m
    return hook


# pairs the final pass flags `bad` after a certified mid-row pass.  (Rays near or past 90 degrees off axis, w <= 0, already fail the
# pre-pass's certificate: r^2 leaves its regime, so those pairs are deferred as uncertified.)
BAD = [dict(w=640, h=360, matrix_hook=_on_axis(lambda n: slice(0, n))), dict(w=1280, h=720, matrix_hook=_on_axis(lambda n: slice(0, n // 3))),
       dict(w=960, h=540, pix="UV8", matrix_hook=_on_axis(lambda n: slice(2 * n // 3, n)))]


@pytest.mark.parametrize("case", NON_INTERIOR)
def test_non_interior_pixels_finished_by_the_tail(case):
    bad, c, launches = _render(case)
    assert bad == 0, (bad, c)
    assert launches == 2 and c["pixels"] > 1000 and not c["overflow"], c


@pytest.mark.parametrize("case", BAD)
def test_bad_pairs_rendered_by_the_tail(case):
    bad, c, _ = _render(case)
    assert bad == 0, (bad, c)
    assert c["bad_pairs"] > 0 and c["pairs"] >= c["bad_pairs"] and not c["overflow"], c


@pytest.mark.parametrize("case", [NON_INTERIOR[0], NON_INTERIOR[1], BAD[1], dict(w=1920, h=1080, video_rotation=33.0)])
def test_full_queue_rerenders_the_whole_frame(case, monkeypatch):
    monkeypatch.setenv("GF_X2_DEFER_CAP", "64")
    bad, c, _ = _render(case, frames=3)        # three frames on one context: both counter sets re-armed in turn
    assert bad == 0, (bad, c)
    assert c["overflow"] and c["pairs"] + c["pixels"] > 64, c


def test_counters_rearmed_between_frames(monkeypatch):
    """An overflowing frame followed by ordinary frames on the same context: the later frames' counters start from zero."""
    monkeypatch.setenv("GF_X2_DEFER_CAP", "100000")
    big, small = dict(w=1280, h=720, fov=3.0, ts=777.0), dict(w=1280, h=720, ts=777.0)
    pb, src, mb, _, dst0, pix, lens, _ = cases.build(big)
    ps, _, ms, _, _, _, _, _ = cases.build(small)
    got = dst0.copy()
    bufs = g.Buffers(g.BufferDescription((1280, 720, pb.stride), src), g.BufferDescription((1280, 720, pb.output_stride), got))
    w = g.CudaWrapper.new(pb, pix, lens, None, bufs)
    try:
        w.undistort_image(bufs, g.FrameTransform(matrices=mb, kernel_params=pb))
        assert w.filter_counts()["overflow"]
        seen = []
        for _ in range(3):
            got[:] = dst0
            w.undistort_image(bufs, g.FrameTransform(matrices=ms, kernel_params=ps))
            seen.append(w.filter_counts())
    finally:
        w.close()
    want = dst0.copy()
    assert oracle_lib.undistort_image(src, want, ps, pix, lens, None, ms, None) == 0
    assert np.array_equal(got, want)
    assert not any(c["overflow"] for c in seen) and seen[0] == seen[1] == seen[2], seen


@pytest.mark.parametrize("cap", [None, "3000"])
def test_render_queue_frames_in_flight(cap, monkeypatch):
    """Zoomed-out frames mixed with ordinary ones, four in flight per queue: with the default queues, and with queues small enough that
    at least the zoomed-out frames overflow."""
    import torch
    if cap:
        monkeypatch.setenv("GF_X2_DEFER_CAP", cap)
    W, H, pix, lens = 640, 360, "RGBA8", "opencv_fisheye"
    n = 10
    p = synth.base_kernel_params(W, H, pixel_type=pix, lens=lens)
    org, sm = cases.gyro()
    cp = g.ComputeParams(p, org, sm, fovs=[(1.0, 2.6, 1.4, 1.0, 4.0)[f % 5] for f in range(n)])
    st = g.stab_config(p, pix)
    src = synth.synthetic_frame(W, H, pix, stride=p.stride)
    tsrc = torch.from_numpy(src).cuda()
    outs = [torch.zeros((H, p.output_stride), dtype=torch.uint8, device="cuda") for _ in range(n)]
    bufs = [g.Buffers(g.BufferDescription((W, H, p.stride), tsrc.data_ptr(), length=tsrc.numel()),
                      g.BufferDescription((W, H, p.output_stride), o.data_ptr(), length=o.numel())) for o in outs]
    q = g.RenderQueue(cp, st, lens, None, bufs[0].input, bufs[0].output, depth=4, checksum=True)
    ts_of = lambda f: 900.0 + f * (1000.0 / 60.0)
    sums = q.render(range(n), ts_of, lambda f: bufs[f])
    q.close()
    dg = g.DeviceGyro(cp)
    mats = torch.zeros((max(W, H), 14), dtype=torch.float32, device="cuda")
    for f in range(n):
        want = _expected(p, cp, st, dg, mats, ts_of(f), f, src, pix, lens, None, bufs[f])
        assert np.array_equal(outs[f].cpu().numpy(), want), "frame %d" % f
        assert sums[f] == render_queue.checksum_host(want)
    dg.close()
