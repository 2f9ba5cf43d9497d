#!/bin/sh
# Runs ON THE GPU BOX: compute-sanitizer memcheck + racecheck + initcheck-free runs over the smoke case, one filtered-pre-pass frame with
# deferred pairs, one two-pass (Lanczos4) case, one fused multi-plane case and a short render-queue run.  Logs -> gpurun_out/sanitizer_*.log
# The Python cases end with a short NV12 frame queue over page-locked HOST planes.
cat > /tmp/san_cases.py <<'PY'
import sys, numpy as np
sys.path.insert(0, ".")
import gyroflow_b200 as g
from gyroflow_b200 import synth
from tests import cases
import __graft_entry__ as ge
ge.smoke()
for case in (dict(w=640, h=360, video_rotation=20.0), dict(w=320, h=180, interp="Lanczos4"), dict(w=320, h=180, pix="RGBAf", lens="sony", ibis=True, mesh=True),
             dict(w=320, h=180, lens="gopro", digital="gopro_warp", fov=2.0), dict(w=203, h=117, pix="RGB8", stride_pad=3),
             dict(w=200, h=120, interp="Lanczos4", pix="Luma8", fov=1.4), dict(w=203, h=117, interp="Bicubic", pix="UV8", stride_pad=2, fov=1.4), dict(w=203, h=117, interp="Lanczos4", pix="RGBA8", stride_pad=4, fov=1.4)):
    p, src, m, mesh, dst0, pix, lens, digital = cases.build(case)
    got = dst0.copy()
    bufs = g.Buffers(g.BufferDescription((case["w"], case["h"], p.stride), src), g.BufferDescription((case["w"], case["h"], p.output_stride), got))
    w = g.CudaWrapper.new(p, pix, lens, digital, bufs)
    w.undistort_image(bufs, g.FrameTransform(matrices=m, kernel_params=p, mesh_data=mesh if mesh is not None else np.zeros(0, np.float32)))
    w.close()
import torch
p = synth.base_kernel_params(320, 180); org, sm = cases.gyro(); cp = g.ComputeParams(p, org, sm); st = g.stab_config(p, "RGBA8")
src = torch.zeros((180, p.stride), dtype=torch.uint8, device="cuda"); outs = [torch.zeros((180, p.output_stride), dtype=torch.uint8, device="cuda") for _ in range(6)]
mk = lambda f: g.Buffers(g.BufferDescription((320, 180, p.stride), src.data_ptr(), length=src.numel()), g.BufferDescription((320, 180, p.output_stride), outs[f].data_ptr(), length=outs[f].numel()))
q = g.RenderQueue(cp, st, "opencv_fisheye", None, mk(0).input, mk(0).output, depth=3, checksum=True)
print(q.render(range(6), lambda f: 100.0 + 16.6 * f, mk)); q.close()
# a small NV12 frame queue with page-locked HOST planes (two warp contexts, one producer launch, one checksum launch per frame)
lay = g.frame_layout("NV12", 321, 181); st = g.stab_config(synth.base_kernel_params(321, 181), "Luma8")
cp = g.ComputeParams(synth.base_kernel_params(321, 181), org, sm, fov_scale=1.5)
hb = [[(torch.from_numpy(synth.synthetic_frame(l["width"], l["height"], l["pixel_type"], frame=f, stride=512)).pin_memory(),
        torch.zeros((l["height"], 512), dtype=torch.uint8).pin_memory()) for l in lay] for f in range(4)]
pk = lambda f: [g.Buffers(g.BufferDescription((l["width"], l["height"], 512), a.numpy()), g.BufferDescription((l["width"], l["height"], 512), b.numpy())) for l, (a, b) in zip(lay, hb[f])]
fq = g.FrameRenderQueue(cp, st, "NV12", "opencv_fisheye", None, [x.input for x in pk(0)], [x.output for x in pk(0)], depth=2, checksum=True)
print(fq.render(range(4), lambda f: 100.0 + 16.6 * f, pk, fill_of=lambda f: f == 2)); fq.close()
print("sanitizer cases done")
PY
for tool in memcheck racecheck; do
  timeout 900 compute-sanitizer --tool $tool --print-limit 20 python /tmp/san_cases.py > gpurun_out/sanitizer_$tool.log 2>&1
  tail -4 gpurun_out/sanitizer_$tool.log
done
