#!/usr/bin/env python3
"""bench.py — 4K frames/sec of the fisheye + rolling-shutter warp (BASELINE.json `metric`), one JSON line.

Workload (N=1 and per rank for N>1): BASELINE config 2 — 3840x2160 RGBA8, opencv_fisheye, rolling shutter ON
(2160 per-scanline matrices from a 240 Hz synthetic gyro), bilinear, synthetic high-entropy frames.
A "step" is one batch of FRAMES_PER_STEP frames, each with its own timestamp (distinct matrices) and drawn from a
ring of input frames larger than L2, so no launch finds its source in cache.

  value     frames/s with frames + tables already resident in HBM (gf_cuda_undistort_image_dev), CUDA-event timed,
            max over ranks
  e2e       frames/s through the reference-facing host-buffer entry points with HOST (pinned) buffers: H2D of the frame +
            tables and D2H of the result inside the timed region, for the same FRAMES_PER_STEP-frame steps.  e2e.value keeps three
            frames in flight (gf_cuda_undistort_image_async on three contexts), e2e.sync_call_value is the strictly sequential
            gf_cuda_undistort_image
  roofline  algorithmic bytes per launch (SURVEY.md §8d: in + out + rows*56 + 368) / mean launch time, vs measured HBM peak
  cpu_baseline  the CPU oracle (C port of the reference CPU path) on this box's host cores, bounded sample

`--impl reference` times the reference CPU path instead (oracle port; the Rust original cannot be built: no rustc).
Side measurements (not the headline): --config 1/3/31/4 (the other BASELINE configurations), --interp (other resamplers),
--lens (other lens models), --planes N (multi-plane frames through gf_cuda_undistort_planes_dev).

`--dump-outputs DIR` writes what the timed path rendered in its last timed step to DIR (see OutputSample), so that two builds
run with the same arguments (hence the same seeded inputs) can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

# BASELINE.json configs.  cfg2 is the one `metric` is quoted on (default); cfg1/3/4 are selectable with --config for the
# per-lens-model ncu captures (profiles/) — they are parity-test cases, not additional headline numbers.
CONFIGS = {
    1: dict(w=3840, h=2160, pix="RGBA8", lens="opencv_fisheye", digital=None, rs=False, identity=True,
            name="cfg1: 3840x2160 RGBA8, opencv_fisheye, rolling-shutter OFF, identity quaternion, bilinear"),
    2: dict(w=3840, h=2160, pix="RGBA8", lens="opencv_fisheye", digital=None, rs=True,
            name="cfg2: 3840x2160 RGBA8, opencv_fisheye + rolling-shutter ON (2160 matrices), 240 Hz synthetic gyro, bilinear"),
    3: dict(w=7680, h=4320, pix="Luma16", lens="opencv_fisheye", digital="gopro_superview", rs=True,
            name="cfg3: 7680x4320 16-bit luma plane of YUV 4:2:2, opencv_fisheye + gopro_superview digital lens, rolling-shutter ON (4320 matrices), bilinear"),
    31: dict(w=7680, h=4320, plane=(3840, 4320), pix="Luma16", lens="opencv_fisheye", digital="gopro_superview", rs=True,
             name="cfg3 chroma: 3840x4320 16-bit U/V plane of 7680x4320 YUV 4:2:2 (source/output rects), opencv_fisheye + gopro_superview, rolling-shutter ON, bilinear"),
    4: dict(w=3840, h=2160, pix="R32f", lens="sony", digital=None, rs=True, ibis=True, mesh=True,
            name="cfg4: 3840x2160 f32 plane (GBRAPF32), sony lens + IBIS rows + 9x9 mesh correction, rolling-shutter ON, bilinear"),
}
CFG = CONFIGS[2]
# dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, one launch, from the committed `ncu --set full` captures
# (ncu flushes the caches before the launch and the output stays in L2 after it, hence traffic < algorithmic bytes)
NCU_TRAFFIC = {(2, "Bilinear"): 23568896 + 1131264}
NCU_TRAFFIC_SOURCE = "profiles/r02h_x2_filtered_fisheye_rgba8_summary.txt"
INTERP = "Bilinear"          # BASELINE configs are bilinear; --interp measures the other resamplers (side measurement, not the headline)
W, H = CFG["w"], CFG["h"]
PIX, LENS = CFG["pix"], CFG["lens"]
FRAMES_PER_STEP = 128
RING = 8                 # 8 x 33.2 MB input frames = 265 MB > 126 MB L2
N_TIMESTAMPS = 32        # distinct matrix tables
METRIC = "4K frames/sec (fisheye+RS warp)"
WORKLOAD = CFG["name"]


def select_config(n):
    global CFG, W, H, PIX, LENS, WORKLOAD, FRAMES_PER_STEP, RING, N_TIMESTAMPS
    CFG = CONFIGS[n]
    W, H, PIX, LENS, WORKLOAD = CFG["w"], CFG["h"], CFG["pix"], CFG["lens"], CFG["name"]
    if n in (3, 31): FRAMES_PER_STEP, RING, N_TIMESTAMPS = 32, 4, 8  # 66 MB planes: 4-frame ring = 265 MB
    if n == 4: FRAMES_PER_STEP, RING, N_TIMESTAMPS = 32, 8, 8


def algorithmic_bytes(p, rows, mesh_len=0, planes=1):
    """SURVEY.md §8(d): sum_planes(in_w*in_h*bpp + out_w*out_h*bpp) + rows*56 + 368 + 4*mesh_len."""
    pw, ph = CFG.get("plane", (p.width, p.height))
    return planes * 2 * pw * ph * p.bytes_per_pixel + rows * 56 + 368 + 4 * mesh_len


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        """Started before the warm-up so that nvidia-smi is already streaming when the (sub-second) timed region begins."""
        self.t0 = self.t1 = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append((time.perf_counter(), l)) for l in self.proc.stdout], daemon=True)
            self.t.start()
            t_wait = time.perf_counter()
            while not self.lines and time.perf_counter() - t_wait < 2.0:     # nvidia-smi takes a few hundred ms to print its first line
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def mark_begin(self): self.t0 = time.perf_counter()
    def mark_end(self): self.t1 = time.perf_counter()
    def samples_inside(self):
        return sum(1 for (t, _) in self.lines if self.t0 is not None and self.t0 <= t <= (self.t1 or time.perf_counter()) + 0.03)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)                                   # let the last sample of the timed region arrive
        self.proc.terminate()
        try: self.proc.wait(timeout=2)
        except Exception: pass
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = (self.t1 if self.t1 is not None else time.perf_counter()) + 0.03
        inside = [l for (t, l) in self.lines if t0 <= t <= t1]
        window = "timed region"
        if len(inside) < 2:                                # region shorter than the sampling period: use the identical extra steps run after it
            inside = [l for (t, l) in self.lines if t >= t0]
            window = "timed region + identical untimed steps right after it (region shorter than the sampling period)"
        sm, mx, reasons = [], None, set()
        for l in inside:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7: continue
            try: sm.append(float(f[0])); mx = float(f[1])
            except ValueError: continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"): reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "window": window}


def base_params():
    from gyroflow_b200 import synth
    p = synth.base_kernel_params(W, H, pixel_type=PIX, lens=LENS, digital_lens=CFG.get("digital"), fov=1.05 if CFG.get("digital") else 1.0,
                                 interpolation=INTERP)
    if CFG.get("plane"):         # a plane smaller than the frame: described by rects, like stabilization/mod.rs:209-231
        from gyroflow_b200 import abi
        pw, ph = CFG["plane"]
        bpp = p.bytes_per_pixel
        p.stride = p.output_stride = (pw * bpp + 255) // 256 * 256
        p.source_rect[:] = [0, 0, pw, ph]; p.output_rect[:] = [0, 0, pw, ph]
        p.flags |= abi.FLAG_HAS_SOURCE_RECT | abi.FLAG_HAS_OUTPUT_RECT
    return p


def make_tables(n):
    """Side-measurement configs: n matrix tables from the PRODUCT's host producer (gf_frame_transform_at_timestamp): synthetic gyro (or
    identity quaternions for config 1), and for config 4 IBIS / OIS rows from Catmull-Rom splines of synthetic sensor data
    (frame_transform.rs:227-287)."""
    import gyroflow_b200 as g
    from gyroflow_b200 import synth
    p = base_params()
    if CFG.get("identity"):
        org = sm = synth.GyroTrack(np.array([0, 10_000_000], np.int64), np.array([[1.0, 0.0, 0.0, 0.0]] * 2))
    else:
        org, sm = synth.synthetic_gyro(4.0)
    stab = synth.synthetic_camera_stab(n, W, H) if CFG.get("ibis") else None
    cp = g.ComputeParams(p, org, sm, frame_readout_time_ms=16.0 if CFG.get("rs") else 0.0, camera_stab=stab,
                         fov_scale=1.05 if CFG.get("digital") else 1.0)
    mats = np.stack([cp.at_timestamp(500.0 + i * (1000.0 / 60.0), i)[1] for i in range(n)])   # 60 fps timestamps
    p.matrix_count = mats.shape[1]
    return p, mats.astype(np.float32)


def make_mesh():
    from gyroflow_b200 import synth
    return synth.synthetic_mesh(W, H) if CFG.get("mesh") else None


DUMP_MAX_VALUES = 12 << 20      # float32 values in frames.npy (48 MB) plus at most 1 Mi float64 sample indices (8 MB): under 64 MB
DUMP_SEED = 20240917


class OutputSample:
    """--dump-outputs: the output buffers the last timed step left behind, as pixel elements (uint8 / uint16 / f16 / f32, all
    exact in float32).  A buffer's image area (rows x row_bytes, stride padding excluded) is kept whole when it fits, otherwise
    at one fixed, seeded set of element positions, the same for every run and build with the same arguments.
      frames.npy        float32 [buffers, n]: the sampled elements of each buffer, oldest frame first
      sample_index.npy  float64 [n]: their row-major element indices inside the image area"""

    def __init__(self, rows, row_bytes, pix, n_bufs):
        from gyroflow_b200 import abi
        self.rows, self.row_bytes, self.dtype = rows, row_bytes, np.dtype(abi.PIXEL_TYPES[pix][2])
        total = rows * row_bytes // self.dtype.itemsize
        n = min(total, DUMP_MAX_VALUES // n_bufs, 1 << 20)
        self.index = np.arange(total) if n == total else np.sort(np.random.default_rng(DUMP_SEED).choice(total, n, replace=False))
        self.byte_index = (self.index[:, None] * self.dtype.itemsize + np.arange(self.dtype.itemsize)).reshape(-1)
        self.samples = []

    def take(self, bufs):
        """bufs: rows x stride uint8 buffers, numpy arrays or torch tensors (gathered on their device: no full-frame copy)."""
        for b in bufs:
            idx = self.byte_index
            if not isinstance(b, np.ndarray):
                import torch
                idx = torch.from_numpy(idx).to(b.device)
            self.samples.append(b[:self.rows, :self.row_bytes].reshape(-1)[idx])

    def write(self, out_dir):
        os.makedirs(out_dir, exist_ok=True)
        host = [s if isinstance(s, np.ndarray) else s.cpu().numpy() for s in self.samples]
        np.save(os.path.join(out_dir, "frames.npy"), np.stack([np.ascontiguousarray(h).view(self.dtype) for h in host]).astype(np.float32))
        np.save(os.path.join(out_dir, "sample_index.npy"), self.index.astype(np.float64))


def last_step_slots(step, planes=1):
    """Ring slots holding the frames of `step` that are still resident after it (frame i of the run lives in slot i % RING, its
    planes in slots (i % RING) * planes + k), oldest first."""
    last = range((step + 1) * FRAMES_PER_STEP - min(RING, FRAMES_PER_STEP), (step + 1) * FRAMES_PER_STEP)
    return [(i % RING) * planes + k for i in last for k in range(planes)]


def cpu_reference_fps(p, mats, frames, threads):
    """The reference's CPU path (oracle port) on `frames` full 4K frames, all host threads."""
    from gyroflow_b200 import synth
    from tests import oracle_lib
    bw, bh = CFG.get("plane", (W, H))
    src = synth.synthetic_frame(bw, bh, PIX, stride=p.stride)
    dst = np.zeros((bh, p.output_stride), np.uint8)
    mesh = make_mesh()
    oracle_lib.undistort_image(src, dst, p, PIX, LENS, CFG.get("digital"), mats[0], mesh, threads)          # warm-up (page faults, thread start)
    t0 = time.perf_counter()
    for i in range(frames):
        rc = oracle_lib.undistort_image(src, dst, p, PIX, LENS, CFG.get("digital"), mats[i % len(mats)], mesh, threads)
        assert rc == 0
    return frames / (time.perf_counter() - t0)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tests import oracle_lib
    cores = oracle_lib.load().gf_oracle_online_cpus()
    p, mats = make_tables(4)
    from gyroflow_b200 import synth
    src = synth.synthetic_frame(W, H, PIX, stride=p.stride)
    dst = np.zeros((H, p.output_stride), np.uint8)
    mesh = make_mesh()
    step = lambda i: oracle_lib.undistort_image(src, dst, p, PIX, LENS, CFG.get("digital"), mats[i % len(mats)], mesh, cores)
    for i in range(args.warmup): step(i)
    t0 = time.perf_counter()
    for i in range(args.steps): assert step(i) == 0
    dt = time.perf_counter() - t0
    fps = args.steps / dt
    if args.dump_outputs:
        sample = OutputSample(H, W * p.bytes_per_pixel, PIX, 1)
        sample.take([dst])
        sample.write(args.dump_outputs)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frames_per_step": 1},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": "%d full 4K frames, 1 frame per step, C port of cpu_undistort.rs (Rust original unbuildable: no rustc)" % args.steps},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def make_job(duration_s):
    """The job description every rank needs: KernelParams template + the two quaternion tracks (built on rank 0, broadcast)."""
    from gyroflow_b200 import synth
    p = base_params()
    org, sm = synth.synthetic_gyro(duration_s)
    return p, org, sm


def broadcast_job(p, org, sm, rank, world, dist, torch, dev):
    """The path's only collective: one NCCL broadcast, at job start, of the KernelParams template and the quaternion tracks
    (240 Hz x clip length x 2 tracks x 40 B; SURVEY §8e)."""
    from gyroflow_b200 import render_queue, synth
    pt = render_queue.params_to_tensor(p, torch).to(dev)
    dist.broadcast(pt, src=0)
    n = torch.tensor([len(org.ts) if rank == 0 else 0], dtype=torch.int64, device=dev)
    dist.broadcast(n, src=0)
    n = int(n.item())
    ts = torch.from_numpy(np.ascontiguousarray(org.ts)).to(dev) if rank == 0 else torch.empty(n, dtype=torch.int64, device=dev)
    qs = (torch.from_numpy(np.stack([org.q, sm.q])).to(dev) if rank == 0 else torch.empty((2, n, 4), dtype=torch.float64, device=dev))
    dist.broadcast(ts, src=0); dist.broadcast(qs, src=0)
    ts = ts.cpu().numpy(); qs = qs.cpu().numpy()
    return render_queue.params_from_tensor(pt), synth.GyroTrack(ts, qs[0]), synth.GyroTrack(ts, qs[1])


def run_pipeline(args, torch, dist, g, rank, world, local, dev):
    """BASELINE config 5 literally, which at N=1 is config 2 over many frames: every frame has its own timestamp; per frame, inside the
    timed region and without a host sync, the on-device FrameTransform producer writes the 2160 x 14 matrix table and its trust verdict,
    then the warp kernel renders the frame (gf_cuda_queue_*: 4 frames in flight on 4 streams).  Frame i of the job runs on GPU i mod G."""
    from gyroflow_b200 import render_queue, synth, abi
    from tests import oracle_lib

    t_pin = g.bind_thread_to_device(local)               # NUMA: before any page-locked allocation (this library's and torch's)
    fps = 60.0
    total_frames = (max(args.warmup, 3) + args.steps + 4) * FRAMES_PER_STEP * world
    if rank == 0:
        p, org, sm = make_job(total_frames / fps + 2.0)
    else:
        p, org, sm = base_params(), None, None
    if world > 1:
        p, org, sm = broadcast_job(p, org, sm, rank, world, dist, torch, dev)
    rows = H
    cp = g.ComputeParams(p, org, sm, frame_readout_time_ms=16.0)
    st = g.stab_config(p, PIX)
    ts_of = lambda f: 500.0 + f * (1000.0 / fps)

    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    rand_frame = lambda: torch.randint(0, 256, (H, p.stride), dtype=torch.uint8, device=dev, generator=gen)
    frames_in = [rand_frame() for _ in range(RING)]
    frames_out = [torch.zeros((H, p.output_stride), dtype=torch.uint8, device=dev) for _ in range(RING)]
    dbufs = [g.Buffers(g.BufferDescription((W, H, p.stride), a.data_ptr(), length=a.numel()),
                       g.BufferDescription((W, H, p.output_stride), b.data_ptr(), length=b.numel())) for a, b in zip(frames_in, frames_out)]
    DEPTH_DEV = max(1, min(args.depth, RING))          # frames in flight on the device-resident path (distinct ring buffers)
    q = g.RenderQueue(cp, st, LENS, None, dbufs[0].input, dbufs[0].output, device=local, depth=DEPTH_DEV, pin_numa=True, checksum=False)
    tstream = torch.cuda.Stream(device=dev)

    def step(s):                                          # FRAMES_PER_STEP frames of this rank: global frames (s * FPS + j) * world + rank
        for j in range(FRAMES_PER_STEP):
            f = (s * FRAMES_PER_STEP + j) * world + rank
            if q.in_flight == DEPTH_DEV: q.wait()
            q.submit(f, ts_of(f), dbufs[(s * FRAMES_PER_STEP + j) % RING])

    clocks = ClockSampler(local); clocks.start()
    W_STEPS = max(args.warmup, 3)
    for s in range(W_STEPS): step(s)
    q.drain(); torch.cuda.synchronize()
    if world > 1: dist.barrier()
    l0 = q.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    clocks.mark_begin()
    e0.record(tstream)                                    # device idle: the event's timestamp is the start of the timed region
    for s in range(args.steps): step(W_STEPS + s)
    q.drain()                                             # every frame of every step has finished on the device
    e1.record(tstream)
    torch.cuda.synchronize()
    clocks.mark_end()
    sample = None
    if args.dump_outputs and rank == 0:                   # before any further step overwrites the ring
        sample = OutputSample(H, W * p.bytes_per_pixel, PIX, min(RING, FRAMES_PER_STEP))
        sample.take([frames_out[k] for k in last_step_slots(W_STEPS + args.steps - 1)])
    if world > 1: dist.barrier()
    total_ms = e0.elapsed_time(e1)
    launches = q.launch_count - l0
    if clocks.proc and clocks.samples_inside() < 3:
        t_extra = time.perf_counter()
        while time.perf_counter() - t_extra < 0.3:
            step(W_STEPS); q.drain()
    clk = clocks.stop()
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    fps_value = world * FRAMES_PER_STEP / (ms_per_step / 1e3)

    # ---- verification pass (untimed): a few frames of the same job with device-side checksums, gathered in frame order -------------
    # inputs with a rank-independent seed (rank 0 re-renders them on the CPU below), one input / output buffer per frame in flight
    vgen = torch.Generator(device=dev); vgen.manual_seed(999)
    vin = [torch.randint(0, 256, (H, p.stride), dtype=torch.uint8, device=dev, generator=vgen) for _ in range(2)]
    vout = [torch.zeros((H, p.output_stride), dtype=torch.uint8, device=dev) for _ in range(2)]
    vbufs = [g.Buffers(g.BufferDescription((W, H, p.stride), a.data_ptr(), length=a.numel()),
                       g.BufferDescription((W, H, p.output_stride), b.data_ptr(), length=b.numel())) for a, b in zip(vin, vout)]
    qv = g.RenderQueue(cp, st, LENS, None, vbufs[0].input, vbufs[0].output, device=local, depth=2, pin_numa=False, checksum=True)
    n_check = 8
    mine = render_queue.shard_frames(n_check, world, rank)
    sums = qv.render(mine, ts_of, lambda f: vbufs[(f // world) % 2]) if mine else {}
    qv.close()
    if world > 1: sums = render_queue.gather_results(sums, dist, torch, dev)

    # ---- the kernel alone, one stream (roofline), and the round-1 style numbers on recycled precomputed tables ---------------------
    dg = g.DeviceGyro(cp, device=local)
    n_tab = N_TIMESTAMPS
    tabs = torch.zeros((n_tab, rows, 14), dtype=torch.float32, device=dev)
    flags = torch.zeros(n_tab, dtype=torch.int32, device=dev)
    kps = []
    for i in range(n_tab):
        kp, r = dg.frame_transform(ts_of(i * world + rank), tabs[i].data_ptr(), rows, frame=i, stream=tstream.cuda_stream,
                                   table_flags_dev=flags[i:].data_ptr())
        kp = g.get_frame_transform_at(st, cp, dbufs[0], kp)
        kps.append(kp)
    tstream.synchronize()
    assert int(flags.abs().sum().item()) == 0, "the producer's tables are tame and IBIS-free: the trusted path must run"
    ctx = g.CudaWrapper.new(kps[0], PIX, LENS, None, dbufs[0], device=local)

    def kernel_loop(n_steps, with_flags):
        evs = []
        for s in range(n_steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(tstream)
            for j in range(FRAMES_PER_STEP):
                i = s * FRAMES_PER_STEP + j
                ctx.undistort_image_dev(dbufs[i % RING], kps[i % n_tab], tabs[i % n_tab].data_ptr(), rows, stream=tstream.cuda_stream,
                                        table_flags_dev=flags[(i % n_tab):].data_ptr() if with_flags else 0)
            b.record(tstream)
            evs.append((a, b))
        tstream.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / n_steps

    side_steps = max(3, min(args.steps, 10))
    kernel_loop(3, True)
    ms_trusted = kernel_loop(side_steps, True)
    kernel_loop(2, False)
    ms_unval = kernel_loop(side_steps, False)
    tt = torch.tensor([ms_trusted, ms_unval], dtype=torch.float64, device=dev)
    if world > 1: dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms_trusted, ms_unval = float(tt[0].item()), float(tt[1].item())
    launch_ms = ms_trusted / FRAMES_PER_STEP

    # ---- e2e: the same queue with HOST buffers: per frame  producer kernel | H2D frame | warp | D2H frame  -------------------------
    e2e = None
    if not args.no_e2e:
        DEPTH = args.e2e_depth
        hin = [rand_frame().cpu().pin_memory() for _ in range(DEPTH)]
        hout = [torch.zeros((H, p.output_stride), dtype=torch.uint8).pin_memory() for _ in range(DEPTH)]
        hb = [g.Buffers(g.BufferDescription((W, H, p.stride), hin[i].numpy()), g.BufferDescription((W, H, p.output_stride), hout[i].numpy())) for i in range(DEPTH)]
        qh = g.RenderQueue(cp, st, LENS, None, hb[0].input, hb[0].output, device=local, depth=DEPTH, pin_numa=True, checksum=False)
        e2e_steps = max(1, min(args.steps, 3))
        e2e_frames = e2e_steps * FRAMES_PER_STEP

        def host_run(n, base):
            for k in range(n):
                f = (base + k) * world + rank
                if qh.in_flight == DEPTH: qh.wait()            # the slot's previous result has landed in host memory
                qh.submit(f, ts_of(f), hb[k % DEPTH])
            qh.drain()
        host_run(2 * DEPTH + 8, 0)
        if world > 1: dist.barrier()
        t0 = time.perf_counter()
        host_run(e2e_frames, 64)
        e2e_dt = time.perf_counter() - t0
        qh.close()
        # the strictly sequential reference-shaped call (process_pixels: host tables, H2D -> kernel -> D2H -> sync), pinned and pageable
        kp0, m0, _, _ = cp.at_timestamp(ts_of(rank))
        kp0 = g.get_frame_transform_at(st, cp, hb[0], kp0)
        itm = g.FrameTransform(matrices=m0, kernel_params=kp0)
        hctx = g.CudaWrapper.new(kp0, PIX, LENS, None, hb[0], device=local)
        for _ in range(3): hctx.undistort_image(hb[0], itm)
        t0 = time.perf_counter()
        for _ in range(32): hctx.undistort_image(hb[0], itm)
        sync_fps = 32 / (time.perf_counter() - t0)
        pin_a, pin_b = np.array(hin[0].numpy(), copy=True), np.zeros((H, p.output_stride), np.uint8)      # ordinary (pageable) Vec<u8>-like memory
        pb = g.Buffers(g.BufferDescription((W, H, p.stride), pin_a), g.BufferDescription((W, H, p.output_stride), pin_b))
        for _ in range(2): hctx.undistort_image(pb, itm)
        t0 = time.perf_counter()
        for _ in range(16): hctx.undistort_image(pb, itm)
        pageable_fps = 16 / (time.perf_counter() - t0)
        g.host_register(pin_a); g.host_register(pin_b)          # the same ordinary buffers, page-locked in place once (gf_cuda_host_register)
        for _ in range(2): hctx.undistort_image(pb, itm)
        t0 = time.perf_counter()
        for _ in range(32): hctx.undistort_image(pb, itm)
        registered_fps = 32 / (time.perf_counter() - t0)
        g.host_unregister(pin_a); g.host_unregister(pin_b)
        hctx.close()
        te = torch.tensor([e2e_dt, 1.0 / sync_fps, 1.0 / pageable_fps, 1.0 / registered_fps], dtype=torch.float64, device=dev)
        if world > 1: dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_fps = world * e2e_frames / float(te[0].item())
        h2d_frame = int(hin[0].numel() + 368)                 # frame + KernelParams (kernel argument); the matrix table is produced on the device
        d2h_frame = int(W * p.bytes_per_pixel * H)
        e2e = {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d_frame * FRAMES_PER_STEP * world, "d2h_bytes_per_step": d2h_frame * FRAMES_PER_STEP * world,
               "h2d_bytes_per_frame": h2d_frame, "d2h_bytes_per_frame": d2h_frame, "frames_per_step": FRAMES_PER_STEP * world, "steps": e2e_steps,
               "h2d_GBps_per_gpu": e2e_fps / world * h2d_frame / 1e9, "d2h_GBps_per_gpu": e2e_fps / world * d2h_frame / 1e9,
               "pipeline_depth": DEPTH, "numa_cpus_bound": t_pin,
               "sync_call_value": world / float(te[1].item()), "sync_call_pageable_value": world / float(te[2].item()),
               "sync_call_registered_value": world / float(te[3].item()),
               "note": "value: gf_cuda_queue with page-locked HOST frames, %d in flight, per frame: on-device FrameTransform producer, H2D, warp, D2H (wall clock, %d frames); "
                       "sync_call_value: strictly sequential gf_cuda_undistort_image with host tables (what process_pixels does), pinned; "
                       "sync_call_pageable_value: the same with ordinary pageable buffers (BufferSource::Cpu hands a plain &mut [u8]); "
                       "sync_call_registered_value: those ordinary buffers after gf_cuda_host_register (page-locked in place once)" % (DEPTH, e2e_frames)}

    if rank == 0:
        peaks = {}
        try: peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception: pass
        peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        abytes = algorithmic_bytes(p, rows)
        achieved = abytes / (launch_ms / 1e3) / 1e9
        cpu = None
        if not args.no_cpu_baseline:
            cores = oracle_lib.load().gf_oracle_online_cpus()
            # 4 full 4K frames of this job on the host cores: timed (cpu_baseline) AND compared with the pipeline's per-frame checksums
            tab = torch.zeros((rows, 14), dtype=torch.float32, device=dev)
            dst = np.zeros((H, p.output_stride), np.uint8)
            checked, cpu_t = [], 0.0
            for f in range(min(4, n_check)):
                src = vin[(f // world) % 2].cpu().numpy()                    # the input the verification pass rendered frame f from (same on every rank)
                kp, r = dg.frame_transform(ts_of(f), tab.data_ptr(), rows, frame=f)
                kp = g.get_frame_transform_at(st, cp, dbufs[0], kp)
                m = tab.cpu().numpy()
                if f == 0: oracle_lib.undistort_image(src, dst, kp, PIX, LENS, None, m, None, cores)      # warm-up (page faults, thread start)
                t0 = time.perf_counter()
                assert oracle_lib.undistort_image(src, dst, kp, PIX, LENS, None, m, None, cores) == 0
                cpu_t += time.perf_counter() - t0
                ok = render_queue.checksum_host(dst) == sums[f]
                checked.append(bool(ok))
            assert all(checked), "pipeline frames differ from the CPU oracle: %r" % (checked,)
            cpu = {"value": len(checked) / cpu_t, "unit": "frames/s", "cores": cores, "kind": "port",
                   "sample": "%d full 4K frames of the same job (C port of cpu_undistort.rs, row-parallel over all host threads); each one's output checksum "
                             "equals the checksum the GPU pipeline produced for that frame (frames 0..%d, gathered in frame order over %d rank(s))" % (len(checked), len(checked) - 1, world),
                   "frames_checked_against_gpu": len(checked)}
        out = {
            "metric": METRIC, "value": fps_value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": W_STEPS,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frame_bytes_in": int(H * p.stride), "frames_per_step": FRAMES_PER_STEP * world, "frames_per_step_per_gpu": FRAMES_PER_STEP,
                       "pipeline": "cfg5 shape: every frame its own timestamp; per frame inside the timed region: on-device FrameTransform producer (2160 x 14 table + trust verdict) -> warp; "
                                   "%d frames in flight per GPU; frame i on GPU i mod %d" % (DEPTH_DEV, world),
                       "l2_policy": "inputs larger than L2: %d-frame ring of %.1f MB inputs (%d MB); every frame a fresh matrix table" % (RING, H * p.stride / 1e6, RING * H * p.stride // 1000000),
                       "parallelism": "frame-sharded x%d, one NCCL broadcast of KernelParams + quaternion tracks at job start" % world},
            "clocks": clk, "gpu_launches": launches,
            "value_trusted_precomputed": world * FRAMES_PER_STEP / (ms_trusted / 1e3),
            "value_unvalidated": world * FRAMES_PER_STEP / (ms_unval / 1e3),
            "value_notes": "value = the per-frame pipeline above (producer + warp kernels, multi-stream, CUDA events around the whole region); value_trusted_precomputed = warp kernel only on "
                           "%d recycled device tables with verdict words (round 1's headline shape); value_unvalidated = the same without verdict words (guarded code path)" % n_tab,
            "e2e": e2e,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": NCU_TRAFFIC.get((args.config, INTERP)),
                         "traffic_source": NCU_TRAFFIC_SOURCE if (args.config, INTERP) in NCU_TRAFFIC else None,
                         "algorithmic_bytes_per_launch": abytes, "launch_ms": launch_ms, "peak_source": peak_src,
                         # SURVEY §8(d): the read-only variant (input planes + tables; north_star says "HBM-read roofline") and the nominal 8 TB/s
                         "read_only": {"bytes_per_launch": abytes - int(W * p.bytes_per_pixel * H), "achieved": (abytes - int(W * p.bytes_per_pixel * H)) / (launch_ms / 1e3) / 1e9,
                                       "frac": (abytes - int(W * p.bytes_per_pixel * H)) / (launch_ms / 1e3) / 1e9 / peak},
                         "frac_of_nominal_8000": achieved / 8000.0,
                         "pipeline_achieved": abytes * fps_value / world / 1e9, "pipeline_frac": abytes * fps_value / world / 1e9 / peak,
                         "kernel": "warp_kernel_x2 (trusted path, filtered pre-pass: main + tail launch), timed alone on one stream with CUDA events: %d frames per step" % FRAMES_PER_STEP,
                         "note": "kernel is FP32-issue bound in bit-exact (-fmad=false) mode, not HBM bound; traffic is the DRAM bytes of ONE cold launch under ncu (output stays in L2), not a steady-state figure; see DESIGN.md"},
            "cpu_baseline": cpu,
        }
        if sample: sample.write(args.dump_outputs)
        print(json.dumps(out))
    ctx.close(); dg.close(); q.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-depth", type=int, default=5, help="frames in flight on the host-buffer path")
    ap.add_argument("--depth", type=int, default=4, help="frames in flight on the device-resident path (<= 8)")
    ap.add_argument("--legacy", action="store_true", help="round-1 measurement shape (recycled precomputed tables) for the default config too")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--lens", default=None, help="override the config's lens model (side measurement), e.g. sony, opencv_standard")
    ap.add_argument("--digital", default=None, help="override the config's digital lens (side measurement), e.g. gopro_superview, digital_stretch, gopro_warp")
    ap.add_argument("--planes", type=int, default=1, help="planes of this geometry per frame, rendered by one gf_cuda_undistort_planes_dev call (side measurement)")
    ap.add_argument("--interp", default="Bilinear", help="Bilinear (BASELINE), Bicubic, Lanczos4, 'EWA: Robidoux', ... (side measurement)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frames the last timed step rendered (rank 0's; a fixed seeded sample) to DIR/frames.npy + DIR/sample_index.npy")
    args = ap.parse_args()
    select_config(args.config)
    global INTERP, LENS, WORKLOAD
    INTERP = args.interp
    if args.lens:
        LENS = args.lens; WORKLOAD = WORKLOAD.replace(CFG["lens"], args.lens)
    if args.digital:
        CFG["digital"] = args.digital; WORKLOAD = WORKLOAD.replace(LENS, LENS + " + " + args.digital + " digital lens", 1)
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import gyroflow_b200 as g
    from gyroflow_b200 import synth

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node %d" % args.gpus
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    lib = g.load_library()
    assert lib.gf_cuda_device_count() > local, "no CUDA device for this rank (there is no CPU fallback)"

    if args.config == 2 and not args.lens and not args.digital and args.planes == 1 and INTERP == "Bilinear" and not args.legacy:
        return run_pipeline(args, torch, dist, g, rank, world, local, dev)

    # ---- tables: rank 0 builds them, NCCL broadcasts them (the only collective of the path) -------------------
    from gyroflow_b200 import render_queue
    p, mats_np = make_tables(N_TIMESTAMPS) if rank == 0 else (base_params(), np.zeros((0, 0, 0), np.float32))
    rows = H if CFG.get("rs") else 1
    mesh_np = make_mesh()
    mesh_dev = torch.from_numpy(mesh_np).to(dev) if mesh_np is not None else None
    if world > 1:
        p, mats = render_queue.broadcast_tables(p, mats_np, dist, torch, dev)      # NCCL: KernelParams + all matrix tables, once
    else:
        mats = torch.from_numpy(mats_np).to(dev)
    assert p.matrix_count == rows and tuple(mats.shape) == (N_TIMESTAMPS, rows, 14)

    # ---- device-resident frames -----------------------------------------------------------------------------
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    def rand_frame(pin=False):
        if PIX in ("R32f", "RGBAf"):     # finite floats in [0, 1)
            t = torch.rand((H, p.stride // 4), dtype=torch.float32, device=dev, generator=gen).view(torch.uint8).reshape(H, p.stride)
        else:
            t = torch.randint(0, 256, (H, p.stride), dtype=torch.uint8, device=dev, generator=gen)
        return t
    NPL = max(1, args.planes)
    BW, BH = CFG.get("plane", (W, H))                 # buffer size of one plane
    frames_in = [rand_frame() for _ in range(RING * NPL)]
    frames_out = [torch.zeros((H, p.output_stride), dtype=torch.uint8, device=dev) for _ in range(RING * NPL)]
    def dbufs(i):
        a, b = frames_in[i % (RING * NPL)], frames_out[i % (RING * NPL)]
        return g.Buffers(g.BufferDescription((BW, BH, p.stride), a.data_ptr(), length=a.numel()),
                         g.BufferDescription((BW, BH, p.output_stride), b.data_ptr(), length=b.numel()))
    ctx = g.CudaWrapper.new(p, PIX, LENS, CFG.get("digital"), dbufs(0), device=local)
    # a real (non-default) stream: kernels, CUDA events and the timed region all live on it
    tstream = torch.cuda.Stream(device=dev)
    stream = tstream.cuda_stream
    assert stream != 0
    all_bufs = [dbufs(i) for i in range(RING * NPL)]
    plane_params = []
    for k in range(NPL):
        q = p.copy(); q.plane_index = k; plane_params.append(q)
    # one verdict word per table, written by the asynchronous scan kernel once, outside the timed region (recycled tables)
    tflags = torch.zeros(N_TIMESTAMPS, dtype=torch.int32, device=dev)
    for i in range(N_TIMESTAMPS): g.scan_tables_dev(mats[i].data_ptr(), rows, tflags[i:].data_ptr(), stream=stream)
    tstream.synchronize()

    def step(s):
        for j in range(FRAMES_PER_STEP):
            i = s * FRAMES_PER_STEP + j
            if NPL == 1:
                ctx.undistort_image_dev(all_bufs[i % RING], p, mats[i % N_TIMESTAMPS].data_ptr(), rows,
                                        mesh_dev.data_ptr() if mesh_dev is not None else 0, mesh_dev.numel() if mesh_dev is not None else 0, stream=stream,
                                        table_flags_dev=tflags[(i % N_TIMESTAMPS):].data_ptr())
            else:       # one multi-plane frame: coordinates once, NPL sampling passes
                b0 = (i % RING) * NPL
                ctx.undistort_planes_dev(all_bufs[b0:b0 + NPL], plane_params, mats[i % N_TIMESTAMPS].data_ptr(), rows,
                                         mesh_dev.data_ptr() if mesh_dev is not None else 0, mesh_dev.numel() if mesh_dev is not None else 0, stream=stream,
                                         table_flags_dev=tflags[(i % N_TIMESTAMPS):].data_ptr())

    clocks = ClockSampler(local); clocks.start()
    torch.cuda.synchronize()
    for s in range(max(args.warmup, 3)):              # never fewer than 3 warm-up steps
        step(s)
    torch.cuda.synchronize()
    if world > 1: dist.barrier()
    l0 = ctx.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    clocks.mark_begin()
    for s in range(args.steps):
        ev[s][0].record(tstream)
        step(s)
        ev[s][1].record(tstream)
    torch.cuda.synchronize()
    clocks.mark_end()
    sample = None
    if args.dump_outputs and rank == 0:                   # before any further step overwrites the ring
        slots = last_step_slots(args.steps - 1, NPL)
        sample = OutputSample(BH, BW * p.bytes_per_pixel, PIX, len(slots))
        sample.take([frames_out[k] for k in slots])
    if world > 1: dist.barrier()
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = ctx.launch_count - l0
    if clocks.proc and clocks.samples_inside() < 3:   # a very short timed region: keep the same load running (untimed) until the sampler has seen it
        t_extra = time.perf_counter()
        while time.perf_counter() - t_extra < 0.3:
            step(0); torch.cuda.synchronize()
    clk = clocks.stop()
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    fps = world * FRAMES_PER_STEP / (ms_per_step / 1e3)

    # ---- e2e: host (pinned) buffers through the C ABI, copies inside the timed region ---------------------------
    # (a) the reference-facing synchronous call gf_cuda_undistort_image: H2D -> kernel -> D2H -> sync, one frame at a time
    # (b) the same work pipelined: DEPTH contexts round-robin through gf_cuda_undistort_image_async + gf_cuda_synchronize,
    #     so frame i+1's upload overlaps frame i's kernel and frame i-1's download.  (b) is the reported e2e value.
    DEPTH = 3
    hin = [rand_frame().cpu().pin_memory() for _ in range(DEPTH)]
    hout = [torch.zeros((H, p.output_stride), dtype=torch.uint8).pin_memory() for _ in range(DEPTH)]
    def hbufs(i):
        a, b = hin[i % DEPTH].numpy(), hout[i % DEPTH].numpy()
        return g.Buffers(g.BufferDescription((BW, BH, p.stride), a), g.BufferDescription((BW, BH, p.output_stride), b))
    hb = [hbufs(i) for i in range(DEPTH)]
    hctx = [g.CudaWrapper.new(p, PIX, LENS, CFG.get("digital"), hb[i], device=local) for i in range(DEPTH)]
    mats_host = mats.cpu().numpy()
    itms = [g.FrameTransform(matrices=mats_host[i % N_TIMESTAMPS], kernel_params=p, mesh_data=mesh_np if mesh_np is not None else np.zeros(0, np.float32))
            for i in range(N_TIMESTAMPS)]
    # an e2e step = the same FRAMES_PER_STEP frames as a device-resident step (--no-e2e: a token 24 frames)
    e2e_steps = 0 if args.no_e2e else max(1, min(args.steps, 3))
    e2e_frames = 24 if args.no_e2e else e2e_steps * FRAMES_PER_STEP
    for i in range(3): hctx[0].undistort_image(hb[0], itms[i % N_TIMESTAMPS])
    if world > 1: dist.barrier()
    t0 = time.perf_counter()
    for i in range(32): hctx[0].undistort_image(hb[0], itms[i % N_TIMESTAMPS])
    sync_fps = 32 / (time.perf_counter() - t0)
    for i in range(DEPTH): hctx[i].undistort_image_async(hb[i], itms[i]); 
    for c in hctx: c.synchronize()
    if world > 1: dist.barrier()
    t0 = time.perf_counter()
    for i in range(e2e_frames):
        c = hctx[i % DEPTH]
        c.synchronize()                                   # the slot's previous frame (i - DEPTH) has fully landed in host memory
        c.undistort_image_async(hb[i % DEPTH], itms[i % N_TIMESTAMPS])
    for c in hctx: c.synchronize()
    e2e_dt = time.perf_counter() - t0
    te = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
    if world > 1: dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_fps = world * e2e_frames / float(te.item())
    h2d_frame = int(hin[0].numel() + rows * 56 + 368 + (mesh_np.size * 4 if mesh_np is not None else 0))    # frame + matrices + KernelParams (+ mesh)
    d2h_frame = int(BW * p.bytes_per_pixel * BH)
    h2d, d2h = h2d_frame * FRAMES_PER_STEP * world, d2h_frame * FRAMES_PER_STEP * world

    if rank == 0:
        peaks = {}
        try: peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception: pass
        peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        abytes = algorithmic_bytes(p, rows, mesh_np.size if mesh_np is not None else 0, NPL)
        launch_ms = total_ms / max(args.steps * FRAMES_PER_STEP, 1)      # per frame: one launch for the headline config; coordinate + sampling passes otherwise
        achieved = abytes / (launch_ms / 1e3) / 1e9
        cpu = None
        if not args.no_cpu_baseline:
            from tests import oracle_lib
            cores = oracle_lib.load().gf_oracle_online_cpus()
            cfps = cpu_reference_fps(p, mats_host, 4 if args.config != 3 else 2, cores)
            cpu = {"value": cfps, "unit": "frames/s", "cores": cores, "kind": "port",
                   "sample": "4 full 4K frames of the same workload (C port of cpu_undistort.rs, row-parallel over all host threads)"}
        out = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD if INTERP == "Bilinear" else WORKLOAD.replace("bilinear", INTERP), "frame_bytes_in": int(H * p.stride), "frames_per_step": FRAMES_PER_STEP, "frames_per_step_per_gpu": FRAMES_PER_STEP,
                       "l2_policy": "inputs larger than L2: %d-frame ring of %.1f MB inputs (%d MB) + %d distinct matrix tables" % (RING, H * p.stride / 1e6, RING * H * p.stride // 1000000, N_TIMESTAMPS),
                       "planes_per_frame": NPL,
                       "parallelism": "frame-sharded x%d, NCCL broadcast of tables only" % world},
            "clocks": clk, "gpu_launches": launches,
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "h2d_bytes_per_frame": h2d_frame, "d2h_bytes_per_frame": d2h_frame, "frames_per_step": FRAMES_PER_STEP * world, "steps": e2e_steps,
                    "sync_call_value": sync_fps * world,
                    "note": "pinned host frame + tables H2D, kernel, D2H per frame; value = %d-deep pipeline over gf_cuda_undistort_image_async, sync_call_value = strictly sequential gf_cuda_undistort_image; %d frames, wall clock" % (DEPTH, e2e_frames)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": NCU_TRAFFIC.get((args.config, INTERP)),
                         "traffic_source": NCU_TRAFFIC_SOURCE if (args.config, INTERP) in NCU_TRAFFIC else None,
                         "algorithmic_bytes_per_launch": abytes, "launch_ms": launch_ms, "peak_source": peak_src,
                         "note": "kernel is FP32-issue bound in bit-exact (-fmad=false) mode; see DESIGN.md"},
            "cpu_baseline": cpu,
        }
        if sample: sample.write(args.dump_outputs)
        print(json.dumps(out))
    for c in hctx: c.close()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
