"""Whole decoder frames through the render queue (gf_frame_layout, gf_background_for_plane, gf_cuda_queue_*_frame).

The reference renders a decoded frame plane by plane (rendering/mod.rs:483-548, :563-651): each plane gets its own pixel type, size,
`yuvi` list, value limit, background converted with PixelType::from_rgb_color (pixel_formats.rs:23-48), plane_index and the per-frame
FILL_WITH_BACKGROUND flag.  The CPU tests check the format table and the colour conversion against transcriptions written here from the
Rust text; the GPU tests render frames through the queue and compare every plane byte for byte with the oracle, which renders each plane
alone from the table read back through DeviceGyro and KernelParams built by the test itself."""
import ctypes as C

import numpy as np
import pytest

import gyroflow_b200 as g
from gyroflow_b200 import abi, render_queue, synth

# ---- literal transcription of rendering/mod.rs:563-651: format -> (log2 chroma w, log2 chroma h, [(type, $ind, $yuvi, $max_val)]) ----
_NV = lambda t1, t2, uv, m: [(t1, 0, [0], m), (t2, 1, uv, m)]
_Y3 = lambda t, m: [(t, 0, [0], m), (t, 1, [1], m), (t, 2, [2], m)]
_Y4 = lambda t, m: _Y3(t, m) + [(t, 3, [3], m)]
TABLE = {
    "NV12": (1, 1, _NV("Luma8", "UV8", [1, 2], 255.0)),
    "NV21": (1, 1, _NV("Luma8", "UV8", [2, 1], 255.0)),
    "P010LE": (1, 1, _NV("Luma16", "UV16", [1, 2], 65535.0)), "P016LE": (1, 1, _NV("Luma16", "UV16", [1, 2], 65535.0)),
    "P210LE": (1, 0, _NV("Luma16", "UV16", [1, 2], 65535.0)), "P216LE": (1, 0, _NV("Luma16", "UV16", [1, 2], 65535.0)),
    "P410LE": (0, 0, _NV("Luma16", "UV16", [1, 2], 65535.0)), "P416LE": (0, 0, _NV("Luma16", "UV16", [1, 2], 65535.0)),
    "YUV420P": (1, 1, _Y3("Luma8", 255.0)), "YUVJ420P": (1, 1, _Y3("Luma8", 255.0)),
    "YUV420P10LE": (1, 1, _Y3("Luma16", 1023.0)), "YUV420P12LE": (1, 1, _Y3("Luma16", 4095.0)),
    "YUV420P14LE": (1, 1, _Y3("Luma16", 16383.0)), "YUV420P16LE": (1, 1, _Y3("Luma16", 65535.0)),
    "YUV422P10LE": (1, 0, _Y3("Luma16", 1023.0)), "YUV422P12LE": (1, 0, _Y3("Luma16", 4095.0)),
    "YUV422P14LE": (1, 0, _Y3("Luma16", 16383.0)), "YUV422P16LE": (1, 0, _Y3("Luma16", 65535.0)),
    "YUV444P10LE": (0, 0, _Y3("Luma16", 1023.0)), "YUV444P12LE": (0, 0, _Y3("Luma16", 4095.0)),
    "YUV444P14LE": (0, 0, _Y3("Luma16", 16383.0)), "YUV444P16LE": (0, 0, _Y3("Luma16", 65535.0)),
    "YUVA444P10LE": (0, 0, _Y4("Luma16", 1023.0)), "YUVA444P12LE": (0, 0, _Y4("Luma16", 4095.0)), "YUVA444P16LE": (0, 0, _Y4("Luma16", 65535.0)),
    "GBRAPF32LE": (0, 0, [("R32f", 0, [2], 255.0), ("R32f", 0, [0], 255.0), ("R32f", 0, [1], 255.0), ("R32f", 0, [3], 255.0)]),
    "GBRPF32LE": (0, 0, [("R32f", 0, [2], 255.0), ("R32f", 0, [0], 255.0), ("R32f", 0, [1], 255.0)]),
    "AYUV64LE": (0, 0, [("AYUV16", 0, [3, 0, 1, 2], 65535.0)]),
    "RGB24": (0, 0, [("RGB8", 0, [], 255.0)]), "RGBA": (0, 0, [("RGBA8", 0, [], 255.0)]),
    "RGB48BE": (0, 0, [("RGB16", 0, [], 65535.0)]), "RGBA64BE": (0, 0, [("RGBA16", 0, [], 65535.0)]),
}


def plane_sizes(fmt, w, h):
    """ffmpeg's plane_width / plane_height for plane $ind: planes 1 and 2 are -((-w) >> log2_chroma_w) wide, the rest full size."""
    cw, ch, planes = TABLE[fmt]
    return [((-((-w) >> cw), -((-h) >> ch)) if ind in (1, 2) else (w, h)) for _, ind, _, _ in planes]


# ---- numpy-f32 restatement of rgb_to_yuv / from_rgb_color (pixel_formats.rs:23-48, :77-298) ------------------------------------
F = np.float32


def np_rgb_to_yuv(v, is_limited):
    v = [F(x) for x in v]
    KR, KB = F(0.2126), F(0.0722)
    KG = F(1.0) - KR - KB
    US = F(1.0) / (F(2.0) - F(2.0) * KB)
    VS = F(1.0) / (F(2.0) - F(2.0) * KR)
    cl = lambda x: np.fmin(np.fmax(x, F(0.0)), F(1.0))
    ret = [cl(KR * v[0] + KG * v[1] + KB * v[2]),
           cl((-KR * US) * v[0] + (-KG * US) * v[1] + ((F(1.0) - KB) * US) * v[2] + F(0.5)),
           cl(((F(1.0) - KR) * VS) * v[0] + (-KG * VS) * v[1] + (-KB * VS) * v[2] + F(0.5)),
           cl(v[3])]
    if is_limited:
        ret[0] = (F(16.0) / F(255.0)) + (ret[0] * ((F(235.0) - F(16.0)) / F(255.0)))
        ret[1] = (F(16.0) / F(255.0)) + (ret[1] * ((F(240.0) - F(16.0)) / F(255.0)))
        ret[2] = (F(16.0) / F(255.0)) + (ret[2] * ((F(240.0) - F(16.0)) / F(255.0)))
    return ret


def np_from_rgb_color(pix, v, ind, is_limited):
    v = [F(x) for x in v]
    z = F(0.0)
    if pix in ("Luma8", "Luma16"):
        return np.array([np_rgb_to_yuv(v, is_limited)[ind[0]], z, z, z], np.float32)
    if pix in ("UV8", "UV16"):
        y = np_rgb_to_yuv(v, is_limited)
        return np.array([y[ind[0]], y[ind[1]], z, z], np.float32)
    if pix == "AYUV16":
        y = np_rgb_to_yuv(v, is_limited)
        return np.array([y[ind[0]], y[ind[1]], y[ind[2]], y[ind[3]]], np.float32)
    if pix == "R32f":
        return np.array([v[ind[0]], z, z, z], np.float32)
    if pix == "BGRA8":
        return np.array([v[2], v[1], v[0], v[3]], np.float32)
    return np.array(v, np.float32)


# ---- CPU tests --------------------------------------------------------------------------------------------------------------------

def test_format_table_matches_the_reference():
    assert sorted(TABLE) == sorted(abi.FRAME_FORMATS)
    for fmt in TABLE:
        for w, h in ((3840, 2160), (641, 361), (1, 1), (7, 4), (1919, 1081)):
            got = g.frame_layout(fmt, w, h)
            want = TABLE[fmt][2]
            assert len(got) == len(want), fmt
            for pl, (t, _, yuvi, m), (pw, ph) in zip(got, want, plane_sizes(fmt, w, h)):
                assert (pl["pixel_type"], pl["width"], pl["height"], list(pl["ind"]), pl["max_value"]) == (t, pw, ph, yuvi, m), (fmt, w, h)
    nv12 = g.frame_layout("NV12", 641, 361)
    assert [(p["width"], p["height"]) for p in nv12] == [(641, 361), (321, 181)]          # odd sizes round up
    assert [(p["width"], p["height"]) for p in g.frame_layout("P210LE", 641, 361)] == [(641, 361), (321, 361)]
    assert [p["ind"] for p in g.frame_layout("GBRAPF32LE", 8, 8)] == [(2,), (0,), (1,), (3,)]
    lib = g.load_library()
    out = (abi.PlaneSpec * 4)(); n = C.c_size_t()
    assert lib.gf_frame_layout(len(TABLE), 64, 64, out, C.byref(n)) == -1
    assert lib.gf_frame_layout(0, 0, 64, out, C.byref(n)) == -1
    assert lib.gf_abi_struct_size(9) == C.sizeof(abi.PlaneSpec)


def test_background_for_plane_is_bit_equal_to_the_rust_restatement():
    rng = np.random.default_rng(11)
    colours = [(0, 0, 0, 0), (1, 1, 1, 1), (1, 0, 0, 1), (0, 1, 0, 0.5), (0, 0, 1, 0), (0.5, 0.5, 0.5, 1)]
    colours += [tuple(rng.uniform(-0.25, 1.25, 4).astype(np.float32)) for _ in range(200)]    # outside 0..1 too: the clamps
    combos = {(t, tuple(yuvi)) for _, _, planes in TABLE.values() for t, _, yuvi, _ in planes}
    combos |= {("BGRA8", ()), ("RGBAf", ()), ("RGBAf16", ())}
    for pix, ind in sorted(combos):
        for c in colours:
            for limited in (False, True):
                got = g.background_for_plane(pix, c, ind, limited)
                want = np_from_rgb_color(pix, c, ind, limited)
                assert got.tobytes() == want.tobytes(), (pix, ind, c, limited, got, want)
    # black: neutral chroma (0.5) in full range, 16/255 luma and 128/255 chroma in limited range
    assert g.background_for_plane("UV8", (0, 0, 0, 0), (1, 2), False)[:2].tolist() == [0.5, 0.5]
    assert g.background_for_plane("Luma8", (0, 0, 0, 0), (0,), True)[0] == F(16.0) / F(255.0)
    with pytest.raises(g.GyroflowCoreError):
        g.background_for_plane("UV8", (0, 0, 0, 0), (1,), False)                               # needs two indices
    with pytest.raises(g.GyroflowCoreError):
        g.background_for_plane("Luma8", (0, 0, 0, 0), (4,), False)


# ---- GPU tests --------------------------------------------------------------------------------------------------------------------
FPS = 30.0
ts_of = lambda f: 400.0 + 37.0 * f                   # distinct, irregular timestamps


def _planes(fmt, w, h):
    return [(t, pw, ph, yuvi, m) for (t, _, yuvi, m), (pw, ph) in zip(TABLE[fmt][2], plane_sizes(fmt, w, h))]


def _stride(pix, pw):
    _, count, sdt = abi.PIXEL_TYPES[pix]
    return (pw * count * np.dtype(sdt).itemsize + 255) // 256 * 256


class Job:
    """One format's frames through a FrameRenderQueue, and the same frames rendered plane by plane by the oracle."""

    def __init__(self, fmt, w=641, h=361, kind="device", depth=4, n=3, lens="opencv_fisheye", background=(0.0, 0.0, 0.0, 0.0),
                 limited=False, base_flags=0, fov_scale=1.0, fill=lambda f: False, ibis=False, mesh=False, src_hook=None):
        import torch
        from tests import cases
        from tests.test_frame_transform import _stab
        self.fmt, self.w, self.h, self.n, self.lens, self.fill = fmt, w, h, n, lens, fill
        self.background, self.limited, self.base_flags = background, limited, base_flags
        self.p = synth.base_kernel_params(w, h, lens=lens)
        org, sm = cases.gyro()
        kw = dict(camera_stab=_stab(n, h), per_frame_time_offsets=[0.25 * i for i in range(n)]) if ibis else {}
        self.cp = g.ComputeParams(self.p, org, sm, fov_scale=fov_scale, **kw)
        self.mesh = synth.synthetic_mesh(w, h) if mesh else None
        self.planes = _planes(fmt, w, h)
        self.srcs, self.outs, self.bufs = [], [], []
        for f in range(n):
            s_f, o_f, b_f = [], [], []
            for i, (t, pw, ph, _, _) in enumerate(self.planes):
                st = _stride(t, pw)
                src = synth.synthetic_frame(pw, ph, t, frame=7 * f + i, stride=st)
                if src_hook:
                    src = src_hook(t, src)
                dst = np.zeros((ph, st), np.uint8)
                if kind == "device":
                    ts, td = torch.from_numpy(src).cuda(), torch.from_numpy(dst).cuda()
                    b = g.Buffers(g.BufferDescription((pw, ph, st), ts.data_ptr(), length=ts.numel()),
                                  g.BufferDescription((pw, ph, st), td.data_ptr(), length=td.numel()))
                else:
                    ts, td = torch.from_numpy(src).pin_memory(), torch.from_numpy(dst).pin_memory()
                    b = g.Buffers(g.BufferDescription((pw, ph, st), ts.numpy()), g.BufferDescription((pw, ph, st), td.numpy()))
                s_f.append(ts); o_f.append(td); b_f.append(b)
            self.srcs.append(s_f); self.outs.append(o_f); self.bufs.append(b_f)
        self.st = g.stab_config(self.p, "Luma8", background=background, base_flags=base_flags)
        self.q = g.FrameRenderQueue(self.cp, self.st, fmt, lens, None, [b.input for b in self.bufs[0]], [b.output for b in self.bufs[0]],
                                    limited_range=limited, depth=depth, checksum=True)

    def render(self):
        self.sums = self.q.render(range(self.n), ts_of, lambda f: self.bufs[f], (lambda f: self.mesh) if self.mesh is not None else None, self.fill)
        self.launches = self.q.launch_count
        self.q.close()
        return self.sums

    def plane_params(self, kp, f, i):
        """The test's own KernelParams of plane i: get_frame_transform_at, then value limit, background, plane_index and fill (:531-541)."""
        t, _, _, yuvi, maxv = self.planes[i]
        k = kp.copy()
        st = g.stab_config(self.p, t, background=np_from_rgb_color(t, self.background, yuvi, self.limited), base_flags=self.base_flags)
        g.get_frame_transform_at(st, self.cp, self.bufs[f][i], k, mesh=self.mesh, frame=f)
        k.pixel_value_limit = maxv; k.max_pixel_value = maxv
        k.plane_index = i
        if self.fill(f):
            k.flags |= abi.FLAG_FILL_WITH_BACKGROUND
        return k

    def expected(self):
        """{frame: [plane bytes]} from the oracle, one plane at a time."""
        import torch
        dg = g.DeviceGyro(self.cp)
        mats = torch.zeros((max(self.w, self.h), 14), dtype=torch.float32, device="cuda")
        self.tables, self.kps, out = {}, {}, {}
        for f in range(self.n):
            kp, rows = dg.frame_transform(ts_of(f), mats.data_ptr(), max(self.w, self.h), frame=f)
            table = mats.cpu().numpy()[:rows].copy()
            self.tables[f] = (kp, rows)
            out[f] = []
            for i, (t, pw, ph, _, _) in enumerate(self.planes):
                k = self.plane_params(kp, f, i)
                want = np.zeros((ph, _stride(t, pw)), np.uint8)
                src = self.srcs[f][i].cpu().numpy()
                from tests import oracle_lib
                assert oracle_lib.undistort_image(src, want, k, t, self.lens, None, table, self.mesh) == 0
                out[f].append(want)
        dg.close()
        return out

    def check(self):
        want = self.expected()
        assert list(self.sums) == list(range(self.n))
        for f in range(self.n):
            for i in range(len(self.planes)):
                got = self.outs[f][i].cpu().numpy()
                assert np.array_equal(got, want[f][i]), "%s frame %d plane %d: %d bytes differ" % (self.fmt, f, i, int((got != want[f][i]).sum()))
                assert self.sums[f][i] == render_queue.checksum_host(want[f][i]), "%s frame %d plane %d checksum" % (self.fmt, f, i)
        return want


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,w,h,kind,depth", [
    ("NV12", 641, 361, "device", 4), ("NV12", 640, 360, "host", 1), ("NV21", 641, 361, "host", 4), ("P010LE", 641, 361, "device", 1),
    ("P210LE", 641, 361, "host", 4), ("YUV420P", 641, 361, "device", 4), ("YUV420P", 641, 361, "host", 4),
    ("YUV420P10LE", 320, 180, "device", 4), ("YUV422P16LE", 641, 361, "device", 1), ("YUVA444P12LE", 641, 361, "host", 4),
    ("GBRAPF32LE", 641, 361, "device", 4), ("GBRAPF32LE", 321, 181, "host", 1), ("AYUV64LE", 641, 361, "device", 4), ("RGBA", 641, 361, "host", 4),
])
def test_frames_match_the_oracle_plane_by_plane(fmt, w, h, kind, depth):
    job = Job(fmt, w, h, kind=kind, depth=depth, n=4, fov_scale=1.3)
    job.render()
    job.check()
    assert len({s for v in job.sums.values() for s in v}) == 4 * len(job.planes)          # distinct frames, distinct planes


@pytest.mark.gpu
@pytest.mark.parametrize("limited", [False, True])
def test_coloured_background_and_fill_on_a_zoomed_out_view(limited):
    for fmt, kind in (("NV12", "device"), ("YUV420P", "host"), ("AYUV64LE", "device"), ("GBRAPF32LE", "host")):
        job = Job(fmt, 641, 361, kind=kind, n=4, fov_scale=2.0, background=(0.9, 0.3, 0.1, 1.0), limited=limited, fill=lambda f: f % 2 == 1)
        job.render()
        want = job.check()
        t, pw = job.planes[0][:2]
        _, count, sdt = abi.PIXEL_TYPES[t]
        filled = want[1][0][:, : pw * count * np.dtype(sdt).itemsize]                            # filled frame: every pixel is the background
        assert len(np.unique(filled.view(np.dtype(sdt)).reshape(-1, count), axis=0)) == 1


@pytest.mark.gpu
def test_default_black_background_gives_neutral_chroma():
    job = Job("NV12", 641, 361, kind="device", n=2, fov_scale=2.0)
    job.render()
    want = job.check()
    uv = want[0][1][:, : 321 * 2]
    y = want[0][0][:, :641]
    assert (y == 0).mean() > 0.05                                                               # background pixels exist
    assert (uv == 0).mean() < 0.01 and ((uv == 127) | (uv == 128)).mean() > 0.05               # 0.5 * 255 on U and V, not 0


@pytest.mark.gpu
def test_yuv420p10_clamps_at_1023():
    job = Job("YUV420P10LE", 641, 361, kind="host", n=2)
    job.render()
    want = job.check()
    src_max = max(int(s.cpu().numpy().view(np.uint16).max()) for s in job.srcs[0])
    assert src_max > 1023                                                                       # the source really exceeds 10 bits
    for pl in want[0]:
        assert int(pl.view(np.uint16).max()) <= 1023


@pytest.mark.gpu
def test_fix_color_range_uses_the_plane_index():
    for fmt in ("NV12", "YUV420P"):
        job = Job(fmt, 641, 361, kind="device", n=3, base_flags=abi.FLAG_FIX_COLOR_RANGE)
        job.render()
        job.check()


@pytest.mark.gpu
def test_sony_ibis_rows_and_per_frame_mesh():
    job = Job("NV12", 641, 361, kind="host", n=4, lens="sony", ibis=True, mesh=True, depth=3)
    job.render()
    job.check()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["NV12", "YUV420P", "GBRAPF32LE", "P010LE"])
def test_launch_accounting(fmt):
    """producer + checksum + the warp launches the same planes take through gf_cuda_undistort_planes_dev_flagged, per frame."""
    import torch
    job = Job(fmt, 641, 361, kind="device", n=3)
    job.render()
    job.expected()
    # the planes of frame 0 rendered alone, grouped like the queue groups them (one pixel type, equal geometry -> one planes call)
    kp, rows = job.tables[0]
    dg = g.DeviceGyro(job.cp)
    mats = torch.zeros((max(job.w, job.h), 14), dtype=torch.float32, device="cuda")
    flags = torch.zeros(1, dtype=torch.int32, device="cuda")
    dg.frame_transform(ts_of(0), mats.data_ptr(), max(job.w, job.h), frame=0, table_flags_dev=flags.data_ptr())
    torch.cuda.synchronize()
    kps = [job.plane_params(kp, 0, i) for i in range(len(job.planes))]
    groups = []
    for i, (t, pw, ph, _, _) in enumerate(job.planes):
        for gr in groups:
            j = gr[0]
            a, b = kps[i].copy(), kps[j].copy()
            a.plane_index = b.plane_index = 0; a.background[:] = b.background[:] = [0.0] * 4
            if job.planes[j][0] == t and bytes(a) == bytes(b) and job.planes[j][1:3] == (pw, ph):
                gr.append(i); break
        else:
            groups.append([i])
    warp = 0
    for gr in groups:
        t = job.planes[gr[0]][0]
        w = g.CudaWrapper.new(kps[gr[0]], t, job.lens, None, job.bufs[0][gr[0]])
        w.undistort_planes_dev([job.bufs[0][i] for i in gr], [kps[i] for i in gr], mats.data_ptr(), rows, table_flags_dev=flags.data_ptr())
        w.synchronize()
        warp += w.launch_count
        w.close()
    dg.close()
    if fmt in ("YUV420P", "GBRAPF32LE"):
        assert any(len(gr) > 1 for gr in groups)                                                # equal-geometry planes share a pass
    assert job.launches == job.n * (1 + 1 + warp), (job.launches, warp, groups)


@pytest.mark.gpu
def test_errors():
    job = Job("NV12", 640, 360, kind="device", depth=2, n=3)
    q, b = job.q, job.bufs
    with pytest.raises(g.GyroflowCoreError) as e:
        q.submit(0, 100.0, b[0][:1])                                                            # one plane of two
    assert e.value.kind == "BadParams"
    bad = [b[0][0], g.Buffers(g.BufferDescription((319, 180, b[0][1].input.size[2]), b[0][1].input.data, length=b[0][1].input.length), b[0][1].output)]
    with pytest.raises(g.GyroflowCoreError) as e:
        q.submit(0, 100.0, bad)                                                                 # chroma plane one pixel narrower than the layout
    assert e.value.kind == "SizeMismatch"
    q.submit(0, 100.0, b[0]); q.submit(1, 120.0, b[1])
    with pytest.raises(g.GyroflowCoreError) as e:
        q.submit(2, 140.0, b[2])                                                                # queue full
    assert e.value.kind == "BadParams"
    assert q.wait()[0] == 0 and q.wait()[0] == 1
    with pytest.raises(g.GyroflowCoreError) as e:
        q.wait()
    assert e.value.kind == "NoStabilizationData"
    q.in_flight = 0
    single = g.RenderQueue(job.cp, g.stab_config(job.p, "Luma8"), "opencv_fisheye", None, b[0][0].input, b[0][0].output, depth=1)
    ins = (abi.BufferDesc * 2)(*[x.input.to_c() for x in b[0]]); outs = (abi.BufferDesc * 2)(*[x.output.to_c() for x in b[0]])
    assert single._lib.gf_cuda_queue_submit_frame(single._h, 0, 100.0, 2, ins, outs, None, 0, 0) == -1      # not a frame queue
    single.close()
    q.close()
