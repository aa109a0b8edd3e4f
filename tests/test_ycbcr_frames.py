"""YCbCr frames with subsampled chroma (I420, I422, I444, NV12, NV21, NV16), read from their planes.

jpgb_encode_batch_device_ycbcr, Encoder.encode_batch_device_ycbcr and Encoder.encode_cuda_ycbcr. A frame means the
full-resolution image whose chroma repeats every plane sample c_h x c_v times; every file is compared byte for byte
with the oracle's Ycbcr encode of that image. Without a GPU: the mapping restated in numpy and pinned with known
answers, the index identity the stage A kernels rely on, and the interface parser."""
import contextlib
import functools

import numpy as np
import pytest

import images
from cases import CT, make_encoder, oracle_encode

gpu = pytest.mark.gpu

SAMPLINGS = [(1, 1), (2, 1), (1, 2), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)]
SUBSAMPLINGS = {"420": (2, 2), "422": (2, 1), "440": (1, 2), "444": (1, 1)}
MODES = {
    "baseline": dict(quality=90, sampling=(2, 2)),
    "optimized": dict(quality=85, sampling=(2, 1), optimize_huffman=True),
    "progressive": dict(quality=80, sampling=(2, 2), progressive_scans=4),
    "restart7": dict(quality=88, sampling=(1, 1), restart_interval=7),
}


# ---- the mapping, restated -------------------------------------------------------------------------------------------
def replicate(y, cb, cr, c_h, c_v):
    """The full-resolution (H, W, 3) image of one frame: pixel (x, y) takes chroma sample (x // c_h, y // c_v)"""
    h, w = y.shape
    rows, cols = np.arange(h) // c_v, np.arange(w) // c_h
    return np.stack([y, cb[rows][:, cols], cr[rows][:, cols]], -1).astype(np.uint8)


def test_replicate_known_answers():
    y = np.arange(15, dtype=np.uint8).reshape(3, 5)
    cb = np.array([[10, 11, 12], [20, 21, 22]], np.uint8)
    cr = cb + 100
    img = replicate(y, cb, cr, 2, 2)
    assert img[..., 0].tolist() == y.tolist()
    assert img[..., 1].tolist() == [[10, 10, 11, 11, 12], [10, 10, 11, 11, 12], [20, 20, 21, 21, 22]]
    assert img[..., 2].tolist() == [[110, 110, 111, 111, 112], [110, 110, 111, 111, 112], [120, 120, 121, 121, 122]]
    # 4:2:2 at an odd width, 4:4:0 at an odd height
    assert replicate(y, cb[:1].repeat(3, 0), cr[:1].repeat(3, 0), 2, 1)[..., 1].tolist() == [[10, 10, 11, 11, 12]] * 3
    c440 = np.arange(10, dtype=np.uint8).reshape(2, 5)
    assert replicate(y, c440, c440, 1, 2)[..., 2].tolist() == [[0, 1, 2, 3, 4], [0, 1, 2, 3, 4], [5, 6, 7, 8, 9]]
    # 1x1, 1xN, Nx1
    one = np.array([[7]], np.uint8)
    assert replicate(one, one + 1, one + 2, 2, 2).tolist() == [[[7, 8, 9]]]
    row = np.arange(5, dtype=np.uint8)[None]
    assert replicate(row, np.array([[1, 2, 3]], np.uint8), np.array([[4, 5, 6]], np.uint8), 2, 2)[0, :, 1].tolist() == [1, 1, 2, 2, 3]
    col = np.arange(5, dtype=np.uint8)[:, None]
    assert replicate(col, np.array([[1], [2], [3]], np.uint8), np.array([[4], [5], [6]], np.uint8), 2, 2)[:, 0, 2].tolist() == [4, 4, 5, 5, 6]


def _grid(n_px, factor, fmax):
    """Full-resolution sample positions get_block reads along one axis for a component sampled `factor` of `fmax`
    (oracle/jpeg_oracle.c get_block: start = block * 8 * stride, stride = fmax / factor, over the MCU-padded grid)"""
    mcus = -(-n_px // (8 * fmax))
    blocks, step = mcus * factor, fmax // factor
    return blocks, step, (np.arange(blocks)[:, None] * 8 * step + np.arange(8)[None] * step)


@pytest.mark.parametrize("sub", list(SUBSAMPLINGS))
@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_plane_indices_match_get_block(sub, sampling):
    """What the stage A kernels read (the plane at its own resolution, its own edge clamp, a step of k * NX / 2 plane
    samples with NX = 2 * decimation / subsampling) equals what get_block reads from the edge-padded, replicated
    full-resolution plane, for every block sample of the padded grid."""
    c_h, c_v = SUBSAMPLINGS[sub]
    hmax, vmax = sampling
    for n_px in (1, 7, 8, 9, 15, 16, 17, 33, 127, 1081):
        for sub_f, fmax in ((c_h, hmax), (c_v, vmax)):
            # chroma is sampled 1 of fmax; luma (fmax of fmax, subsampling 1) is the step-1 plane read
            for factor, s in ((1, sub_f), (fmax, 1)):
                blocks, step, pos = _grid(n_px, factor, fmax)
                n_plane = -(-n_px // s)
                padded = np.minimum(pos, n_px - 1)                  # edge-replicated full-resolution buffer
                want = padded // s                                  # the replicated buffer's plane sample
                nx = 2 * step // s
                kernel = np.minimum(np.arange(blocks)[:, None] * 4 * nx + (np.arange(8)[None] * nx) // 2, n_plane - 1)
                assert (kernel == want).all(), (n_px, factor, fmax, s)
                assert (np.minimum(pos // s, n_plane - 1) == want).all()


# ---- the interface parser (no GPU) -----------------------------------------------------------------------------------
def _iface(shape, strides=None, data=0x10000, typestr="|u1", **extra):
    d = dict(shape=shape, strides=strides, data=(data, False), typestr=typestr, version=3)
    d.update(extra)
    return d


def _parse(*a):
    from jpeg_encoder_b200.encoder import _cuda_ycbcr_layout
    return _cuda_ycbcr_layout(*a)


def test_parse_i420_batch_and_single():
    n, h, w = 4, 37, 51
    ch, cw = 19, 26
    y = _iface((n, h, w), data=0x100000)
    cb = _iface((n, ch, cw), data=0x200000)
    cr = _iface((n, ch, cw), data=0x300000)
    assert _parse(y, cb, cr) == (0x100000, 0x200000, 0x300000, n, w, h, h * w, w, ch * cw, cw, 1, 2, 2)
    assert _parse(_iface((h, w)), _iface((ch, cw), data=2), _iface((ch, cw), data=3)) == (0x10000, 2, 3, 1, w, h, 0, w, 0, cw, 1, 2, 2)


def test_parse_i422_i444_i440():
    assert _parse(_iface((8, 10)), _iface((8, 5)), _iface((8, 5)))[-2:] == (2, 1)
    assert _parse(_iface((8, 10)), _iface((8, 10)), _iface((8, 10)))[-2:] == (1, 1)
    assert _parse(_iface((9, 10)), _iface((5, 10)), _iface((5, 10)))[-2:] == (1, 2)
    # a width or height of 1 reads the same either way: 1
    assert _parse(_iface((1, 1)), _iface((1, 1)), _iface((1, 1)))[-2:] == (1, 1)


def test_parse_nv12_nv21_frame_buffer():
    h, w = 6, 8
    base = 0x40000
    # f of shape (H * 3 // 2, W): y = f[:H], uv = f[H:].view(H // 2, W // 2, 2)
    y = _iface((h, w), (w, 1), data=base)
    uv = base + h * w
    cb = _iface((h // 2, w // 2), (w, 2), data=uv)
    cr = _iface((h // 2, w // 2), (w, 2), data=uv + 1)
    assert _parse(y, cb, cr) == (base, uv, uv + 1, 1, w, h, 0, w, 0, w, 2, 2, 2)
    assert _parse(y, cr, cb)[1:3] == (uv + 1, uv)  # NV21
    # a batch of NV12 frames (N, H * 3 // 2, W)
    n, fs = 3, h * w * 3 // 2
    got = _parse(_iface((n, h, w), (fs, w, 1), data=base), _iface((n, h // 2, w // 2), (fs, w, 2), data=uv),
                 _iface((n, h // 2, w // 2), (fs, w, 2), data=uv + 1))
    assert got == (base, uv, uv + 1, n, w, h, fs, w, fs, w, 2, 2, 2)


def test_parse_crops():
    # a (100, 200) luma crop [10:50, 8:108] and its 4:2:0 chroma [5:25, 4:54] of (50, 100) planes
    y = _iface((40, 100), (200, 1), data=0x10000 + 10 * 200 + 8)
    cb = _iface((20, 50), (100, 1), data=0x20000 + 5 * 100 + 4)
    cr = _iface((20, 50), (100, 1), data=0x30000 + 5 * 100 + 4)
    assert _parse(y, cb, cr) == (0x10000 + 2008, 0x20000 + 504, 0x30000 + 504, 1, 100, 40, 0, 200, 0, 100, 1, 2, 2)


@pytest.mark.parametrize("args,what", [
    ((_iface((8, 10)), _iface((4, 5), (10, 1)), _iface((4, 5), (5, 1))), "cb and cr strides differ"),
    ((_iface((8, 10)), _iface((4, 5)), _iface((4, 4))), "cb and cr shapes differ"),
    ((_iface((8, 10)), _iface((4, 5), (20, 4)), _iface((4, 5), (20, 4))), "chroma x stride 4"),
    ((_iface((8, 10)), _iface((4, 5), (20, 3)), _iface((4, 5), (20, 3))), "chroma x stride 3"),
    ((_iface((8, 10)), _iface((4, 4)), _iface((4, 4))), "chroma width 4 fits no subsampling"),
    ((_iface((8, 10)), _iface((3, 5)), _iface((3, 5))), "chroma height 3 fits no subsampling"),
    ((_iface((8, 10)), _iface((4, 6)), _iface((4, 6))), "chroma width 6 fits no subsampling"),
    ((_iface((8, 10), typestr="<u2"), _iface((4, 5)), _iface((4, 5))), "uint8 planes only"),
    ((_iface((8, 10)), _iface((4, 5), typestr="<f4"), _iface((4, 5))), "uint8 planes only"),
    ((_iface((8, 10)), _iface((4, 5)), _iface((4, 5), typestr="|i1")), "uint8 planes only"),
    ((_iface((1, 8, 10, 3)), _iface((4, 5)), _iface((4, 5))), "2-D .one frame. or 3-D .batch."),
    ((_iface((2, 8, 10)), _iface((4, 5)), _iface((4, 5))), "all be batches or all single frames"),
    ((_iface((2, 8, 10)), _iface((3, 4, 5)), _iface((3, 4, 5))), "y holds 2 frames"),
    ((_iface((8, 10), (20, 2)), _iface((4, 5)), _iface((4, 5))), "y x stride 2"),
    ((_iface((2, 8, 10), (-80, 10, 1)), _iface((2, 4, 5)), _iface((2, 4, 5))), "negative n stride"),
    ((_iface((8, 10)), _iface((4, 5), mask=object()), _iface((4, 5))), "masked"),
    ((_iface((8, 70000)), _iface((4, 35000)), _iface((4, 35000))), "above 65535"),
])
def test_parse_rejections(args, what):
    with pytest.raises(ValueError, match=what):
        _parse(*args)


def test_library_exports_the_entry():
    import jpeg_encoder_b200 as je
    assert hasattr(je.load_library(), "jpgb_encode_batch_device_ycbcr")


# ---- GPU helpers -------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _planes(w, h, c_h, c_v, seed):
    """(y, cb, cr) of one photo-like frame: chroma planes of ceil(w / c_h) x ceil(h / c_v) samples"""
    img = images.photo_like(w, h, 3, seed=seed).reshape(h, w, 3)
    return (np.ascontiguousarray(img[..., 0]), np.ascontiguousarray(img[::c_v, ::c_h, 1]), np.ascontiguousarray(img[::c_v, ::c_h, 2]))


_ORACLE = {}


def _want(w, h, c_h, c_v, seed, cfg):
    key = (w, h, c_h, c_v, seed, repr(sorted(cfg.items())))
    if key not in _ORACLE:
        y, cb, cr = _planes(w, h, c_h, c_v, seed)
        _ORACLE[key] = oracle_encode(replicate(y, cb, cr, c_h, c_v), w, h, "ycbcr", cfg)
    return _ORACLE[key]


@contextlib.contextmanager
def _context():
    import jpeg_encoder_b200 as je
    dev = je.Device(0)
    try:
        yield dev
    finally:
        dev.close()


def _files(dev, d_files, offs):
    blob = dev.download(d_files, offs[-1]) if offs[-1] else b""
    return [bytes(blob[offs[i]:offs[i + 1]]) for i in range(len(offs) - 1)]


def _check(files, want):
    assert len(files) == len(want)
    bad = [i for i, (g, x) in enumerate(zip(files, want)) if g != x]
    assert not bad, "files %r differ (first: %d vs %d bytes)" % (bad[:8], len(files[bad[0]]), len(want[bad[0]]))


def _junk(nbytes, seed, fill):
    if fill == "ff":
        return np.full(nbytes, 0xFF, np.uint8)
    return np.random.default_rng(seed).integers(0, 256, nbytes, dtype=np.uint8)


def _put(buf, off, strides, data):
    """data (n, rows, cols) into buf at off + i*strides[0] + r*strides[1] + c*strides[2]"""
    v = np.lib.stride_tricks.as_strided(buf[off:], shape=data.shape, strides=strides)
    v[...] = data


class Frames:
    """Frames laid out in device buffers full of junk: `layout` planar (three planes), interleaved (Cb, Cr pairs),
    interleaved_cr (Cr, Cb pairs) or split2 (Cb and Cr each at a sample stride of 2 in separate buffers, the other
    byte of each pair junk, Cr at odd addresses). y_pad / c_pad: bytes of junk behind each row; gap: behind each image;
    shift: bytes in front of the first sample (unaligned bases)."""

    def __init__(self, planes, c_h, c_v, layout="planar", y_pad=0, c_pad=0, gap=0, shift=0, fill="random", seed=3):
        import torch
        ys, cbs, crs = (np.stack(p) for p in zip(*planes))
        n, h, w = ys.shape
        _, ch, cw = cbs.shape
        ss = 1 if layout == "planar" else 2
        self.y_row, self.c_row = w + y_pad, cw * ss + c_pad
        self.y_img, self.c_img = h * self.y_row + gap, ch * self.c_row + gap
        ybuf = _junk(shift + n * self.y_img + 64, seed, fill)
        _put(ybuf, shift, (self.y_img, self.y_row, 1), ys)
        cbuf = _junk(shift + n * self.c_img + 64, seed + 1, fill)
        offs = {"planar": (0, 0), "interleaved": (0, 1), "interleaved_cr": (1, 0), "split2": (0, 1)}[layout]
        if layout in ("planar", "split2"):
            rbuf = _junk(shift + n * self.c_img + 64, seed + 2, fill)
        else:
            rbuf = cbuf
        _put(cbuf, shift + offs[0], (self.c_img, self.c_row, ss), cbs)
        _put(rbuf, shift + offs[1], (self.c_img, self.c_row, ss), crs)
        self.bufs = [torch.from_numpy(b).cuda() for b in (ybuf, cbuf, rbuf)]
        torch.cuda.synchronize()
        self.ptrs = (self.bufs[0].data_ptr() + shift, self.bufs[1].data_ptr() + shift + offs[0], self.bufs[2].data_ptr() + shift + offs[1])
        self.n, self.w, self.h, self.ss, self.c_h, self.c_v = n, w, h, ss, c_h, c_v

    def args(self, **over):
        a = dict(y=self.ptrs[0], cb=self.ptrs[1], cr=self.ptrs[2], n=self.n, width=self.w, height=self.h, y_image_stride=self.y_img,
                 y_row_stride=self.y_row, c_image_stride=self.c_img, c_row_stride=self.c_row, c_sample_stride=self.ss, c_h=self.c_h,
                 c_v=self.c_v)
        a.update(over)
        return a

    def encode(self, dev, cfg, **over):
        return _files(dev, *make_encoder(cfg, dev).encode_batch_device_ycbcr(**self.args(**over)))


def _run(w, h, sub, cfg, layout="planar", n=1, seeds=None, **kw):
    c_h, c_v = SUBSAMPLINGS[sub]
    seeds = seeds or [11 + i for i in range(n)]
    fr = Frames([_planes(w, h, c_h, c_v, s) for s in seeds], c_h, c_v, layout, **kw)
    with _context() as dev:
        got = fr.encode(dev, cfg)
    _check(got, [_want(w, h, c_h, c_v, s, cfg) for s in seeds])


# ---- every subsampling x layout x mode -------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("layout", ["planar", "interleaved", "interleaved_cr"])
@pytest.mark.parametrize("sub", list(SUBSAMPLINGS))
def test_subsampling_layout_mode(sub, layout, mode):
    _run(333, 75, sub, MODES[mode], layout, n=2, y_pad=5, c_pad=3)


@gpu
@pytest.mark.parametrize("layout", ["planar", "interleaved"])
@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_i420_nv12_every_sampling(sampling, layout):
    _run(544, 100, "420", dict(quality=87, sampling=sampling), layout, n=2)


@gpu
@pytest.mark.parametrize("layout", ["planar", "split2"])
@pytest.mark.parametrize("sampling", SAMPLINGS)
@pytest.mark.parametrize("sub", ["422", "440", "444"])
def test_other_subsamplings_every_sampling(sub, sampling, layout):
    _run(290, 70, sub, dict(quality=86, sampling=sampling), layout)


@gpu
@pytest.mark.parametrize("size", [(1, 1), (1, 17), (17, 1), (3, 5), (31, 33), (17, 40), (273, 45), (1041, 19)])
@pytest.mark.parametrize("sub", ["420", "422"])
@pytest.mark.parametrize("layout", ["planar", "interleaved"])
def test_ragged_sizes(size, sub, layout):
    w, h = size
    for cfg in (dict(quality=90, sampling=(2, 2)), dict(quality=92, sampling=(1, 1)), dict(quality=85, sampling=(4, 1))):
        _run(w, h, sub, cfg, layout)


@gpu
@pytest.mark.parametrize("pads", [(0, 0, 0), (16, 16, 0), (1, 3, 1), (7, 1, 3), (512, 256, 16)])
@pytest.mark.parametrize("layout", ["planar", "interleaved", "interleaved_cr", "split2"])
def test_pitches_and_unaligned_bases(pads, layout):
    """row pitches with junk in the gap, and unaligned bases and pitches: the edge staging and cp.async both run"""
    y_pad, c_pad, shift = pads
    for cfg in (dict(quality=90, sampling=(2, 2)), dict(quality=95, sampling=(1, 1))):
        _run(1000, 70, "420", cfg, layout, n=2, y_pad=y_pad, c_pad=c_pad, shift=shift, gap=shift * 5)


@gpu
@pytest.mark.parametrize("fill", ["ff", "random"])
def test_junk_everywhere_outside_the_samples(fill):
    for layout in ("planar", "split2", "interleaved_cr"):
        for sub in ("420", "422"):
            _run(401, 77, sub, dict(quality=90, sampling=(2, 2)), layout, n=3, y_pad=9, c_pad=7, gap=4096 + 3, fill=fill)


@gpu
def test_contiguous_i420_buffer_and_separate_tensors_and_image_stride_0():
    import torch
    w, h, c_h, c_v = 640, 360, 2, 2
    cfg = dict(quality=90, sampling=(2, 2))
    y, cb, cr = _planes(w, h, c_h, c_v, 31)
    want = _want(w, h, c_h, c_v, 31, cfg)
    frame = torch.from_numpy(np.concatenate([y.reshape(-1), cb.reshape(-1), cr.reshape(-1)])).cuda()
    ty, tcb, tcr = (torch.from_numpy(p).cuda() for p in (y, cb, cr))
    n_cb = cb.size
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        one = frame[:w * h].view(h, w), frame[w * h:w * h + n_cb].view(h // 2, w // 2), frame[w * h + n_cb:].view(h // 2, w // 2)
        _check(_files(dev, *enc.encode_cuda_ycbcr(*one)), [want])
        _check(_files(dev, *enc.encode_cuda_ycbcr(ty, tcb, tcr)), [want])
        # image stride 0: every image is the same frame
        _check(_files(dev, *enc.encode_batch_device_ycbcr(ty.data_ptr(), tcb.data_ptr(), tcr.data_ptr(), 4, w, h, 0, w, 0, w // 2, 1, 2, 2)),
               [want] * 4)


@gpu
def test_nv12_frame_buffer_views_and_nv21():
    import torch
    n, w, h = 3, 320, 240
    cfg = dict(quality=88, sampling=(2, 2))
    seeds = [41, 42, 43]
    fs = []
    for s in seeds:
        y, cb, cr = _planes(w, h, 2, 2, s)
        fs.append(np.concatenate([y, np.stack([cb, cr], -1).reshape(h // 2, w)]))
    f = torch.from_numpy(np.stack(fs)).cuda()  # (N, H * 3 // 2, W)
    uv = f[:, h:].view(n, h // 2, w // 2, 2)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        want = [_want(w, h, 2, 2, s, cfg) for s in seeds]
        _check(_files(dev, *enc.encode_cuda_ycbcr(f[:, :h], uv[..., 0], uv[..., 1])), want)
        # NV21 of the same buffer: the channels swap roles
        swapped = [oracle_encode(replicate(*(lambda p: (p[0], p[2], p[1]))(_planes(w, h, 2, 2, s)), 2, 2), w, h, "ycbcr", cfg) for s in seeds]
        _check(_files(dev, *enc.encode_cuda_ycbcr(f[:, :h], uv[..., 1], uv[..., 0])), swapped)


@gpu
@pytest.mark.parametrize("sampling", [(1, 1), (2, 2), (2, 1)])
def test_i444_matches_strided_planar(sampling):
    w, h, n = 500, 90, 2
    cfg = dict(quality=90, sampling=sampling)
    import torch
    planes = [_planes(w, h, 1, 1, 51 + i) for i in range(n)]
    t = torch.from_numpy(np.stack([np.stack(p) for p in planes])).cuda()  # (N, 3, H, W)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        strided = _files(dev, *enc.encode_batch_device_strided(t.data_ptr(), n, w, h, CT["ycbcr"][1], 3 * h * w, w, h * w))
        frames = _files(dev, *enc.encode_cuda_ycbcr(t[:, 0], t[:, 1], t[:, 2]))
    assert frames == strided
    _check(frames, [_want(w, h, 1, 1, 51 + i, cfg) for i in range(n)])


# ---- cross-checks and context hooks ----------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("hook", ["JPGB_FORCE_GENERIC_STAGE_A", "JPGB_NO_TMA", "JPGB_POISON_ALLOC"])
@pytest.mark.parametrize("sub", ["420", "444", "440"])
def test_hooks(hook, sub, monkeypatch):
    monkeypatch.setenv(hook, "1")
    for layout in ("planar", "interleaved_cr"):
        for cfg in (dict(quality=90, sampling=(2, 2)), dict(quality=95, sampling=(1, 1)), MODES["progressive"], dict(quality=80, sampling=(4, 2))):
            _run(357, 66, sub, cfg, layout, n=2, y_pad=3, c_pad=5)


@gpu
@pytest.mark.parametrize("tight", ["pool", "stream", "out", "pool,stream,out"])
def test_tight_caps_retries(tight, monkeypatch):
    c_h, c_v = 2, 2
    w, h = 640, 200
    cfg = dict(quality=90, sampling=(2, 2))
    fr = Frames([_planes(w, h, c_h, c_v, 61 + i) for i in range(3)], c_h, c_v, "interleaved")
    want = [_want(w, h, c_h, c_v, 61 + i, cfg) for i in range(3)]
    counts = []
    with _context() as dev:
        for k in range(3):
            if k == 0:
                monkeypatch.setenv("JPGB_TIGHT_CAPS", tight)
            _check(fr.encode(dev, cfg), want)
            counts.append(dev.last_launch_count())
            if k == 0:
                monkeypatch.delenv("JPGB_TIGHT_CAPS")
    assert counts[1] == counts[2] < counts[0], counts


@gpu
def test_launch_count_is_the_packed_calls():
    """stage A runs once per call (one launch per plane, counted as one colour+DCT pass like the planar entries);
    everything behind it is the packed Ycbcr call's launch sequence"""
    import torch
    w, h = 1920, 1080
    cfg = dict(quality=90, sampling=(2, 2))
    y, cb, cr = _planes(w, h, 2, 2, 71)
    packed = torch.from_numpy(replicate(y, cb, cr, 2, 2)).cuda()
    fr = Frames([(y, cb, cr)], 2, 2, "interleaved")
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        counts = {"packed": [], "frames": []}
        for _ in range(3):
            enc.encode_batch_device(packed.data_ptr(), w * h * 3, 1, w, h, CT["ycbcr"][1])
            counts["packed"].append(dev.last_launch_count())
            _check(fr.encode(dev, cfg), [_want(w, h, 2, 2, 71, cfg)])
            counts["frames"].append(dev.last_launch_count())
    assert counts["frames"][1:] == counts["packed"][1:], counts


@gpu
def test_rejections():
    import torch
    import jpeg_encoder_b200 as je
    w, h = 64, 48
    fr = Frames([_planes(w, h, 2, 2, 81)], 2, 2, "interleaved")
    with _context() as dev:
        enc = make_encoder(dict(quality=90, sampling=(2, 2)), dev)

        def rejected(what, code=5, **over):
            a = fr.args(**over)
            with pytest.raises(je.EncodingError) as e:
                enc.encode_batch_device_ycbcr(**a)
            assert e.value.code == code, (e.value.code, str(e.value))
            assert what in dev.last_error(), dev.last_error()
            assert dev.last_launch_count() == 0

        _check(fr.encode(dev, dict(quality=90, sampling=(2, 2))), [_want(w, h, 2, 2, 81, dict(quality=90, sampling=(2, 2)))])
        assert dev.last_launch_count() > 0
        rejected("null argument", y=None)
        rejected("null argument", cr=None)
        rejected("null argument", n=0)
        rejected("Image dimensions must be non zero", code=2, width=0)
        rejected("c_h = 4", c_h=4)
        rejected("c_v = 0", c_v=0)
        rejected("c_sample_stride 3", c_sample_stride=3)
        rejected("y_row_stride 63", y_row_stride=w - 1)
        rejected("c_row_stride 62", c_row_stride=62)
        rejected("64-bit", n=3, c_image_stride=1 << 63)
        host = np.zeros(1 << 16, np.uint8)
        rejected("y is not device or managed memory", y=host.ctypes.data)
        rejected("cb is not device or managed memory", cb=host.ctypes.data)
        rejected("cr is not device or managed memory", cr=host.ctypes.data + 1)
        rejected("past the end of the allocation that holds cb", n=2, c_image_stride=1 << 30)
        rejected("past the end of the allocation that holds y", n=2, y_image_stride=1 << 30)
        # cr one byte past the end of the caching allocator's segment (the range cuMemGetAddressRange reports)
        seg = next(s for s in torch.cuda.memory_snapshot()
                   if s["address"] <= fr.ptrs[2] < s["address"] + s["total_size"])
        end = seg["address"] + seg["total_size"]
        cw = w // 2
        last = (h // 2 - 1) * fr.c_row + (cw - 1) * 2  # offset of cr's last sample
        rejected("1 bytes past the end of the allocation that holds cr", cr=end - last)
        enc.encode_batch_device_ycbcr(**fr.args(cr=end - 1 - last))  # ends on the segment's last byte: accepted
        assert dev.last_launch_count() > 0
        # color_type other than Ycbcr: the parameter block of another colour type
        p = enc._params(w, h, je.ColorType.Rgb)
        import ctypes as C
        from jpeg_encoder_b200.encoder import _DeviceYcbcr
        a = fr.args()
        f = _DeviceYcbcr(a["y"], a["cb"], a["cr"], a["y_image_stride"], a["y_row_stride"], a["c_image_stride"], a["c_row_stride"],
                         a["c_sample_stride"], a["c_h"], a["c_v"])
        d_files, offs = C.c_void_p(), (C.c_uint64 * 2)()
        assert dev.lib.jpgb_encode_batch_device_ycbcr(dev.handle, C.byref(p), C.byref(f), 1, C.byref(d_files), offs) == 5
        assert "color_type Ycbcr" in dev.last_error() and dev.last_launch_count() == 0


# ---- full size -------------------------------------------------------------------------------------------------------
@gpu
def test_full_size_nv12_batch_every_file():
    """96 NV12 1080p frames, q90 4:2:0, in one call: every file byte for byte"""
    import torch
    w, h, n, distinct = 1920, 1080, 96, 6
    cfg = dict(quality=90, sampling=(2, 2))
    frames = []
    for s in range(distinct):
        img = images.synth_frame(w, h, 3, seed=s).reshape(h, w, 3)
        frames.append((np.ascontiguousarray(img[..., 0]), np.ascontiguousarray(img[::2, ::2, 1]), np.ascontiguousarray(img[::2, ::2, 2])))
    want = [oracle_encode(replicate(*f, 2, 2), w, h, "ycbcr", cfg) for f in frames]
    order = [(i * 5 + i // 7) % distinct for i in range(n)]
    bufs = [torch.from_numpy(np.concatenate([f[0], np.stack([f[1], f[2]], -1).reshape(h // 2, w)])) for f in frames]
    t = torch.stack([bufs[k] for k in order]).cuda()
    uv = t[:, h:].view(n, h // 2, w // 2, 2)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        _check(_files(dev, *enc.encode_cuda_ycbcr(t[:, :h], uv[..., 0], uv[..., 1])), [want[k] for k in order])


@gpu
def test_8192_i420_upsampled_to_444():
    """one 8192 x 8192 I420 frame at q95, F_1_1: the half-sample steps at size"""
    w = h = 8192
    cfg = dict(quality=95, sampling=(1, 1))
    _run(w, h, "420", cfg, "planar")
