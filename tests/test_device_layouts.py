"""Device images read where they lie: a row pitch, crops of a tensor, channel-planar (NCHW) batches.

jpgb_encode_batch_device_strided and Encoder.encode_cuda_array. Every file is compared byte for byte with the oracle's
encode of the packed, contiguous copy of the same pixels. The GPU tests build their own contexts (je.Device). The
layout parser of the `__cuda_array_interface__` is checked without a GPU."""
import contextlib
import functools

import numpy as np
import pytest

import images
from cases import BPP, CT, make_encoder, oracle_encode

gpu = pytest.mark.gpu

SAMPLINGS = [(1, 1), (2, 1), (1, 2), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)]
MODES = {
    "baseline": dict(quality=90, sampling=(2, 2)),
    "optimized": dict(quality=85, sampling=(2, 1), optimize_huffman=True),
    "progressive": dict(quality=80, sampling=(2, 2), progressive_scans=4),
    "restart7": dict(quality=88, sampling=(1, 1), restart_interval=7),
}


# ---- the interface parser (no GPU) ---------------------------------------------------------------------------------
def _iface(shape, strides=None, data=0x10000, typestr="|u1", **extra):
    d = dict(shape=shape, strides=strides, data=(data, False), typestr=typestr, version=3)
    d.update(extra)
    return d


def _layout(*a, **k):
    from jpeg_encoder_b200.encoder import _cuda_array_layout
    return _cuda_array_layout(*a, **k)


def test_layout_contiguous_nhwc_and_nchw():
    assert _layout(_iface((5, 40, 30, 3)), 3, False) == (0x10000, 5, 30, 40, 40 * 30 * 3, 90, 0)
    assert _layout(_iface((5, 3, 40, 30)), 3, True) == (0x10000, 5, 30, 40, 3 * 40 * 30, 30, 40 * 30)


def test_layout_crops():
    # t[:, 10:50, 7:107, :] of a (4, 100, 200, 4) tensor: the rows keep the parent's pitch, data moves
    base, full = 0x20000, (100 * 200 * 4, 200 * 4, 4, 1)
    got = _layout(_iface((4, 40, 100, 4), full, data=base + 10 * 800 + 7 * 4), 4, False)
    assert got == (base + 10 * 800 + 28, 4, 100, 40, 80000, 800, 0)
    # t[:, :, 3:43, 5:105] of a (2, 3, 60, 120) tensor
    got = _layout(_iface((2, 3, 40, 100), (3 * 60 * 120, 60 * 120, 120, 1), data=base + 3 * 120 + 5), 3, True)
    assert got == (base + 365, 2, 100, 40, 3 * 60 * 120, 120, 7200)


def test_layout_hcw_rows():
    # an (H, C, W) tensor seen as (C, H, W): the planes interleave row by row
    h, c, w = 50, 3, 64
    assert _layout(_iface((c, h, w), (w, c * w, 1)), 3, True) == (0x10000, 1, w, h, 0, c * w, w)


def test_layout_single_image_and_luma():
    assert _layout(_iface((20, 30, 4)), 4, False) == (0x10000, 1, 30, 20, 0, 120, 0)
    assert _layout(_iface((1, 20, 30)), 1, True) == (0x10000, 1, 30, 20, 0, 30, 0)  # one plane is packed luma


@pytest.mark.parametrize("iface,bpp,cf,what", [
    (_iface((2, 10, 10, 3), (-300, 30, 3, 1)), 3, False, "negative n stride"),
    (_iface((10, 10, 3), (30, 3, 2)), 3, False, "channel stride 2"),
    (_iface((10, 10, 3), (40, 4, 1)), 3, False, "pixel stride 4"),
    (_iface((10, 10, 4)), 3, False, "takes 3 channels"),
    (_iface((3, 10, 10)), 4, True, "takes 4 channels"),
    (_iface((3, 10, 10), (100, 10, 2)), 3, True, "x stride 2"),
    (_iface((10, 10, 3), typestr="<u2"), 3, False, "uint8"),
    (_iface((10, 10, 3), mask=object()), 3, False, "masked"),
    (_iface((10, 30)), 3, False, "shape"),
    (_iface((1, 2, 10, 10, 3)), 3, False, "shape"),
])
def test_layout_rejections(iface, bpp, cf, what):
    with pytest.raises(ValueError, match=what):
        _layout(iface, bpp, cf)
    if "stride" in what:
        with pytest.raises(ValueError, match="contiguous"):
            _layout(iface, bpp, cf)


# ---- GPU helpers ---------------------------------------------------------------------------------------------------
_ORACLE = {}


@functools.lru_cache(maxsize=None)
def _img(w, h, ch, seed):
    """(H, W, C) uint8, photo-like"""
    return np.ascontiguousarray(images.photo_like(w, h, ch, seed=seed).reshape(h, w, ch))


def _want(w, h, ch, seed, color, cfg):
    key = (w, h, ch, seed, color, repr(sorted(cfg.items())))
    if key not in _ORACLE:
        _ORACLE[key] = oracle_encode(_img(w, h, ch, seed), w, h, color, cfg)
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


def _junk(nbytes, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, 256, (nbytes,), dtype=torch.uint8, device="cuda", generator=g)


def _pitched(imgs, pitch, image_gap=0, seed=1):
    """Images packed into rows of `pitch` bytes (junk in the gap), images h*pitch + image_gap apart: (buffer, image stride)"""
    import torch
    h, w, ch = imgs[0].shape
    image_stride = h * pitch + image_gap
    buf = _junk(len(imgs) * image_stride, seed)
    for i, im in enumerate(imgs):
        view = buf[i * image_stride:i * image_stride + h * pitch].view(h, pitch)
        view[:, :w * ch].copy_(torch.from_numpy(im.reshape(h, w * ch)))
    torch.cuda.synchronize()
    return buf, image_stride


def _planar(imgs, plane_stride=None, seed=2):
    """NCHW: channel c of image i at i*C*plane_stride + c*plane_stride (junk between planes): (buffer, plane stride)"""
    import torch
    h, w, ch = imgs[0].shape
    plane_stride = plane_stride or h * w
    buf = _junk(len(imgs) * ch * plane_stride, seed)
    for i, im in enumerate(imgs):
        for c in range(ch):
            o = (i * ch + c) * plane_stride
            buf[o:o + h * w].copy_(torch.from_numpy(np.ascontiguousarray(im[..., c]).reshape(-1)))
    torch.cuda.synchronize()
    return buf, plane_stride


def _encode_pitched(dev, color, cfg, imgs, pad, image_gap=0, seed=1):
    h, w, ch = imgs[0].shape
    pitch = ((w * ch + 511) & ~511) if pad == "512" else w * ch + pad
    buf, image_stride = _pitched(imgs, pitch, image_gap, seed)
    enc = make_encoder(cfg, dev)
    return _files(dev, *enc.encode_batch_device_strided(buf.data_ptr(), len(imgs), w, h, CT[color][1], image_stride, pitch))


def _encode_planar(dev, color, cfg, imgs, plane_stride=None, seed=2):
    h, w, ch = imgs[0].shape
    buf, ps = _planar(imgs, plane_stride, seed)
    enc = make_encoder(cfg, dev)
    return _files(dev, *enc.encode_batch_device_strided(buf.data_ptr(), len(imgs), w, h, CT[color][1], ch * ps, w, ps))


# ---- pitched packed ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("color", list(CT))
def test_pitched_packed_color_types(color, mode):
    w, h, ch = 320, 72, BPP[color]
    cfg = MODES[mode]
    pad = {"baseline": 16, "optimized": 64, "progressive": 1, "restart7": 3}[mode]
    with _context() as dev:
        _check(_encode_pitched(dev, color, cfg, [_img(w, h, ch, 5)], pad), [_want(w, h, ch, 5, color, cfg)])


@gpu
@pytest.mark.parametrize("pad", [16, 64, 1, 3, "512"])
def test_pitched_packed_pitches(pad):
    w, h = 1000, 270
    cfg = dict(quality=90, sampling=(2, 2))
    with _context() as dev:
        _check(_encode_pitched(dev, "rgb", cfg, [_img(w, h, 3, 6)], pad), [_want(w, h, 3, 6, "rgb", cfg)])


@gpu
@pytest.mark.parametrize("sampling", SAMPLINGS)
def test_pitched_rgb_samplings(sampling):
    w, h = 544, 100
    cfg = dict(quality=87, sampling=sampling)
    with _context() as dev:
        _check(_encode_pitched(dev, "rgb", cfg, [_img(w, h, 3, 7)], 64), [_want(w, h, 3, 7, "rgb", cfg)])


@gpu
@pytest.mark.parametrize("size", [(1, 1), (17, 9), (255, 2), (513, 31), (200, 40), (100, 7)])
@pytest.mark.parametrize("color", ["rgb", "luma", "cmyk"])
def test_pitched_ragged_sizes(size, color):
    w, h = size
    ch = BPP[color]
    cfg = dict(quality=90, sampling=(2, 2))
    with _context() as dev:
        _check(_encode_pitched(dev, color, cfg, [_img(w, h, ch, 8)], 3), [_want(w, h, ch, 8, color, cfg)])


@gpu
def test_pitched_batch_image_stride():
    w, h, n = 640, 200, 7
    cfg = dict(quality=90, sampling=(2, 2))
    imgs = [_img(w, h, 3, 20 + i % 3) for i in range(n)]
    with _context() as dev:
        _check(_encode_pitched(dev, "rgb", cfg, imgs, 16, image_gap=4096), [_want(w, h, 3, 20 + i % 3, "rgb", cfg) for i in range(n)])


@gpu
@pytest.mark.parametrize("x0", [0, 1, 5, 16])
def test_crops_of_one_tensor(x0):
    import torch
    n, H, W, y0, y1, cw = 3, 300, 700, 10, 250, 600
    cfg = dict(quality=90, sampling=(2, 2))
    full = np.stack([_img(W, H, 3, 30 + i) for i in range(n)])
    t = torch.from_numpy(full).cuda()
    torch.cuda.synchronize()
    crop = t[:, y0:y1, x0:x0 + cw, :]
    want = [oracle_encode(np.ascontiguousarray(full[i, y0:y1, x0:x0 + cw]), cw, y1 - y0, "rgb", cfg) for i in range(n)]
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        _check(_files(dev, *enc.encode_cuda_array(crop, CT["rgb"][1])), want)


# ---- channel-planar ------------------------------------------------------------------------------------------------
def _nchw(imgs):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(np.stack(imgs).transpose(0, 3, 1, 2))).cuda()
    torch.cuda.synchronize()
    return t


@gpu
@pytest.mark.parametrize("color", list(CT))
def test_planar_nchw_color_types(color):
    w, h, ch = 520, 130, BPP[color]
    cfg = dict(quality=85, sampling=(2, 2))
    imgs = [_img(w, h, ch, 40), _img(w, h, ch, 41)]
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        got = _files(dev, *enc.encode_cuda_array(_nchw(imgs), CT[color][1], channels_first=True))
        _check(got, [_want(w, h, ch, 40, color, cfg), _want(w, h, ch, 41, color, cfg)])


@gpu
@pytest.mark.parametrize("sampling", SAMPLINGS)
@pytest.mark.parametrize("color", ["rgb", "cmyk_as_ycck"])
def test_planar_samplings(color, sampling):
    w, h, ch = 544, 100, BPP[color]
    cfg = dict(quality=87, sampling=sampling)
    with _context() as dev:
        _check(_encode_planar(dev, color, cfg, [_img(w, h, ch, 42)]), [_want(w, h, ch, 42, color, cfg)])


@gpu
@pytest.mark.parametrize("color", ["bgr", "bgra", "rgba"])
@pytest.mark.parametrize("sampling", [(1, 1), (2, 2), (4, 1)])
def test_planar_plane_order(color, sampling):
    w, h, ch = 700, 90, BPP[color]
    cfg = dict(quality=90, sampling=sampling)
    with _context() as dev:
        _check(_encode_planar(dev, color, cfg, [_img(w, h, ch, 43)]), [_want(w, h, ch, 43, color, cfg)])


@gpu
@pytest.mark.parametrize("color", ["rgb", "ycbcr"])
def test_planar_hcw_rows(color):
    import torch
    w, h = 640, 120
    cfg = dict(quality=90, sampling=(2, 2))
    im = _img(w, h, 3, 44)
    hcw = torch.from_numpy(np.ascontiguousarray(im.transpose(0, 2, 1))).cuda()  # (H, C, W)
    torch.cuda.synchronize()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        got = _files(dev, *enc.encode_cuda_array(hcw.permute(1, 0, 2), CT[color][1], channels_first=True))
        _check(got, [_want(w, h, 3, 44, color, cfg)])


@gpu
@pytest.mark.parametrize("x0", [0, 3, 16])
def test_planar_crop(x0):
    n, H, W, y0, y1, cw = 2, 200, 800, 7, 180, 700
    cfg = dict(quality=88, sampling=(2, 2))
    full = [_img(W, H, 3, 45 + i) for i in range(n)]
    t = _nchw(full)
    want = [oracle_encode(np.ascontiguousarray(f[y0:y1, x0:x0 + cw]), cw, y1 - y0, "rgb", cfg) for f in full]
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        _check(_files(dev, *enc.encode_cuda_array(t[:, :, y0:y1, x0:x0 + cw], CT["rgb"][1], channels_first=True)), want)


@gpu
@pytest.mark.parametrize("color", ["rgb", "cmyk", "ycbcr"])
def test_planar_unaligned_plane_stride(color):
    w, h, ch = 512, 64, BPP[color]
    cfg = dict(quality=90, sampling=(2, 2))
    with _context() as dev:
        got = _encode_planar(dev, color, cfg, [_img(w, h, ch, 46), _img(w, h, ch, 47)], plane_stride=w * h + 5)
        _check(got, [_want(w, h, ch, 46, color, cfg), _want(w, h, ch, 47, color, cfg)])


@gpu
@pytest.mark.parametrize("size", [(1920, 1080), (8192, 8192)])
def test_planar_420_large(size):
    w, h = size
    cfg = dict(quality=90, sampling=(2, 2))
    with _context() as dev:
        _check(_encode_planar(dev, "rgb", cfg, [_img(w, h, 3, 48)]), [_want(w, h, 3, 48, "rgb", cfg)])


# ---- bytes outside the description ---------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("color", ["rgba", "bgra", "rgb"])
def test_bytes_outside_the_description_never_matter(color):
    w, h, ch = 600, 80, BPP[color]
    cfg = dict(quality=90, sampling=(2, 2))
    imgs = [_img(w, h, ch, 50), _img(w, h, ch, 51)]
    want = [_want(w, h, ch, 50, color, cfg), _want(w, h, ch, 51, color, cfg)]
    with _context() as dev:
        runs = [_encode_pitched(dev, color, cfg, imgs, 48, image_gap=512, seed=s) for s in (11, 12)]
        if ch == 4:  # the alpha plane is junk too: RGB(A) planes at c * plane_stride, alpha overwritten
            import torch
            outs = []
            for s in (13, 14):
                buf, ps = _planar(imgs, w * h + 256, seed=s)
                for i in range(len(imgs)):
                    buf[(i * ch + 3) * ps:(i * ch + 3) * ps + h * w].copy_(_junk(h * w, s + 100))
                torch.cuda.synchronize()
                enc = make_encoder(cfg, dev)
                outs.append(_files(dev, *enc.encode_batch_device_strided(buf.data_ptr(), len(imgs), w, h, CT[color][1], ch * ps, w, ps)))
            runs += outs
        else:
            runs += [_encode_planar(dev, color, cfg, imgs, plane_stride=w * h + 256, seed=s) for s in (13, 14)]
    for r in runs:
        _check(r, want)


# ---- the cross-checks: the generic kernel, and the cp.async staging without TMA ------------------------------------
CROSS = [("pitched", "rgb", (2, 2), 16), ("pitched", "cmyk", (1, 1), 3), ("pitched", "ycck", (2, 1), 64),
         ("planar", "rgb", (2, 2), None), ("planar", "bgra", (1, 1), None), ("planar", "cmyk_as_ycck", (2, 1), None),
         ("planar", "cmyk", (4, 1), None), ("planar", "ycbcr", (2, 2), None), ("planar", "luma", (1, 1), None),
         ("planar", "rgb", (1, 1), 7)]


@gpu
@pytest.mark.parametrize("env", ["JPGB_FORCE_GENERIC_STAGE_A", "JPGB_NO_TMA"])
@pytest.mark.parametrize("kind,color,sampling,extra", CROSS)
def test_cross_checks(env, kind, color, sampling, extra, monkeypatch):
    monkeypatch.setenv(env, "1")
    w, h, ch = 768, 96, BPP[color]
    cfg = dict(quality=90, sampling=sampling)
    imgs = [_img(w, h, ch, 52), _img(w, h, ch, 53)]
    want = [_want(w, h, ch, 52, color, cfg), _want(w, h, ch, 53, color, cfg)]
    with _context() as dev:
        if kind == "pitched":
            got = _encode_pitched(dev, color, cfg, imgs, extra)
        else:
            got = _encode_planar(dev, color, cfg, imgs, plane_stride=(w * h + extra) if extra else None)
        _check(got, want)


@gpu
@pytest.mark.parametrize("env", ["JPGB_FORCE_GENERIC_STAGE_A", "JPGB_NO_TMA"])
def test_cross_check_crop(env, monkeypatch):
    import torch
    monkeypatch.setenv(env, "1")
    W, H, cw = 700, 120, 600
    cfg = dict(quality=90, sampling=(2, 2))
    full = _img(W, H, 3, 54)
    t = torch.from_numpy(full).cuda()
    torch.cuda.synchronize()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        got = _files(dev, *enc.encode_cuda_array(t[:, 1:1 + cw], CT["rgb"][1]))
    _check(got, [oracle_encode(np.ascontiguousarray(full[:, 1:1 + cw]), cw, H, "rgb", cfg)])


# ---- image_stride 0, one path, retries ------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("plane", [False, True])
def test_image_stride_zero(plane):
    import torch
    w, h, n = 640, 120, 5
    cfg = dict(quality=90, sampling=(2, 2))
    im = _img(w, h, 3, 55)
    src = np.ascontiguousarray(im.transpose(2, 0, 1)) if plane else im
    t = torch.from_numpy(src).cuda()
    torch.cuda.synchronize()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        args = (w, h * w) if plane else (w * 3, 0)  # row_stride, plane_stride
        got = _files(dev, *enc.encode_batch_device_strided(t.data_ptr(), n, w, h, CT["rgb"][1], 0, *args))
    _check(got, [_want(w, h, 3, 55, "rgb", cfg)] * n)


@gpu
def test_one_path_launch_counts():
    """The contiguous descriptor is jpgb_encode_batch_device; pitched and planar RGB take its launches; alternating
    layouts on one context keep replaying the captured graphs."""
    w, h, n = 1920, 1080, 4
    cfg = dict(quality=90, sampling=(2, 2))
    imgs = [_img(w, h, 3, 60 + i) for i in range(n)]
    want = [_want(w, h, 3, 60 + i, "rgb", cfg) for i in range(n)]
    packed, stride = _pitched(imgs, w * 3)
    pitched, pstride = _pitched(imgs, w * 3 + 64)
    planar, ps = _planar(imgs)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        ct = CT["rgb"][1]
        calls = {
            "device": lambda: enc.encode_batch_device(packed.data_ptr(), stride, n, w, h, ct),
            "contiguous": lambda: enc.encode_batch_device_strided(packed.data_ptr(), n, w, h, ct, stride, w * 3),
            "pitched": lambda: enc.encode_batch_device_strided(pitched.data_ptr(), n, w, h, ct, pstride, w * 3 + 64),
            "planar": lambda: enc.encode_batch_device_strided(planar.data_ptr(), n, w, h, ct, 3 * ps, w, ps),
        }
        counts = {}
        for rnd in range(3):
            for name, call in calls.items():
                _check(_files(dev, *call()), want)
                counts.setdefault(name, []).append(dev.last_launch_count())
    print(counts)
    steady = counts["device"][1]
    for name, c in counts.items():
        assert c[1:] == [steady, steady], "%s: launches %r, steady %d" % (name, c, steady)
    assert counts["contiguous"][0] == steady


@gpu
@pytest.mark.parametrize("tight", ["pool", "stream", "out"])
def test_forced_retry_planar(tight, monkeypatch):
    w, h, n = 1280, 720, 3
    cfg = dict(quality=90, sampling=(2, 2))
    imgs = [_img(w, h, 3, 70 + i) for i in range(n)]
    want = [_want(w, h, 3, 70 + i, "rgb", cfg) for i in range(n)]
    buf, ps = _planar(imgs)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        counts = []
        for k in range(3):
            if k == 0:
                monkeypatch.setenv("JPGB_TIGHT_CAPS", tight)
            _check(_files(dev, *enc.encode_batch_device_strided(buf.data_ptr(), n, w, h, CT["rgb"][1], 3 * ps, w, ps)), want)
            counts.append(dev.last_launch_count())
            if k == 0:
                monkeypatch.delenv("JPGB_TIGHT_CAPS")
    assert counts[1] == counts[2] < counts[0], counts


@gpu
def test_full_size_nchw_batch_every_file():
    """96 NCHW 1080p RGB frames, q90 4:2:0, in one call: every file byte for byte."""
    import torch
    import jpeg_encoder_b200 as je
    w, h, n, distinct = 1920, 1080, 96, 6
    cfg = dict(quality=90, sampling=(2, 2))
    frames = [images.synth_frame(w, h, 3, seed=s) for s in range(distinct)]
    want = [oracle_encode(f, w, h, "rgb", cfg) for f in frames]
    order = [(i * 5 + i // 7) % distinct for i in range(n)]
    planes = [torch.from_numpy(np.ascontiguousarray(f.transpose(2, 0, 1))).cuda() for f in frames]
    t = torch.stack([planes[k] for k in order])
    torch.cuda.synchronize()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        for _ in range(2):
            _check(_files(dev, *enc.encode_cuda_array(t, je.ColorType.Rgb, channels_first=True)), [want[k] for k in order])


class _OnStream:
    """A producer's array as CUDA Array Interface v3 describes it: the data plus the stream it is being written on
    (torch's own interface is v2 and names no stream)."""

    def __init__(self, t, stream):
        self.__cuda_array_interface__ = dict(t.__cuda_array_interface__, version=3, stream=stream.cuda_stream)


@gpu
def test_wait_stream_orders_the_encode_after_the_producer():
    """Pixels written on a side stream behind a long kernel; the encode reads them through the interface's stream,
    with no host synchronize in between."""
    import torch
    w, h = 1920, 1080
    cfg = dict(quality=90, sampling=(2, 2))
    im = _img(w, h, 3, 80)
    src = torch.from_numpy(im).cuda()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        with torch.cuda.stream(side):
            dst = torch.zeros_like(src)
            torch.cuda._sleep(200_000_000)  # keeps the side stream busy well past the encode's launch
            dst.copy_(src)
            d_files, offs = enc.encode_cuda_array(_OnStream(dst, side), CT["rgb"][1])
        got = _files(dev, d_files, offs)
    _check(got, [_want(w, h, 3, 80, "rgb", cfg)])


# ---- rejections: each before anything is enqueued ------------------------------------------------------------------
def _rejected(dev, enc, call, text):
    import jpeg_encoder_b200 as je
    with pytest.raises(je.EncodingError) as e:
        call()
    assert e.value.code == 5, e.value
    assert text in dev.last_error(), dev.last_error()
    assert dev.last_launch_count() == 0


@gpu
def test_rejections():
    import torch
    w, h = 640, 100
    cfg = dict(quality=90, sampling=(2, 2))
    buf, ps = _planar([_img(w, h, 3, 90)])
    ct = CT["rgb"][1]
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        ok = lambda: enc.encode_batch_device_strided(buf.data_ptr(), 1, w, h, ct, 3 * ps, w, ps)  # noqa: E731
        _check(_files(dev, *ok()), [_want(w, h, 3, 90, "rgb", cfg)])
        assert dev.last_launch_count() > 0
        _rejected(dev, enc, lambda: enc.encode_batch_device_strided(buf.data_ptr(), 1, w, h, ct, 0, w * 3 - 1), "row_stride")
        _rejected(dev, enc, lambda: enc.encode_batch_device_strided(buf.data_ptr(), 1, w, h, ct, 0, w - 1, ps), "row_stride")
        _rejected(dev, enc, lambda: enc.encode_batch_device_strided(buf.data_ptr(), 1, w, h, ct, 0, w, w - 1), "plane_stride")
        _rejected(dev, enc, lambda: enc.encode_batch_device_strided(buf.data_ptr(), 3, w, h, ct, 1 << 63, w, ps), "64-bit")
        host = np.zeros(w * h * 3, np.uint8)
        _rejected(dev, enc, lambda: enc.encode_batch_device_strided(host.ctypes.data, 1, w, h, ct, 0, w * 3), "device or managed")
        # one byte past the end of the caching allocator's segment (the range cuMemGetAddressRange reports)
        seg = next(s for s in torch.cuda.memory_snapshot()
                   if s["address"] <= buf.data_ptr() < s["address"] + s["total_size"])
        end = seg["address"] + seg["total_size"]
        lw = 1000
        data = end - lw  # luma, one row: the last byte read is data + lw - 1 = end - 1
        _rejected(dev, enc, lambda: enc.encode_batch_device_strided(data, 1, lw + 1, 1, CT["luma"][1], 0, lw + 1), "1 bytes past the end")
        enc.encode_batch_device_strided(data, 1, lw, 1, CT["luma"][1], 0, lw)  # ends on the segment's last byte: accepted
        assert dev.last_launch_count() > 0
