"""Device images of float32, float16, bfloat16 and uint16 samples: jpgb_encode_batch_device_samples and
Encoder.encode_cuda_samples.

Stage A converts every element to the 8-bit sample clamp(rint(fadd(fmul(x, scale), offset)), 0, 255), NaN -> 0, while it
stages the pixels. Every file must be byte-identical to the oracle's encode of the image that conversion defines, here
restated in numpy. The conversion and the interface parser are checked without a GPU."""
import contextlib
import functools

import numpy as np
import pytest

import images
from cases import BPP, CT, make_encoder, oracle_encode

gpu = pytest.mark.gpu

TYPES = ["f32", "f16", "bf16", "u16"]
COLORS = ["luma", "rgb", "bgr", "rgba", "bgra"]
SAMPLINGS = [(1, 1), (2, 1), (1, 2), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)]
MODES = {  # the modes of test_device_layouts.py
    "baseline": dict(quality=90, sampling=(2, 2)),
    "optimized": dict(quality=85, sampling=(2, 1), optimize_huffman=True),
    "progressive": dict(quality=80, sampling=(2, 2), progressive_scans=4),
    "restart7": dict(quality=88, sampling=(1, 1), restart_interval=7),
}
RANGES = {"f32": (-1.0, 1.0), "f16": (0.0, 1.0), "bf16": (0.0, 1.0), "u16": (0.0, 65535.0)}


def _st(name):
    from jpeg_encoder_b200 import SampleType
    return SampleType[name.upper()]


# ---- the conversion, restated (no GPU) -----------------------------------------------------------------------------
def convert(x32, scale, offset):
    """The contract: float32 x * scale, rounded; + offset, rounded (never fused); NaN -> 0; else clamp(rint(y), 0, 255)."""
    x32 = np.asarray(x32, np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        y = np.multiply(x32, np.float32(scale), dtype=np.float32)
        y = np.add(y, np.float32(offset), dtype=np.float32)
        r = np.clip(np.rint(y), 0, 255)
    return np.where(np.isnan(y), 0, r).astype(np.uint8)


def test_conversion_known_answers():
    half = np.array([0.5, 1.5, 2.5, 254.5, 255.5, -0.5, -0.0, 0.0], np.float32)
    assert convert(half, 1.0, 0.0).tolist() == [0, 2, 2, 254, 255, 0, 0, 0]
    special = np.array([np.nan, np.inf, -np.inf, 1e30, -1e30, np.float32(1e-45), np.float32(-1e-45), np.float32(1.17e-38)], np.float32)
    assert convert(special, 255.0, 0.0).tolist() == [0, 255, 0, 255, 0, 0, 0, 0]
    assert convert(special, 127.5, 127.5).tolist() == [0, 255, 0, 255, 0, 128, 128, 128]
    from jpeg_encoder_b200 import sample_scale_offset
    s, o = sample_scale_offset(_st("f32"))
    assert convert(np.array([0, 0.5 / 255, 1.5 / 255, 0.5, 1, 1.01, -0.01], np.float32), s, o).tolist() == [0, 0, 2, 128, 255, 255, 0]
    s, o = sample_scale_offset(_st("f16"), (-1, 1))
    assert convert(np.array([-1, 0, 1, -2, 2], np.float32), s, o).tolist() == [0, 128, 255, 0, 255]
    s, o = sample_scale_offset(_st("u16"))
    assert convert(np.array([0, 128, 129, 257, 32896, 65535], np.float32), s, o).tolist() == [0, 0, 1, 1, 128, 255]


def test_conversion_equals_torch_for_the_unit_range():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.uniform(-0.1, 1.1, 200000), (np.arange(-2, 260) + 0.5) / 255, np.arange(0, 256) / 255]).astype(np.float32)
    from jpeg_encoder_b200 import sample_scale_offset
    s, o = sample_scale_offset(_st("f32"))
    want = (torch.from_numpy(x) * 255).round().clamp(0, 255).to(torch.uint8).numpy()
    assert np.array_equal(convert(x, s, o), want)


@pytest.mark.parametrize("st,rng,want", [
    ("f32", None, (255.0, 0.0)), ("bf16", None, (255.0, 0.0)), ("u16", None, (np.float32(255 / 65535), 0.0)),
    ("f16", (-1, 1), (127.5, 127.5)), ("f32", (0, 255), (1.0, 0.0)), ("u16", (0, 4095), (np.float32(255 / 4095), 0.0)),
    ("f32", (0.25, 0.75), (510.0, -127.5)), ("f32", (1, 0), (-255.0, 255.0)),
])
def test_value_range_to_scale_offset(st, rng, want):
    from jpeg_encoder_b200 import sample_scale_offset
    s, o = sample_scale_offset(_st(st), rng)
    assert (np.float32(s), np.float32(o)) == (np.float32(want[0]), np.float32(want[1]))


@pytest.mark.parametrize("rng", [(1, 1), (0, float("inf")), (float("nan"), 1), (0, 1e-300)])
def test_value_range_rejections(rng):
    from jpeg_encoder_b200 import sample_scale_offset
    with pytest.raises(ValueError):
        sample_scale_offset(_st("f32"), rng)


# ---- the interface parser (no GPU) ---------------------------------------------------------------------------------
def _iface(shape, strides=None, data=0x10000, typestr="<f4", **extra):
    d = dict(shape=shape, strides=strides, data=(data, False), typestr=typestr, version=3)
    d.update(extra)
    return d


def _layout(*a, **k):
    from jpeg_encoder_b200.encoder import _cuda_samples_layout
    return _cuda_samples_layout(*a, **k)


def test_samples_layout_typestrs():
    assert _layout(_iface((5, 40, 30, 3)), 3, False) == (_st("f32"), 0x10000, 5, 30, 40, 40 * 30 * 12, 360, 0)
    assert _layout(_iface((5, 3, 40, 30), typestr="<f2"), 3, True) == (_st("f16"), 0x10000, 5, 30, 40, 3 * 40 * 30 * 2, 60, 40 * 30 * 2)
    assert _layout(_iface((40, 30, 4), typestr="<u2"), 4, False) == (_st("u16"), 0x10000, 1, 30, 40, 0, 240, 0)
    assert _layout(_iface((1, 40, 30), typestr="<f4"), 1, True) == (_st("f32"), 0x10000, 1, 30, 40, 0, 120, 0)
    # crop t[:, :, 3:43, 5:105] of a (2, 3, 60, 120) float16 tensor: byte strides
    got = _layout(_iface((2, 3, 40, 100), (2 * 3 * 60 * 120, 2 * 60 * 120, 240, 2), data=0x20000 + 3 * 240 + 10, typestr="<f2"), 3, True)
    assert got == (_st("f16"), 0x20000 + 730, 2, 100, 40, 2 * 3 * 60 * 120, 240, 2 * 7200)


def test_samples_layout_bf16():
    bf = (_st("bf16"), 0x10000, 1, 30, 40, 0, 180, 0)
    assert _layout(_iface((40, 30, 3), typestr="<V2"), 3, False, "bf16") == bf
    assert _layout(_iface((40, 30, 3), typestr="<V2"), 3, False, _st("bf16")) == bf
    assert _layout(_iface((40, 30, 3), typestr="<V2"), 3, False, None, True) == bf
    with pytest.raises(ValueError, match="ambiguous"):
        _layout(_iface((40, 30, 3), typestr="<V2"), 3, False)
    with pytest.raises(ValueError, match="ambiguous"):
        _layout(_iface((40, 30, 3), typestr="<V2"), 3, False, "f16")
    with pytest.raises(ValueError, match="not the requested"):
        _layout(_iface((40, 30, 3), typestr="<f2"), 3, False, "bf16")


@pytest.mark.parametrize("iface,bpp,cf,what", [
    (_iface((10, 10, 3), typestr="|u1"), 3, False, "encode_cuda_array"),
    (_iface((10, 10, 3), typestr="<f8"), 3, False, "got '<f8'"),
    (_iface((10, 10, 3), typestr=">f4"), 3, False, "got '>f4'"),
    (_iface((10, 10, 3), (120, 12, 6)), 3, False, "channel stride 6"),  # not a multiple of 4 and not adjacent
    (_iface((10, 10, 3), (120, 16, 4)), 3, False, "pixel stride 16"),
    (_iface((3, 10, 10), (400, 40, 8)), 3, True, "x stride 8"),
    (_iface((10, 10, 3), (122, 12, 4)), 3, False, "row stride 122 is not a multiple"),
    (_iface((2, 10, 10, 3), (1202, 120, 12, 4)), 3, False, "image stride 1202 is not a multiple"),
    (_iface((3, 10, 10), (401, 40, 4)), 3, True, "plane stride 401 is not a multiple"),
    (_iface((10, 10, 3), typestr="<u2", data=0x10001), 3, False, "data 65537 is not a multiple"),
    (_iface((2, 10, 10, 3), (-1200, 120, 12, 4)), 3, False, "negative n stride"),
    (_iface((10, 10, 4)), 3, False, "takes 3 channels"),
    (_iface((10, 10, 3), mask=object()), 3, False, "masked"),
    (_iface((10, 30)), 3, False, "shape"),
    (_iface((1, 2, 10, 10, 3)), 3, False, "shape"),
    (_iface((10, 70000, 1)), 1, False, "above 65535"),
])
def test_samples_layout_rejections(iface, bpp, cf, what):
    with pytest.raises(ValueError, match=what):
        _layout(iface, bpp, cf)


def test_u8_layout_unchanged():
    from jpeg_encoder_b200.encoder import _cuda_array_layout
    assert _cuda_array_layout(_iface((5, 3, 40, 30), typestr="|u1"), 3, True) == (0x10000, 5, 30, 40, 3 * 40 * 30, 30, 40 * 30)
    with pytest.raises(ValueError, match="uint8"):
        _cuda_array_layout(_iface((10, 10, 3), typestr="<f4"), 3, False)


# ---- GPU helpers ---------------------------------------------------------------------------------------------------
_TORCH = {"f32": "float32", "f16": "float16", "bf16": "bfloat16", "u16": "uint16"}


@functools.lru_cache(maxsize=None)
def _u8(w, h, ch, seed):
    return np.ascontiguousarray(images.photo_like(w, h, ch, seed=seed).reshape(h, w, ch))


def _samples(w, h, ch, seed, st, rng=None):
    """(H, W, C) CPU torch tensor of type `st`: a photo-like image scaled into the value range, with sub-step noise"""
    import torch
    lo, hi = rng or RANGES[st]
    u8 = _u8(w, h, ch, seed).astype(np.float64)
    noise = np.random.default_rng(seed).uniform(-0.6, 0.6, u8.shape)
    x = lo + (u8 + noise) * (hi - lo) / 255.0
    if st == "u16":
        return torch.from_numpy(np.clip(np.rint(x), 0, 65535).astype(np.uint16).astype(np.int32)).to(torch.uint16)
    return torch.from_numpy(x.astype(np.float32)).to(getattr(torch, _TORCH[st]))


def _converted(x, st, rng=None):
    """the uint8 image the contract defines for the CPU tensor x (any shape)"""
    from jpeg_encoder_b200 import sample_scale_offset
    s, o = sample_scale_offset(_st(st), rng or RANGES[st])
    import torch
    x32 = x.to(torch.int32).numpy() if st == "u16" else x.float().numpy()
    out = convert(x32, s, o)
    return out


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


def _want(u8, color, cfg):
    """oracle files of (N, H, W, C) uint8 images"""
    n, h, w, _ = u8.shape
    return [oracle_encode(np.ascontiguousarray(u8[i]), w, h, color, cfg) for i in range(n)]


def _encode(dev, cfg, x, color, st, layout, rng=None):
    """encode_cuda_samples of the (N, H, W, C) CPU tensor x, uploaded in `layout` (nhwc / nchw)"""
    t = (x.permute(0, 3, 1, 2) if layout == "nchw" else x).contiguous().cuda()
    enc = make_encoder(cfg, dev)
    return _files(dev, *enc.encode_cuda_samples(t, CT[color][1], channels_first=layout == "nchw", value_range=rng or RANGES[st]))


def _run(cfg, color, st, layout, w, h, n=1, seed=1):
    import torch
    ch = BPP[color]
    x = torch.stack([_samples(w, h, ch, seed + i, st) for i in range(n)])
    with _context() as dev:
        got = _encode(dev, cfg, x, color, st, layout)
    _check(got, _want(_converted(x, st), color, cfg))


# ---- the matrix ------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("color", COLORS)
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
@pytest.mark.parametrize("st", TYPES)
def test_types_layouts_colors(st, layout, color):
    _run(MODES["baseline"], color, st, layout, 520, 72, n=2, seed=10)


@gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("st", TYPES)
def test_modes(st, mode):
    _run(MODES[mode], "rgb", st, "nhwc" if mode in ("baseline", "progressive") else "nchw", 320, 72, seed=20)


@gpu
@pytest.mark.parametrize("sampling", SAMPLINGS)
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
@pytest.mark.parametrize("st", ["f32", "bf16"])
def test_samplings(st, layout, sampling):
    _run(dict(quality=87, sampling=sampling), "rgb", st, layout, 544, 100, seed=30)


@gpu
@pytest.mark.parametrize("size", [(1, 1), (17, 9), (255, 2), (513, 31)])
@pytest.mark.parametrize("color,st,layout", [("rgb", "f32", "nhwc"), ("rgba", "u16", "nhwc"), ("bgr", "f16", "nchw"), ("luma", "bf16", "nhwc")])
def test_ragged_sizes(color, st, layout, size):
    _run(dict(quality=90, sampling=(2, 2)), color, st, layout, *size, seed=40)


@gpu
@pytest.mark.parametrize("st", TYPES)
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_row_pitch_not_16_bytes(st, layout):
    """rows `pad` elements longer than the image (a multiple of the element size, not of 16 bytes), junk NaN in the pad"""
    import torch
    w, h, n, pad = 300, 50, 2, 3
    cfg = dict(quality=90, sampling=(2, 2))
    x = torch.stack([_samples(w, h, 3, 50 + i, st) for i in range(n)])
    junk = 0 if st == "u16" else float("nan")
    if layout == "nhwc":
        buf = torch.full((n, h, (w + pad) * 3), junk, dtype=x.dtype)
        buf[:, :, :w * 3] = x.reshape(n, h, w * 3)
        view = buf.cuda()[:, :, :w * 3].view(n, h, w, 3)
    else:
        buf = torch.full((n, 3, h, w + pad), junk, dtype=x.dtype)
        buf[..., :w] = x.permute(0, 3, 1, 2)
        view = buf.cuda()[..., :w]
    es = x.element_size()
    assert (view.stride(-2 if layout == "nchw" else 1) * es) % 16 != 0
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        got = _files(dev, *enc.encode_cuda_samples(view, CT["rgb"][1], channels_first=layout == "nchw", value_range=RANGES[st]))
    _check(got, _want(_converted(x, st), "rgb", cfg))


@gpu
@pytest.mark.parametrize("x0", [1, 3, 16])
@pytest.mark.parametrize("st,layout", [("f32", "nhwc"), ("f16", "nchw"), ("bf16", "nhwc"), ("u16", "nchw")])
def test_crops(st, layout, x0):
    import torch
    n, H, W, y0, y1, cw = 2, 120, 700, 5, 110, 600
    cfg = dict(quality=90, sampling=(2, 2))
    full = torch.stack([_samples(W, H, 3, 60 + i, st) for i in range(n)])
    crop = full[:, y0:y1, x0:x0 + cw]
    t = full.permute(0, 3, 1, 2).contiguous().cuda()[:, :, y0:y1, x0:x0 + cw] if layout == "nchw" else full.cuda()[:, y0:y1, x0:x0 + cw]
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        got = _files(dev, *enc.encode_cuda_samples(t, CT["rgb"][1], channels_first=layout == "nchw", value_range=RANGES[st]))
    _check(got, _want(_converted(crop.contiguous(), st), "rgb", cfg))


@gpu
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_image_stride_zero(layout):
    w, h, n = 640, 96, 3
    cfg = dict(quality=90, sampling=(2, 2))
    x = _samples(w, h, 3, 70, "f32")
    src = (x.permute(2, 0, 1) if layout == "nchw" else x).contiguous().cuda()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        rs, ps = (w * 4, h * w * 4) if layout == "nchw" else (w * 12, 0)
        got = _files(dev, *enc.encode_batch_device_samples(src.data_ptr(), n, w, h, CT["rgb"][1], _st("f32"), 0, rs, ps, RANGES["f32"]))
    _check(got, _want(_converted(x[None], "f32"), "rgb", cfg) * n)


@gpu
@pytest.mark.parametrize("st", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("layout", ["nhwc", "nchw"])
def test_special_values(st, layout):
    """exact half-way values, NaN, +-inf and values far outside the range, scattered over the image"""
    import torch
    w, h = 520, 72
    cfg = dict(quality=90, sampling=(2, 1))
    x = _samples(w, h, 3, 80, st, (0.0, 255.0))[None].clone()
    rng = np.random.default_rng(81)
    specials = torch.tensor([0.5, 1.5, 2.5, 127.5, 253.5, 254.5, 255.5, -0.5, -0.0, float("nan"), float("inf"), float("-inf"),
                             1e4, -1e4, 60000.0, 3e38 if st != "f16" else 65504.0], dtype=torch.float32).to(x.dtype)
    flat = x.view(-1)
    idx = torch.from_numpy(rng.choice(flat.numel(), flat.numel() // 5, replace=False))
    flat[idx] = specials[torch.from_numpy(rng.integers(0, len(specials), len(idx)))]
    u8 = _converted(x, st, (0.0, 255.0))
    assert (u8 == 0).any() and (u8 == 255).any()
    with _context() as dev:
        got = _encode(dev, cfg, x, "rgb", st, layout, (0.0, 255.0))
    _check(got, _want(u8, "rgb", cfg))


@gpu
@pytest.mark.parametrize("color", ["rgba", "bgra"])
def test_junk_never_matters(color):
    """NaN and random junk in the row pitch, in the alpha channel or plane, and between images change no byte"""
    import torch
    w, h, n, pitch, gap = 600, 80, 2, 600 * 4 + 12, 1024
    cfg = dict(quality=90, sampling=(2, 2))
    x = torch.stack([_samples(w, h, 4, 90 + i, "f32") for i in range(n)])
    want = _want(_converted(x, "f32"), color, cfg)
    g = torch.Generator().manual_seed(91)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        for junk in ("nan", "random"):
            fill = (lambda k: torch.full((k,), float("nan"))) if junk == "nan" else (lambda k: torch.randn(k, generator=g) * 1e6)
            # packed rows of `pitch` elements, images h * pitch + gap elements apart
            istride = h * pitch + gap
            buf = fill(n * istride)
            for i in range(n):
                rows = buf[i * istride:i * istride + h * pitch].view(h, pitch)
                rows[:, :w * 4] = x[i].reshape(h, w * 4)
                rows[:, 3:w * 4:4] = fill(h * w).view(h, w)  # alpha
            d = buf.cuda()
            _check(_files(dev, *enc.encode_batch_device_samples(d.data_ptr(), n, w, h, CT[color][1], _st("f32"), istride * 4, pitch * 4,
                                                                          value_range=RANGES["f32"])), want)
            # planes `ps` elements apart (junk between them), the alpha plane junk
            ps = h * w + 256
            buf = fill(n * 4 * ps)
            for i in range(n):
                for c in range(3):
                    buf[(i * 4 + c) * ps:(i * 4 + c) * ps + h * w] = x[i, ..., c].reshape(-1)
            d = buf.cuda()
            _check(_files(dev, *enc.encode_batch_device_samples(d.data_ptr(), n, w, h, CT[color][1], _st("f32"), 4 * ps * 4, w * 4, ps * 4,
                                                                          value_range=RANGES["f32"])), want)


@gpu
@pytest.mark.parametrize("env", ["JPGB_FORCE_GENERIC_STAGE_A", "JPGB_NO_TMA"])
@pytest.mark.parametrize("color,st,layout,sampling", [("rgb", "f32", "nhwc", (2, 2)), ("bgra", "bf16", "nhwc", (1, 1)),
                                                      ("rgba", "u16", "nchw", (2, 1)), ("bgr", "f16", "nchw", (4, 2)),
                                                      ("luma", "f32", "nchw", (1, 1))])
def test_cross_checks(env, color, st, layout, sampling, monkeypatch):
    monkeypatch.setenv(env, "1")
    _run(dict(quality=90, sampling=sampling), color, st, layout, 777, 61, n=2, seed=100)


@gpu
@pytest.mark.parametrize("tight", ["pool", "stream", "out"])
def test_forced_retry(tight, monkeypatch):
    import torch
    w, h, n = 1280, 720, 3
    cfg = dict(quality=90, sampling=(2, 2))
    x = torch.stack([_samples(w, h, 3, 110 + i, "bf16") for i in range(n)])
    want = _want(_converted(x, "bf16"), "rgb", cfg)
    t = x.permute(0, 3, 1, 2).contiguous().cuda()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        counts = []
        for k in range(3):
            if k == 0:
                monkeypatch.setenv("JPGB_TIGHT_CAPS", tight)
            _check(_files(dev, *enc.encode_cuda_samples(t, CT["rgb"][1], channels_first=True)), want)
            counts.append(dev.last_launch_count())
            if k == 0:
                monkeypatch.delenv("JPGB_TIGHT_CAPS")
    assert counts[1] == counts[2] < counts[0], counts


@gpu
def test_launch_count_equals_the_u8_entry():
    """one stage A launch: every call takes as many launches as the uint8 strided entry in the same layout"""
    import torch
    w, h, n = 1920, 1080, 2
    cfg = dict(quality=90, sampling=(2, 2))
    x = torch.stack([_samples(w, h, 3, 120 + i, "f16") for i in range(n)])
    u8 = _converted(x, "f16")
    want = _want(u8, "rgb", cfg)
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        counts = {}
        for layout in ("nhwc", "nchw"):
            cf = layout == "nchw"
            t8 = torch.from_numpy(u8).cuda()
            t8 = t8.permute(0, 3, 1, 2).contiguous() if cf else t8
            tx = (x.permute(0, 3, 1, 2) if cf else x).contiguous().cuda()
            for rnd in range(2):
                _check(_files(dev, *enc.encode_cuda_array(t8, CT["rgb"][1], channels_first=cf)), want)
                counts.setdefault(layout + "_u8", []).append(dev.last_launch_count())
                _check(_files(dev, *enc.encode_cuda_samples(tx, CT["rgb"][1], channels_first=cf)), want)
                counts.setdefault(layout + "_f16", []).append(dev.last_launch_count())
    print(counts)
    for layout in ("nhwc", "nchw"):
        assert counts[layout + "_f16"][1] == counts[layout + "_u8"][1], counts


def _rejected(dev, call, text):
    import jpeg_encoder_b200 as je
    with pytest.raises(je.EncodingError) as e:
        call()
    assert e.value.code == 5, e.value
    assert text in dev.last_error(), dev.last_error()
    assert dev.last_launch_count() == 0


@gpu
def test_rejections():
    import torch
    import ctypes as C
    from jpeg_encoder_b200.encoder import _DeviceImages, _SampleFormat
    w, h = 640, 100
    cfg = dict(quality=90, sampling=(2, 2))
    x = _samples(w, h, 3, 130, "f32")
    t = x.permute(2, 0, 1).contiguous().cuda()
    ps = h * w * 4
    ct, f32 = CT["rgb"][1], _st("f32")
    with _context() as dev:
        enc = make_encoder(cfg, dev)

        def raw(ptr=t.data_ptr(), n=1, color=ct, st=int(f32), scale=255.0, offset=0.0, istride=3 * ps, rs=w * 4, pls=ps, fmt=True):
            p = enc._params(w, h, color)
            im = _DeviceImages(ptr, istride, rs, pls)
            f = _SampleFormat(st, scale, offset)
            d_files, offs = C.c_void_p(), (C.c_uint64 * (n + 1))()
            rc = dev.lib.jpgb_encode_batch_device_samples(dev.handle, C.byref(p), C.byref(im), C.byref(f) if fmt else None, n, C.byref(d_files), offs)
            if rc:
                enc._raise(rc)
            return d_files.value, list(offs)

        _check(_files(dev, *raw()), _want(_converted(x[None], "f32", (0, 1)), "rgb", cfg))
        assert dev.last_launch_count() > 0
        _rejected(dev, lambda: raw(fmt=False), "null argument")
        _rejected(dev, lambda: raw(n=0), "null argument")
        _rejected(dev, lambda: raw(st=0), "uint8")
        _rejected(dev, lambda: raw(st=5), "unknown sample type")
        for bad in ("ycbcr", "cmyk", "cmyk_as_ycck", "ycck"):
            _rejected(dev, lambda: raw(color=CT[bad][1]), "Luma, Rgb")
        for s, o in ((float("inf"), 0.0), (float("nan"), 0.0), (255.0, float("-inf")), (255.0, float("nan"))):
            _rejected(dev, lambda: raw(scale=s, offset=o), "finite")
        _rejected(dev, lambda: raw(ptr=t.data_ptr() + 2), "multiples of the element size")
        _rejected(dev, lambda: raw(rs=w * 4 + 2), "multiples of the element size")
        _rejected(dev, lambda: raw(pls=ps + 2), "multiples of the element size")
        _rejected(dev, lambda: raw(istride=3 * ps + 2), "multiples of the element size")
        _rejected(dev, lambda: raw(rs=w * 4 - 4), "row_stride")
        _rejected(dev, lambda: raw(pls=w * 4 - 4), "plane_stride")
        _rejected(dev, lambda: raw(n=3, istride=1 << 63), "64-bit")
        host = np.zeros(w * h * 3, np.float32)
        _rejected(dev, lambda: raw(ptr=host.ctypes.data), "device or managed")
        # extent in elements: a float32 luma row of lw elements ending one element past the allocator's segment
        seg = next(s for s in torch.cuda.memory_snapshot() if s["address"] <= t.data_ptr() < s["address"] + s["total_size"])
        end = seg["address"] + seg["total_size"]
        lw = 1000
        data = end - lw * 4
        luma = CT["luma"][1]
        _rejected(dev, lambda: enc.encode_batch_device_samples(data, 1, lw + 1, 1, luma, f32, 0, (lw + 1) * 4), "4 bytes past the end")
        enc.encode_batch_device_samples(data, 1, lw, 1, luma, f32, 0, lw * 4)  # ends on the segment's last byte: accepted
        assert dev.last_launch_count() > 0


# ---- full size -------------------------------------------------------------------------------------------------------
@gpu
def test_full_size_f32_nchw_batch_every_file():
    """96 NCHW 1080p float32 RGB frames in [0, 1], q90 4:2:0, in one call: every file byte for byte"""
    import torch
    w, h, n, distinct = 1920, 1080, 96, 6
    cfg = dict(quality=90, sampling=(2, 2))
    rng = np.random.default_rng(140)
    frames = [torch.from_numpy(images.synth_frame(w, h, 3, seed=s).astype(np.float32) / 255 + rng.uniform(-0.002, 0.002, (h, w, 3)).astype(np.float32))
              for s in range(distinct)]
    want = [_want(_converted(f[None], "f32", (0, 1)), "rgb", cfg)[0] for f in frames]
    order = [(i * 5 + i // 7) % distinct for i in range(n)]
    planes = [f.permute(2, 0, 1).contiguous().cuda() for f in frames]
    t = torch.stack([planes[k] for k in order])
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        _check(_files(dev, *enc.encode_cuda_samples(t, CT["rgb"][1], channels_first=True)), [want[k] for k in order])


@gpu
def test_8192_bf16_nhwc():
    import torch
    w = h = 8192
    cfg = dict(quality=90, sampling=(2, 2))
    x = _samples(w, h, 3, 150, "bf16")[None]
    with _context() as dev:
        got = _encode(dev, cfg, x, "rgb", "bf16", "nhwc")
    _check(got, _want(_converted(x, "bf16"), "rgb", cfg))
