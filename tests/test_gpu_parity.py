"""Parity tests proper: the CUDA path through the C ABI against the CPU oracle, byte for byte."""
import io

import numpy as np
import pytest
from PIL import Image

import images
from cases import BPP, CT, gpu_encode, make_encoder, oracle_encode
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


def _img(color, w, h, seed=1):
    ch = BPP[color]
    return images.photo_like(w, h, ch, seed=seed)


def _same(color, w, h, cfg, img=None, seed=1):
    img = _img(color, w, h, seed) if img is None else img
    got = gpu_encode(img, w, h, color, cfg)
    want = oracle_encode(img, w, h, color, cfg)
    if got != want:
        n = min(len(got), len(want))
        first = next((i for i in range(n) if got[i] != want[i]), n)
        pytest.fail("bytes differ for %s %dx%d %r: len %d vs %d, first diff at %d" % (color, w, h, cfg, len(got), len(want), first))
    return got


# ---- committed fixtures: no oracle code runs in this test ----------------------------------------
def test_committed_file_hashes():
    """GPU file bytes against tests/golden/oracle_jpegs.json (SHA-256 written by make_golden.py in the build container)."""
    import hashlib, json, os, sys
    gold = os.path.join(os.path.dirname(__file__), "golden")
    sys.path.insert(0, gold)
    import make_golden
    want = json.load(open(os.path.join(gold, "oracle_jpegs.json")))
    for name, maker, size, color, cfg in make_golden.golden_matrix():
        data = gpu_encode(getattr(images, maker)(*size), size[0], size[1], color, cfg)
        assert (hashlib.sha256(data).hexdigest(), len(data)) == (want[name]["sha256"], want[name]["len"]), name


# ---- stage A on its own: coefficients bit-exact --------------------------------------------------
@pytest.mark.parametrize("optimize", [False, True])  # interleaved (MCU-ordered buffer) / sequential (raster of the true grids)
@pytest.mark.parametrize("color,sampling", [("rgb", (2, 2)), ("rgb", (1, 1)), ("rgb", (4, 1)), ("rgb", (2, 4)), ("luma", (1, 1)),
                                            ("cmyk_as_ycck", (1, 1)), ("cmyk", (2, 2)), ("bgra", (2, 1)), ("ycck", (1, 2))])
def test_stage_a_coefficients(color, sampling, optimize):
    import torch
    import jpeg_encoder_b200 as je
    w, h = 203, 131
    img = _img(color, w, h)
    cfg = dict(quality=85, sampling=sampling, optimize_huffman=optimize)
    enc = make_encoder(cfg)
    lay = enc.coef_layout(w, h, CT[color][1])
    d_px = torch.from_numpy(img.reshape(-1).copy()).cuda()
    d_coef = torch.full((lay.blocks_per_image * 64,), 12345, dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    enc.stage_a_device(d_px.data_ptr(), d_px.numel(), 1, d_coef.data_ptr(), w, h, CT[color][1])
    je.default_device(0)  # same context
    import ctypes
    # the context runs on its own stream: synchronise the device before reading
    torch.cuda.synchronize()
    got = d_coef.cpu().numpy().reshape(-1, 64)
    want = orc.coefficients(img, w, h, CT[color][0], **cfg)
    seen = np.zeros(lay.blocks_per_image, bool)
    for c in range(lay.n_components):
        pw, ph = lay.blocks_w[c], lay.blocks_h[c]
        assert pw * ph == want[c].shape[0]  # the oracle holds the MCU-padded grid of every component, raster order
        by, bx = np.divmod(np.arange(pw * ph), pw)
        if lay.mcu_order:  # interleaved scan: blocks in coding order (include/jpegenc_b200.h, jpgb_coef_layout)
            H, V = lay.comp_h[c], lay.comp_v[c]
            idx = ((by // V) * lay.mcu_cols + bx // H) * lay.blocks_per_mcu + lay.slot_base[c] + (by % V) * H + bx % H
            keep = np.ones(pw * ph, bool)
        else:              # raster of the true grid; MCU padding blocks are not stored
            keep = (by < lay.true_h[c]) & (bx < lay.true_w[c])
            idx = lay.block_offset[c] + by * lay.true_w[c] + bx
        np.testing.assert_array_equal(got[idx[keep]], want[c][keep], err_msg="component %d" % c)
        assert not seen[idx[keep]].any()
        seen[idx[keep]] = True
    assert seen.all(), "every block of the buffer belongs to exactly one component position"


def test_generic_and_fast_stage_a_kernels_agree(monkeypatch):
    """Formats served by the fast kernel must also be exact through the generic one (and vice versa)."""
    for color, sampling in (("rgb", (2, 2)), ("bgr", (2, 1)), ("rgba", (1, 2)), ("bgra", (1, 1)), ("luma", (1, 1)),
                            ("cmyk_as_ycck", (2, 2)), ("cmyk_as_ycck", (1, 1)), ("ycbcr", (2, 2)), ("ycbcr", (1, 1)), ("ycbcr", (2, 1)),
                            ("ycbcr", (1, 2)), ("ycck", (2, 2)), ("ycck", (1, 1)), ("ycck", (2, 1)), ("cmyk", (2, 2)), ("cmyk", (1, 1)),
                            ("cmyk", (2, 1)), ("cmyk", (1, 2)),
                            # factors of 4 (sequential scans): four 1x1 components' worth of lanes share a chroma task
                            ("rgb", (4, 1)), ("rgb", (4, 2)), ("rgb", (1, 4)), ("rgb", (2, 4)), ("bgra", (4, 2)), ("cmyk_as_ycck", (4, 1)),
                            ("cmyk_as_ycck", (2, 4)), ("ycbcr", (4, 1)), ("ycbcr", (1, 4)), ("ycck", (4, 2)), ("cmyk", (4, 1)), ("cmyk", (2, 4))):
        cfg = dict(quality=83, sampling=sampling)
        img = _img(color, 333, 77, seed=11)
        want = oracle_encode(img, 333, 77, color, cfg)
        assert gpu_encode(img, 333, 77, color, cfg) == want
        monkeypatch.setenv("JPGB_FORCE_GENERIC_STAGE_A", "1")
        assert gpu_encode(img, 333, 77, color, cfg) == want
        monkeypatch.delenv("JPGB_FORCE_GENERIC_STAGE_A")


# ---- the reference's own end-to-end cases (src/lib.rs:188-553), now compared on bytes -----------
REF_RGB_CASES = {
    "rgb_100": dict(quality=100),
    "rgb_80": dict(quality=80),
    "custom_q_table": dict(quality=100, qtables=([1] * 64, [1] * 64)),
    "2_2": dict(quality=100, sampling=(2, 2)),
    "2_1": dict(quality=100, sampling=(2, 1)),
    "4_1": dict(quality=100, sampling=(4, 1)),
    "1_1": dict(quality=100, sampling=(1, 1)),
    "1_4": dict(quality=100, sampling=(1, 4)),
    "progressive": dict(quality=100, sampling=(2, 1), progressive_scans=4),
    "optimized": dict(quality=100, sampling=(2, 2), optimize_huffman=True),
    "optimized_progressive": dict(quality=100, sampling=(2, 1), progressive_scans=4, optimize_huffman=True),
    "restart": dict(quality=100, restart_interval=32),
    "restart_4_1": dict(quality=100, sampling=(4, 1), restart_interval=32),
    "restart_progressive": dict(quality=85, progressive_scans=4, restart_interval=32),
    "app_segment": dict(quality=100, app_segments=[(15, b"HOHOHO\0")]),
}


@pytest.mark.parametrize("name", sorted(REF_RGB_CASES))
def test_reference_rgb_cases(name):
    jpg = _same("rgb", 258, 128, REF_RGB_CASES[name], img=images.ref_img_rgb())
    im = Image.open(io.BytesIO(jpg))
    im.load()
    assert im.size == (258, 128)
    assert np.abs(np.asarray(im).astype(int) - images.ref_img_rgb().astype(int)).max() < 20  # src/lib.rs:176-185


def test_reference_other_color_cases():
    _same("luma", 258, 128, dict(quality=100), img=images.ref_img_gray())
    _same("rgba", 258, 128, dict(quality=80), img=images.ref_img_rgba())
    _same("cmyk", 258, 192, dict(quality=100), img=images.ref_img_cmyk())
    _same("cmyk_as_ycck", 258, 192, dict(quality=100), img=images.ref_img_cmyk())
    data = np.array([[[0xFB, 0x15, 0x15]]], np.uint8)  # src/lib.rs:541-553
    _same("rgb", 1, 1, dict(quality=100, sampling=(2, 2), optimize_huffman=True), img=data)


def test_icc_profile():
    import jpeg_encoder_b200 as je
    icc = bytes(i % 255 for i in range(128 * 1024))
    enc = je.Encoder(100)
    enc.add_icc_profile(icc)
    img = images.ref_img_rgb()
    jpg = enc.encode(img, 258, 128, je.ColorType.Rgb)
    maxc = 65535 - 2 - 12 - 2
    chunks = [icc[i:i + maxc] for i in range(0, len(icc), maxc)]
    segs = [(2, b"ICC_PROFILE\0" + bytes([i + 1, len(chunks)]) + c) for i, c in enumerate(chunks)]
    assert jpg == orc.encode(img, 258, 128, orc.RGB, quality=100, app_segments=segs)
    assert Image.open(io.BytesIO(jpg)).info.get("icc_profile") == icc


# ---- the wider matrix ----------------------------------------------------------------------------
@pytest.mark.parametrize("color", sorted(CT))
@pytest.mark.parametrize("mode", ["baseline", "optimized", "progressive", "restart7", "opt_prog_restart"])
def test_color_types_by_mode(color, mode):
    cfg = dict(quality=77, sampling=(2, 2))
    if mode == "optimized":
        cfg["optimize_huffman"] = True
    elif mode == "progressive":
        cfg["progressive_scans"] = 4
    elif mode == "restart7":
        cfg["restart_interval"] = 7
    elif mode == "opt_prog_restart":
        cfg.update(optimize_huffman=True, progressive_scans=6, restart_interval=5)
    _same(color, 150, 91, cfg, seed=hash((color, mode)) % 1000)


@pytest.mark.parametrize("sampling", [(1, 1), (1, 2), (2, 1), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)])
@pytest.mark.parametrize("color", ["rgb", "cmyk", "ycck"])
def test_sampling_factors(color, sampling):
    for extra in (dict(), dict(restart_interval=3), dict(progressive_scans=3, restart_interval=11)):
        _same(color, 97, 75, dict(quality=60, sampling=sampling, **extra))


@pytest.mark.parametrize("w,h", [(1, 1), (7, 3), (8, 8), (9, 17), (16, 16), (17, 1), (1, 33), (255, 2), (513, 31), (640, 480)])
def test_ragged_sizes(w, h):
    for cfg in (dict(quality=90, sampling=(2, 2)), dict(quality=50, sampling=(1, 1), optimize_huffman=True),
                dict(quality=95, sampling=(4, 2), progressive_scans=2)):
        _same("rgb", w, h, cfg, seed=w * 1000 + h)
        _same("luma", w, h, cfg, seed=w * 1000 + h + 1)


@pytest.mark.parametrize("kind", range(9))
def test_preset_quantization_tables(kind):
    _same("rgb", 120, 80, dict(quality=70, qtables=(kind, (kind + 3) % 9)))


def test_custom_tables_including_truncated_dqt():
    rng = np.random.default_rng(5)
    t1 = rng.integers(1, 256, 64).tolist()
    t2 = rng.integers(1, 3000, 64).tolist()  # > 255: DQT byte is truncated, quantizer uses the full value (Q10)
    t2[0] = 0  # clamped to 1
    _same("rgb", 160, 120, dict(quality=33, qtables=(t1, t2), sampling=(2, 1)))
    _same("cmyk_as_ycck", 64, 48, dict(quality=95, qtables=(t1, t1), sampling=(1, 1)))


@pytest.mark.parametrize("q", [1, 10, 49, 50, 51, 89, 90, 100])
def test_quality_sweep_default_sampling(q):
    _same("rgb", 100, 60, dict(quality=q, sampling=None))


@pytest.mark.parametrize("scans", [2, 3, 4, 5, 16, 33, 34, 63, 64])
def test_progressive_scan_counts(scans):
    _same("rgb", 64, 40, dict(quality=80, sampling=(2, 2), progressive_scans=scans))
    _same("ycck", 40, 24, dict(quality=100, sampling=(1, 1), progressive_scans=scans, restart_interval=2))


@pytest.mark.parametrize("ri", [1, 2, 8, 9, 64, 1000, 65535])
def test_restart_intervals(ri):
    _same("rgb", 200, 120, dict(quality=85, sampling=(2, 2), restart_interval=ri))
    _same("rgb", 200, 120, dict(quality=85, sampling=(2, 2), restart_interval=ri, optimize_huffman=True))  # Q18


def test_noise_and_extremes():
    rng = np.random.default_rng(9)
    noise = rng.integers(0, 256, (96, 136, 3), dtype=np.uint8)
    for cfg in (dict(quality=100, sampling=(1, 1)), dict(quality=100, sampling=(2, 2), optimize_huffman=True),
                dict(quality=100, qtables=([1] * 64, [1] * 64), progressive_scans=4)):
        _same("rgb", 136, 96, cfg, img=noise)
    for v in (0, 255):
        _same("rgb", 40, 40, dict(quality=90, sampling=(2, 2)), img=np.full((40, 40, 3), v, np.uint8))
    cb = ((np.indices((64, 64)).sum(axis=0) % 2) * 255).astype(np.uint8)
    _same("luma", 64, 64, dict(quality=100), img=cb)
    _same("rgb", 64, 64, dict(quality=100, sampling=(1, 1)), img=np.stack([cb, 255 - cb, cb], -1))
    ff = images.bench_img(320, 200)  # many 0xFF bytes in the entropy stream
    _same("rgb", 320, 200, dict(quality=100, sampling=(1, 1)), img=ff)


def test_maximum_dimensions():
    """u16 limits of the API (src/encoder.rs:440-446): 65535 wide and 65535 tall."""
    for w, h in ((65535, 9), (9, 65535)):
        _same("rgb", w, h, dict(quality=80, sampling=(2, 2)), seed=3)
        _same("luma", w, h, dict(quality=80, progressive_scans=3, restart_interval=999), seed=4)
        _same("cmyk", w, h, dict(quality=80, sampling=(4, 2), optimize_huffman=True), seed=5)


def test_density_and_trailing_bytes():
    _same("rgb", 33, 21, dict(quality=90, density=(1, 300, 300)))
    _same("rgb", 33, 21, dict(quality=90, density=(2, 118, 59)))
    img = _img("rgb", 33, 21)
    extra = np.concatenate([img.reshape(-1), np.arange(77, dtype=np.uint8)])
    assert gpu_encode(extra, 33, 21, "rgb", dict(quality=90)) == oracle_encode(img, 33, 21, "rgb", dict(quality=90))


def test_errors_mirror_reference():
    import jpeg_encoder_b200 as je
    with pytest.raises(je.EncodingError) as e:
        je.Encoder(90).encode(np.zeros(10, np.uint8), 4, 4, je.ColorType.Rgb)
    assert e.value.kind == "BadImageData"
    with pytest.raises(je.EncodingError) as e:
        je.Encoder(90).encode(np.zeros(10, np.uint8), 0, 4, je.ColorType.Rgb)
    assert e.value.kind == "ZeroImageDimensions"


def test_sink_and_batch():
    import jpeg_encoder_b200 as je
    img = _img("rgb", 120, 72)
    cfg = dict(quality=88, sampling=(2, 2))
    buf = io.BytesIO()
    make_encoder(cfg).encode_to(buf, img, 120, 72, je.ColorType.Rgb)
    assert buf.getvalue() == oracle_encode(img, 120, 72, "rgb", cfg)
    imgs = [_img("rgb", 120, 72, seed=s) for s in range(7)]
    for c in (cfg, dict(quality=70, sampling=(2, 2), optimize_huffman=True, restart_interval=9), dict(quality=70, progressive_scans=4)):
        outs = make_encoder(c).encode_batch(imgs, 120, 72, je.ColorType.Rgb)
        assert len(outs) == 7
        for im, o in zip(imgs, outs):
            assert o == oracle_encode(im, 120, 72, "rgb", c)


# ---- BASELINE.json configurations at full size (oracle finishes in seconds up to C2) -------------
def test_config1_1080p_baseline():
    _same("rgb", 1920, 1080, dict(quality=90, sampling=(2, 2)), img=images.bench_img(1920, 1080))
    _same("rgb", 1920, 1080, dict(quality=90, sampling=(2, 2)), img=images.photo_like(1920, 1080, 3))


def test_config2_4096_optimized_restart64():
    _same("rgb", 4096, 4096, dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=64),
          img=images.photo_like(4096, 4096, 3, seed=2))


def test_config4_small_scale_gray_and_ycck_custom_tables():
    rng = np.random.default_rng(4)
    t = rng.integers(1, 64, 64).tolist()
    _same("luma", 2048, 1024, dict(quality=95, sampling=(1, 1), qtables=(t, t)), img=images.photo_like(2048, 1024, 1))
    _same("cmyk_as_ycck", 1024, 768, dict(quality=95, sampling=(1, 1), qtables=(t, t)), img=images.photo_like(1024, 768, 4))


def test_config5_progressive_420_medium():
    _same("rgb", 2048, 2048, dict(quality=90, sampling=(2, 2), progressive_scans=4, restart_interval=2048),
          img=images.photo_like(2048, 2048, 3, seed=6))


# ---- BASELINE.json configurations 3, 4 and 5 at FULL size ------------------------------------------
def _bench_custom_table():
    import bench
    return bench.custom_table()


def _torch_frame(w, h, ch, seed):
    """images.synth_frame evaluated on the GPU (seconds instead of minutes at 8192^2 and above), as a host array."""
    import torch
    rows = max(1, (1 << 27) // (w * ch))  # bounded temporaries: ~128 MB of output per slab (int64 intermediates are 8x)
    parts = [images.synth_frame_torch(w, h, ch, seed=seed, row0=r, rows=min(rows, h - r), device="cuda").cpu() for r in range(0, h, rows)]
    torch.cuda.empty_cache()
    return torch.cat(parts).numpy()


def test_config3_device_batch_every_file():
    """jpgb_encode_batch_device (the timed path of bench.py): every file of a 96-frame batch, byte for byte."""
    import torch
    import jpeg_encoder_b200 as je
    w, h, n, distinct = 1920, 1080, 96, 6
    cfg = dict(quality=90, sampling=(2, 2))
    frames = [images.synth_frame(w, h, 3, seed=s) for s in range(distinct)]
    want = [oracle_encode(f, w, h, "rgb", cfg) for f in frames]
    stride = (w * h * 3 + 255) & ~255
    d_in = torch.zeros(n * stride, dtype=torch.uint8, device="cuda")
    order = [(i * 5 + i // 7) % distinct for i in range(n)]
    for i, k in enumerate(order):
        d_in[i * stride:i * stride + w * h * 3].copy_(torch.from_numpy(frames[k].reshape(-1)))
    torch.cuda.synchronize()
    dev = je.default_device(0)
    enc = make_encoder(cfg, dev)
    for _ in range(2):  # the second call runs with learnt buffer sizes and cached plan / tables
        d_files, offs = enc.encode_batch_device(d_in.data_ptr(), stride, n, w, h, je.ColorType.Rgb)
        blob = dev.download(d_files, offs[-1])
        assert offs[0] == 0
        bad = [i for i in range(n) if bytes(blob[offs[i]:offs[i + 1]]) != want[order[i]]]
        assert not bad, "files differ: %r" % bad[:10]


def test_config4a_full_size_gray_custom_tables():
    t = _bench_custom_table()
    img = _torch_frame(8192, 8192, 1, seed=3)
    _same("luma", 8192, 8192, dict(quality=95, sampling=(1, 1), qtables=(t, t)), img=img)


def test_config4b_full_size_cmyk_as_ycck_custom_tables():
    t = _bench_custom_table()
    img = _torch_frame(8192, 8192, 4, seed=4)
    _same("cmyk_as_ycck", 8192, 8192, dict(quality=95, sampling=(1, 1), qtables=(t, t)), img=img)


def test_config4_tables_above_255_parity_only():
    """Q10: table entries > 255 are truncated in the DQT segment but quantize with their full value; such files
    do not decode correctly, so this case is compared on bytes only (SURVEY 8d)."""
    rng = np.random.default_rng(44)
    t = [int(v) for v in rng.integers(1, 1200, 64)]
    for color, w, h in (("luma", 2048, 2048), ("cmyk_as_ycck", 2048, 1024)):
        _same(color, w, h, dict(quality=95, sampling=(1, 1), qtables=(t, t)), img=_torch_frame(w, h, BPP[color], seed=5))


def test_config5_full_size_progressive_8_strips_one_gpu():
    """16384 x 16384 RGB progressive 4:2:0, restart interval 2048, cut into 8 restart-aligned strips that are
    encoded one after the other on this GPU and concatenated scan-major: equal to the whole-image oracle file."""
    w = h = 16384
    cfg = dict(quality=90, sampling=(2, 2), progressive_scans=4, restart_interval=2048)
    img = _torch_frame(w, h, 3, seed=7)
    got, n = _encode_by_strips(img, w, h, "rgb", cfg, 8)
    assert n == 8
    want = oracle_encode(img, w, h, "rgb", cfg)
    assert len(got) == len(want) and got == want


def test_config5_full_size_whole_image_one_call():
    """The same image through the ordinary Encoder::encode call (no strips): 805 MB of pixels, 12 scans."""
    w = h = 16384
    cfg = dict(quality=90, sampling=(2, 2), progressive_scans=4, restart_interval=2048)
    img = _torch_frame(w, h, 3, seed=7)
    _same("rgb", w, h, cfg, img=img)


# ---- one image cut into restart-aligned strips (BASELINE config 5 mechanics, on one GPU) ---------
def _encode_by_strips(img, w, h, color, cfg, max_strips):
    import torch
    import jpeg_encoder_b200 as je
    from jpeg_encoder_b200 import sharding
    enc = make_encoder(cfg)
    ct = CT[color][1]
    strips = enc.plan_strips(w, h, ct, max_strips)
    dev = je.default_device(0)
    flat = np.ascontiguousarray(img).reshape(h, -1)
    d_px = [torch.from_numpy(flat[r0:r0 + rows].copy()).cuda() for r0, rows in strips]
    torch.cuda.synchronize()
    hist_total = None
    if cfg.get("optimize_huffman"):  # what sharding.exchange_strip_histograms does across ranks, here in one process
        hists, edges = [], []
        for i, (r0, rows) in enumerate(strips):
            hi, ed = enc.strip_histogram_device(d_px[i].data_ptr(), i, len(strips), r0, rows, w, h, ct)
            hists.append(hi)
            edges += ed
        hist_total = enc.merge_strip_histograms([sum(col) for col in zip(*hists)], edges, w, h, ct)
    pieces = []
    for i, (r0, rows) in enumerate(strips):
        d_bytes, offs = enc.encode_strip_device(d_px[i].data_ptr(), i, len(strips), r0, rows, w, h, ct, hist_total=hist_total)
        pieces.append(sharding.split_pieces(dev.download(d_bytes, offs[-1]), offs))
    return sharding.assemble_pieces(pieces), len(strips)


@pytest.mark.parametrize("name,color,w,h,cfg,max_strips", [
    ("progressive_420", "rgb", 512, 400, dict(quality=85, sampling=(2, 2), progressive_scans=4, restart_interval=32), 4),
    ("progressive_420_odd", "rgb", 509, 397, dict(quality=85, sampling=(2, 2), progressive_scans=4, restart_interval=64), 8),
    ("interleaved_restart", "rgb", 640, 360, dict(quality=90, sampling=(2, 2), restart_interval=20), 6),
    ("sequential_4_1", "rgb", 512, 256, dict(quality=75, sampling=(4, 1), restart_interval=16), 4),
    ("luma", "luma", 384, 512, dict(quality=95, restart_interval=48), 8),
    ("ycck_progressive", "cmyk_as_ycck", 256, 256, dict(quality=90, sampling=(1, 1), progressive_scans=3, restart_interval=32), 4),
    ("optimized_420", "rgb", 512, 400, dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=64), 4),
    ("optimized_progressive", "rgb", 384, 384, dict(quality=70, sampling=(2, 1), optimize_huffman=True, progressive_scans=5, restart_interval=48), 8),
    ("optimized_cmyk", "cmyk", 256, 320, dict(quality=90, sampling=(2, 2), optimize_huffman=True, restart_interval=16), 5),
])
def test_strips_concatenate_to_the_whole_image(name, color, w, h, cfg, max_strips):
    img = _img(color, w, h, seed=21)
    got, n = _encode_by_strips(img, w, h, color, cfg, max_strips)
    assert n > 1, "test geometry must actually split"
    assert got == oracle_encode(img, w, h, color, cfg)


def test_device_huffman_tables_equal_host_and_oracle():
    """csrc/tables.cu (Annex K.2 on the device, what the optimized encode path runs) against the host planner and the
    oracle on 600 histograms: skewed, flat, sparse, all-equal (every tie goes to the largest symbol), single-symbol,
    Fibonacci-like (code lengths beyond 16 bits: Figure K.3) and beyond 32 bits (the reference panics: an error here)."""
    import ctypes as C
    import jpeg_encoder_b200 as je
    dev = je.default_device(0)
    lib = dev.lib
    rng = np.random.default_rng(12)
    # symbols 8-bit JPEG can produce: AC run/size with size 1..10 plus EOB (0x00) and ZRL (0xF0); DC categories 0..11
    ac_syms = np.array([0x00, 0xF0] + [(r << 4) | z for r in range(16) for z in range(1, 11)])
    dc_syms = np.arange(12)

    def make_cases(syms):
        cases = []
        for i in range(280):
            f = np.zeros(257, np.uint32)
            k = int(rng.integers(1, len(syms) + 1))
            idx = rng.choice(syms, k, replace=False)
            r = rng.random()
            if r < 0.5:
                f[idx] = (rng.pareto(0.7, k) * 10 + 1).astype(np.uint32)
            elif r < 0.75:
                f[idx] = rng.integers(1, 50, k)
            elif r < 0.9:
                f[idx] = int(rng.integers(1, 4))  # all equal: nothing but ties
            else:
                f[idx] = rng.integers(1, 3, k)
            cases.append(f)
        for n_fib in (5, 10, 12, 20, 30, 40, 45):  # 30 and more force the length limiting; 40+ exceed 32 bits
            if n_fib > len(syms):
                continue
            fib = np.zeros(257, np.uint32)
            a, b = 1, 1
            for i in range(n_fib):
                fib[syms[i]] = min(a, 2 ** 32 - 1)
                a, b = b, a + b
            cases.append(fib)
        for k in (0, 1, 2):  # no symbol at all / one / two
            f = np.zeros(257, np.uint32)
            f[syms[:k]] = 7
            cases.append(f)
        for f in cases:
            f[256] = 1
        return cases

    total_bad = 0
    for ac, syms in ((1, ac_syms), (0, dc_syms)):
        cases = make_cases(syms)
        n = len(cases)
        flat = np.ascontiguousarray(np.stack(cases).astype(np.uint32))
        lengths = (C.c_uint8 * (16 * n))()
        values = (C.c_uint8 * (256 * n))()
        nv = (C.c_uint32 * n)()
        words = (C.c_uint32 * (256 * n))()
        status = (C.c_int * n)()
        rc = lib.jpgb_optimized_huffman_tables_device(dev.handle, flat.ctypes.data_as(C.POINTER(C.c_uint32)), n, ac, lengths, values, nv, words, status)
        assert rc == 0, dev.last_error()
        for i, f in enumerate(cases):
            hl, hv, hn = (C.c_uint8 * 16)(), (C.c_uint8 * 256)(), C.c_uint32()
            hrc = lib.jpgb_optimized_huffman_table(f.ctypes.data_as(C.POINTER(C.c_uint32)), hl, hv, C.byref(hn))
            assert (hrc == 0) == (status[i] == 0), "case %d: host rc %d, device status %d" % (i, hrc, status[i])
            if hrc != 0:  # a code longer than 32 bits: the reference panics
                total_bad += 1
                continue
            assert list(lengths[16 * i:16 * i + 16]) == list(hl), "case %d lengths" % i
            assert nv[i] == hn.value and list(values[256 * i:256 * i + nv[i]]) == list(hv)[:hn.value], "case %d values" % i
            want_len, want_vals = orc.huffman_optimized(f.tolist())
            assert list(hl) == want_len and list(hv)[:hn.value] == want_vals
            # the code words the coding kernel reads: (length + size) << 27 | code << size, canonical codes in order of `values`
            code, k = 0, 0
            expect = {}
            for bits in range(1, 17):
                for _ in range(hl[bits - 1]):
                    expect[hv[k]] = (bits, code)
                    code += 1
                    k += 1
                code <<= 1
            for sym in range(256 if ac else 16):
                z = (sym & 15) if ac else sym
                l, c = expect.get(sym, (0, 0))
                assert words[256 * i + sym] == (((l + z) << 27) | (c << z)) & 0xFFFFFFFF, "case %d symbol %#x" % (i, sym)
    assert total_bad >= 1


def test_device_placed_gather_of_strip_pieces():
    """csrc/gather.cu on one GPU: the strips are encoded one after the other, and each time the placement kernel stores
    that strip's pieces at their final scan-major offsets inside the gather target, exactly as rank i of an N-GPU job
    does through a peer pointer. The assembled buffer must be the whole-image file."""
    import ctypes as C
    import torch
    import jpeg_encoder_b200 as je
    from jpeg_encoder_b200 import sharding
    w, h, color = 640, 496, "rgb"
    cfg = dict(quality=85, sampling=(2, 2), progressive_scans=4, restart_interval=40)
    img = _img(color, w, h, seed=33)
    want = oracle_encode(img, w, h, color, cfg)
    enc = make_encoder(cfg)
    ct = CT[color][1]
    dev = je.default_device(0)
    strips = enc.plan_strips(w, h, ct, 5)
    assert len(strips) > 2
    flat = np.ascontiguousarray(img).reshape(h, -1)
    d_px = [torch.from_numpy(flat[r0:r0 + rows].copy()).cuda() for r0, rows in strips]
    torch.cuda.synchronize()
    table = []
    for i, (r0, rows) in enumerate(strips):  # pass 1: every strip's piece offsets (what the all-gather distributes)
        _, offs = enc.encode_strip_device(d_px[i].data_ptr(), i, len(strips), r0, rows, w, h, ct)
        table.append(list(offs))
    dest, total = sharding.piece_destinations(table)
    assert total == len(want)
    target, handle = C.c_void_p(), (C.c_uint8 * 64)()
    assert dev.lib.jpgb_gather_target_create(dev.handle, total + 1000, C.byref(target), handle) == 0
    d_table = torch.tensor([v for row in table for v in row], dtype=torch.int64, device="cuda")
    d_total = torch.zeros(1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    for i, (r0, rows) in enumerate(strips):  # pass 2: encode again, place as "rank i"
        enc.encode_strip_device(d_px[i].data_ptr(), i, len(strips), r0, rows, w, h, ct)
        rc = dev.lib.jpgb_gather_place_pieces(dev.handle, target, total + 1000, C.c_void_p(d_table.data_ptr()), len(strips), i, C.c_void_p(d_total.data_ptr()))
        assert rc == 0, dev.last_error()
    got = dev.download(target.value, total)
    assert int(d_total.item()) == total
    assert got == want
    assert dev.lib.jpgb_gather_target_close(dev.handle, target, 0) == 0


def test_cpp_mirror_on_gpu(tmp_path):
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "jpeg_encoder_b200")
    exe = str(tmp_path / "mirror_smoke")
    subprocess.check_call(["g++", "-std=c++17", "-I" + os.path.join(root, "include"), os.path.join(root, "tests", "cpp", "mirror_smoke.cpp"),
                           "-o", exe, "-L" + pkg, "-ljpegenc_b200", "-Wl,-rpath," + pkg])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "tail ok" in r.stdout, r.stdout + r.stderr


def test_pipelined_host_batch_many_chunks():
    """Large enough to span several upload/encode/download chunks (two pixel and two output buffers in flight)."""
    import ctypes as C
    import jpeg_encoder_b200 as je
    w, h, n = 1920, 1080, 40
    frames = [images.synth_frame(w, h, 3, seed=s) for s in range(4)]
    cfg = dict(quality=90, sampling=(2, 2))
    want = [oracle_encode(f, w, h, "rgb", cfg) for f in frames]
    enc = make_encoder(cfg)
    outs = enc.encode_batch([frames[i % 4] for i in range(n)], w, h, je.ColorType.Rgb)
    assert [o == want[i % 4] for i, o in enumerate(outs)] == [True] * n
    cfg2 = dict(quality=80, sampling=(2, 2), optimize_huffman=True, restart_interval=100)
    outs = make_encoder(cfg2).encode_batch([frames[i % 4] for i in range(20)], w, h, je.ColorType.Rgb)
    want2 = [oracle_encode(f, w, h, "rgb", cfg2) for f in frames]
    assert [o == want2[i % 4] for i, o in enumerate(outs)] == [True] * 20


# ---- Encoder::encode_image<I: ImageBuffer> (src/encoder.rs:506-515): planar samples, taken verbatim ----
class _RgbImageBuffer:
    """The doc example of the trait (src/image_buffer.rs:48-84): an RGB image converted row by row."""

    def __init__(self, rgb):
        self.rgb = rgb

    def get_jpeg_color_type(self):
        import jpeg_encoder_b200 as je
        return je.JpegColorType.Ycbcr

    def width(self):
        return self.rgb.shape[1]

    def height(self):
        return self.rgb.shape[0]

    def fill_buffers(self, y, buffers):
        r, g, b = (self.rgb[y, :, i].astype(np.int32) for i in range(3))
        buffers[0] += ((19595 * r + 38470 * g + 7471 * b + 0x7FFF) >> 16).astype(np.uint8).tobytes()
        buffers[1] += ((-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 0x7FFF) >> 16).astype(np.uint8).tobytes()
        buffers[2] += ((32768 * r - 27439 * g - 5329 * b + (128 << 16) + 0x7FFF) >> 16).astype(np.uint8).tobytes()


def test_encode_image_trait_equals_encode_rgb():
    img = _img("rgb", 203, 131, seed=8)
    for cfg in (dict(quality=88, sampling=(2, 2)), dict(quality=70, sampling=(4, 1), optimize_huffman=True),
                dict(quality=95, sampling=(1, 1), progressive_scans=4, restart_interval=10)):
        got = make_encoder(cfg).encode_image(_RgbImageBuffer(img))
        assert got == oracle_encode(img, 203, 131, "rgb", cfg)


@pytest.mark.parametrize("kind", ["luma", "ycbcr", "cmyk", "ycck"])
def test_encode_planes_all_jpeg_color_types(kind):
    import jpeg_encoder_b200 as je
    w, h = 150, 91
    jct = {"luma": je.JpegColorType.Luma, "ycbcr": je.JpegColorType.Ycbcr, "cmyk": je.JpegColorType.Cmyk, "ycck": je.JpegColorType.Ycck}[kind]
    n = jct.get_num_components()
    planes = [images.photo_like(w, h, 1, seed=30 + c) for c in range(n)]
    packed = planes[0] if n == 1 else np.stack(planes, -1)
    for cfg in (dict(quality=80, sampling=(2, 2)), dict(quality=80, sampling=(2, 4), restart_interval=6), dict(quality=80, sampling=(1, 2), progressive_scans=3)):
        got = make_encoder(cfg).encode_planes(planes, w, h, jct)
        # the packed adaptors copy Luma/Ycbcr/Ycck samples verbatim and invert Cmyk (src/image_buffer.rs:115-121, 221-229, 247-256, 303-312)
        ref_in = 255 - packed if kind == "cmyk" else packed
        assert got == oracle_encode(ref_in, w, h, kind, cfg)


@pytest.mark.parametrize("sampling", [(1, 1), (1, 2), (2, 1), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)])
def test_planar_warp_kernel_against_generic_kernel_and_oracle(sampling, monkeypatch):
    """Planar input has its own warp kernel (one launch per plane, the plane's decimation as template arguments):
    interior tiles (cp.async of whole rows), right / bottom edges (replication, Q4), unaligned widths, every sampling."""
    import jpeg_encoder_b200 as je
    for kind, (w, h) in (("ycbcr", (1040, 100)), ("ycck", (531, 70)), ("cmyk", (1296, 41)), ("luma", (1029, 67))):
        jct = {"luma": je.JpegColorType.Luma, "ycbcr": je.JpegColorType.Ycbcr, "cmyk": je.JpegColorType.Cmyk, "ycck": je.JpegColorType.Ycck}[kind]
        n = jct.get_num_components()
        planes = [images.photo_like(w, h, 1, seed=70 + c) for c in range(n)]
        packed = planes[0] if n == 1 else np.stack(planes, -1)
        ref_in = 255 - packed if kind == "cmyk" else packed
        for cfg in (dict(quality=85, sampling=sampling), dict(quality=85, sampling=sampling, restart_interval=9, optimize_huffman=True)):
            want = oracle_encode(ref_in, w, h, kind, cfg)
            assert make_encoder(cfg).encode_planes(planes, w, h, jct) == want, (kind, cfg)
            monkeypatch.setenv("JPGB_FORCE_GENERIC_STAGE_A", "1")
            assert make_encoder(cfg).encode_planes(planes, w, h, jct) == want, (kind, cfg, "generic")
            monkeypatch.delenv("JPGB_FORCE_GENERIC_STAGE_A")


def test_unstuffed_stream_is_fully_written_without_a_clear(monkeypatch):
    """The unstuffed stream is never cleared as a whole: chunks store the words they own and OR into the words they
    share, which the lead kernel zeroes. With JPGB_POISON_STREAM=1 the buffer starts as all ones before every call, so any
    byte that is neither stored nor zeroed corrupts the file."""
    monkeypatch.setenv("JPGB_POISON_STREAM", "1")
    cases = [("rgb", 333, 77, dict(quality=83, sampling=(2, 2))),
             ("rgb", 640, 480, dict(quality=95, sampling=(2, 2), restart_interval=1)),
             ("rgb", 641, 479, dict(quality=40, sampling=(2, 1), restart_interval=7, progressive_scans=5)),
             ("luma", 1027, 517, dict(quality=99)),
             ("luma", 5, 3, dict(quality=10, optimize_huffman=True)),
             ("cmyk_as_ycck", 259, 131, dict(quality=75, sampling=(1, 1), optimize_huffman=True, restart_interval=3)),
             ("ycbcr", 97, 75, dict(quality=60, sampling=(4, 1), restart_interval=2)),
             ("rgb", 2048, 1024, dict(quality=90, sampling=(2, 2), progressive_scans=12, optimize_huffman=True))]
    for color, w, h, cfg in cases:
        img = _img(color, w, h, seed=5)
        assert gpu_encode(img, w, h, color, cfg) == oracle_encode(img, w, h, color, cfg), (color, w, h, cfg)
    import jpeg_encoder_b200 as je
    frames = [_img("rgb", 320, 240, seed=60 + i) for i in range(9)]
    cfg = dict(quality=88, sampling=(2, 2))
    assert make_encoder(cfg).encode_batch(frames, 320, 240, je.ColorType.Rgb) == [oracle_encode(f, 320, 240, "rgb", cfg) for f in frames]


def test_concurrent_contexts_on_threads():
    """One jpgb_encoder context per host thread (the reference's Encoder is Send, not shared): four threads
    encode different configurations at the same time on their own streams; every result must stay exact."""
    import threading
    import jpeg_encoder_b200 as je
    cfgs = [("rgb", dict(quality=90, sampling=(2, 2))), ("luma", dict(quality=70, progressive_scans=3)),
            ("cmyk_as_ycck", dict(quality=85, sampling=(1, 1), optimize_huffman=True)), ("bgr", dict(quality=60, sampling=(2, 1), restart_interval=5))]
    imgs = [_img(c, 640, 360, seed=40 + i) for i, (c, _) in enumerate(cfgs)]
    want = [oracle_encode(imgs[i], 640, 360, c, cfg) for i, (c, cfg) in enumerate(cfgs)]
    errors = []

    def work(i):
        try:
            dev = je.Device(0)
            color, cfg = cfgs[i]
            for _ in range(12):
                if make_encoder(cfg, dev).encode(imgs[i], 640, 360, CT[color][1]) != want[i]:
                    errors.append("thread %d: bytes differ" % i)
                    break
            dev.close()
        except Exception as e:  # noqa: BLE001
            errors.append("thread %d: %r" % (i, e))

    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


# ---- randomized sweep over the whole settings space (seeded: the same 96 cases every run) -----------------------
def _random_cases(n=None, seed=None):
    import os
    n = int(os.environ.get("JPGB_SWEEP_CASES", "96")) if n is None else n       # a longer hunt: JPGB_SWEEP_CASES=2000
    seed = int(os.environ.get("JPGB_SWEEP_SEED", "20260117")) if seed is None else seed
    max_dim = int(os.environ.get("JPGB_SWEEP_MAXDIM", "120"))
    rng = np.random.default_rng(seed)
    colors = sorted(BPP)
    samplings = [(1, 1), (2, 1), (1, 2), (2, 2), (4, 1), (4, 2), (1, 4), (2, 4)]
    out = []
    for i in range(n):
        color = colors[int(rng.integers(len(colors)))]
        w, h = int(rng.integers(1, max_dim)), int(rng.integers(1, max_dim))
        cfg = dict(quality=int(rng.integers(1, 101)), sampling=samplings[int(rng.integers(len(samplings)))])
        if rng.random() < 0.4:
            cfg["progressive_scans"] = int(rng.integers(2, 65))
        if rng.random() < 0.5:
            cfg["restart_interval"] = int(rng.integers(1, 60))
        if rng.random() < 0.4:
            cfg["optimize_huffman"] = True
        r = rng.random()
        if r < 0.3:
            cfg["qtables"] = (int(rng.integers(0, 9)), int(rng.integers(0, 9)))
        elif r < 0.45:
            cfg["qtables"] = ([int(v) for v in rng.integers(1, 300, 64)], [int(v) for v in rng.integers(1, 40, 64)])
        kind = ["photo", "noise", "flat"][int(rng.integers(3))]
        out.append((i, color, w, h, cfg, kind))
    return out


def _sweep_image(i, color, w, h, kind):
    rng = np.random.default_rng(1000 + i)
    if kind == "photo":
        return _img(color, w, h, seed=i)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, BPP[color]), dtype=np.uint8)
    return np.full((h, w, BPP[color]), int(rng.integers(0, 256)), np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", range(8))
def test_random_settings_sweep(chunk):
    """96 seeded random combinations of colour type, geometry, quality, sampling, tables, progressive scan count,
    restart interval and optimized tables (including the Q18 inputs whose streams are knowingly undecodable): the GPU
    file must equal the oracle's byte for byte."""
    failures = []
    for i, color, w, h, cfg, kind in _random_cases()[chunk::8]:
        img = _sweep_image(i, color, w, h, kind)
        got = gpu_encode(img, w, h, color, cfg)
        want = oracle_encode(img, w, h, color, cfg)
        if got != want:
            failures.append("case %d: %s %dx%d %r (%s): %d vs %d bytes" % (i, color, w, h, {k: v for k, v in cfg.items() if k != "qtables"},
                                                                           kind, len(got), len(want)))
    assert not failures, "\n".join(failures)
