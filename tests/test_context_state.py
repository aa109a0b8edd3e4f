"""State that an encode context carries from one call to the next, checked on purpose.

Every test builds its own contexts (je.Device) and closes them; none uses the shared default context, so what a test
sees does not depend on what ran before it. Every file is compared byte for byte with the oracle (strips: with the
whole-image oracle file). Covered: each capacity-retry branch forced with JPGB_TIGHT_CAPS on the first call of a fresh
context and the state it leaves for the next calls; the same under JPGB_POISON_ALLOC (fresh allocations filled with
ones); reuse of the strip histogram's coefficients by the strip encode and its invalidation; the sliced upload of one
large packed image; and one context running a long mixed sequence of calls."""
import contextlib
import functools
import io

import numpy as np
import pytest

import images
from cases import BPP, CT, make_encoder, oracle_encode

pytestmark = pytest.mark.gpu

_ORACLE = {}


def _want(tag, img, w, h, color, cfg):
    """oracle_encode, cached per (image, settings): the same inputs recur across parameters and calls."""
    key = (tag, w, h, color, repr(sorted(cfg.items())))
    if key not in _ORACLE:
        _ORACLE[key] = oracle_encode(img, w, h, color, cfg)
    return _ORACLE[key]


@functools.lru_cache(maxsize=None)
def _photo(w, h, ch, seed):
    return images.photo_like(w, h, ch, seed=seed)


@functools.lru_cache(maxsize=None)
def _blocky(w, h, ch, seed):
    """photo_like at an eighth of the size, every sample repeated 8 x 8: 60-180 KB per 1080p file instead of 340-540."""
    small = images.photo_like(w // 8, h // 8, ch, seed=seed)
    return np.ascontiguousarray(np.repeat(np.repeat(small, 8, 0), 8, 1))


@contextlib.contextmanager
def _context():
    import jpeg_encoder_b200 as je
    dev = je.Device(0)
    try:
        yield dev
    finally:
        dev.close()


def _diff(got, want):
    n = min(len(got), len(want))
    first = next((i for i in range(n) if got[i] != want[i]), n)
    return "len %d vs %d, first difference at byte %d" % (len(got), len(want), first)


# ---- the entry paths, one call each: (files, launch count of the call) --------------------------------------------
def _encode_strips(dev, img, w, h, color, cfg, max_strips):
    """All strips of one image on `dev` (the histograms first when the tables are optimized), assembled scan-major.
    The launch count is the sum over the strip encodes."""
    import torch
    from jpeg_encoder_b200 import sharding
    enc = make_encoder(cfg, dev)
    ct = CT[color][1]
    strips = enc.plan_strips(w, h, ct, max_strips)
    flat = np.ascontiguousarray(img).reshape(h, -1)
    d_px = [torch.from_numpy(flat[r0:r0 + rows].copy()).cuda() for r0, rows in strips]
    torch.cuda.synchronize()
    hist_total = None
    if cfg.get("optimize_huffman"):
        hists, edges = [], []
        for i, (r0, rows) in enumerate(strips):
            hi, ed = enc.strip_histogram_device(d_px[i].data_ptr(), i, len(strips), r0, rows, w, h, ct)
            hists.append(hi)
            edges += ed
        hist_total = enc.merge_strip_histograms([sum(col) for col in zip(*hists)], edges, w, h, ct)
    pieces, launches = [], 0
    for i, (r0, rows) in enumerate(strips):
        d_bytes, offs = enc.encode_strip_device(d_px[i].data_ptr(), i, len(strips), r0, rows, w, h, ct, hist_total=hist_total)
        launches += dev.last_launch_count()
        pieces.append(sharding.split_pieces(dev.download(d_bytes, offs[-1]), offs))
    return sharding.assemble_pieces(pieces), launches, len(strips)


# Every call below needs more than 128 KiB of pool: a context that kept a pool of that size must overflow. The
# batches take blocky frames: a chunk of the pipelined host path holds ~96 MB of pixels, and with photo-like frames its
# stream would come close to 8 MiB, where the launch count changes with the capacity alone (the 0xFF count scan).
W, H = 1920, 1080
BATCH_N = 20  # two chunks of the pipelined host path
DEVICE_N = 7

CONFIGS = [
    ("rgb", dict(quality=90, sampling=(2, 2))),                                               # 4:2:0 interleaved
    ("rgb", dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=30)),
    ("rgb", dict(quality=88, sampling=(2, 1), progressive_scans=5, restart_interval=60)),
    ("cmyk", dict(quality=80, sampling=(4, 1))),                                              # factor 4: sequential scans
]
STRIP_CONFIGS = {
    "strips": [("rgb", dict(quality=88, sampling=(2, 1), progressive_scans=5, restart_interval=60)),
               ("cmyk", dict(quality=80, sampling=(4, 1), restart_interval=20))],
    "strips_optimized": [("rgb", dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=30)),
                         ("cmyk", dict(quality=80, sampling=(4, 1), optimize_huffman=True, restart_interval=20))],
}
PATHS = ["encode", "encode_to", "encode_batch", "encode_batch_device", "encode_planes", "strips", "strips_optimized"]


class _Case:
    """One path and configuration: builds the inputs and the expected files once, runs one call on a context."""

    def __init__(self, path, color, cfg):
        import jpeg_encoder_b200 as je
        self.path, self.color, self.cfg = path, color, cfg
        ch = BPP[color]
        if path == "encode_planes":
            self.jct = je.JpegColorType.Cmyk if color == "cmyk" else je.JpegColorType.Ycbcr
            n = self.jct.get_num_components()
            self.planes = [_photo(W, H, 1, 40 + c) for c in range(n)]
            packed = np.stack(self.planes, -1)
            # the packed adaptors take Ycbcr samples verbatim and invert Cmyk (src/image_buffer.rs:221-229, 247-256)
            ref = 255 - packed if color == "cmyk" else packed
            self.want = [_want(("planes", color), ref, W, H, "cmyk" if color == "cmyk" else "ycbcr", cfg)]
        elif path in ("encode_batch", "encode_batch_device"):
            frames = [_blocky(W, H, ch, 10 + k) for k in range(4)]
            n = BATCH_N if path == "encode_batch" else DEVICE_N
            self.frames = [frames[(i * 3) % 4] for i in range(n)]
            self.want = [_want(("blocky", (i * 3) % 4), frames[(i * 3) % 4], W, H, color, cfg) for i in range(n)]
            if path == "encode_batch":
                stride = (W * H * ch + 255) & ~255
                assert BATCH_N > (96 << 20) // stride, "the batch must span two pipeline chunks"
        else:
            self.img = _photo(W, H, ch, 3)
            self.want = [_want(("photo", "one"), self.img, W, H, color, cfg)]
        assert sum(len(f) for f in self.want) > 256 << 10
        self.d_in = None

    def run(self, dev):
        enc = make_encoder(self.cfg, dev)
        ct = CT[self.color][1]
        if self.path == "encode":
            files = [enc.encode(self.img, W, H, ct)]
        elif self.path == "encode_to":
            buf = io.BytesIO()
            enc.encode_to(buf, self.img, W, H, ct)
            files = [buf.getvalue()]
        elif self.path == "encode_planes":
            files = [enc.encode_planes(self.planes, W, H, self.jct)]
        elif self.path == "encode_batch":
            files = enc.encode_batch(self.frames, W, H, ct)
        elif self.path == "encode_batch_device":
            import torch
            stride = (W * H * BPP[self.color] + 255) & ~255
            if self.d_in is None:
                self.d_in = torch.zeros(DEVICE_N * stride, dtype=torch.uint8, device="cuda")
                for i, f in enumerate(self.frames):
                    self.d_in[i * stride:i * stride + f.size].copy_(torch.from_numpy(f.reshape(-1)))
                torch.cuda.synchronize()
            d_files, offs = enc.encode_batch_device(self.d_in.data_ptr(), stride, DEVICE_N, W, H, ct)
            blob = dev.download(d_files, offs[-1])
            files = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(DEVICE_N)]
        else:
            f, launches, n = _encode_strips(dev, self.img, W, H, self.color, self.cfg, 4)
            assert n > 1
            return [f], launches
        return files, dev.last_launch_count()

    def check(self, files, what):
        assert len(files) == len(self.want)
        bad = [i for i, (g, w) in enumerate(zip(files, self.want)) if g != w]
        assert not bad, "%s %s %r, %s: file %d: %s" % (self.path, self.color, self.cfg, what, bad[0], _diff(files[bad[0]], self.want[bad[0]]))


def _path_configs(path):
    return STRIP_CONFIGS.get(path, CONFIGS)


@pytest.mark.parametrize("poison", [False, True], ids=["plain", "poisoned"])
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("tight", ["pool", "stream", "out", "pool,stream,out"])
def test_forced_retry_leaves_a_steady_context(tight, path, poison, monkeypatch):
    """The first call on a fresh context starts from the floor of the named capacities, so its status block, pool and
    buffers must grow and the retry branch runs (pool: recode; stream / out: the tail again with a larger stream /
    output). Its files must be exact, and the sizes it leaves behind must let the next calls run without a retry: two
    more calls with the same settings and input are exact and take as many launches as the steady call of a context
    that never saw the hook."""
    if poison:
        monkeypatch.setenv("JPGB_POISON_ALLOC", "1")
    for color, cfg in _path_configs(path):
        case = _Case(path, color, cfg)
        with _context() as dev:  # the reference: no hook, the second call runs with sizes learnt from the first
            case.check(case.run(dev)[0], "reference call 1")
            files, steady = case.run(dev)
            case.check(files, "reference call 2")
        with _context() as dev:
            monkeypatch.setenv("JPGB_TIGHT_CAPS", tight)
            try:
                files, forced = case.run(dev)
            finally:
                monkeypatch.delenv("JPGB_TIGHT_CAPS")
            case.check(files, "forced call")
            counts = [forced]
            for k in range(2):
                files, launches = case.run(dev)
                case.check(files, "call %d after the forced one" % (k + 1))
                counts.append(launches)
        print("%s %s %s %r: launches forced %d, then %d %d (steady %d)" % (tight, path, color, cfg, forced, counts[1], counts[2], steady))
        assert counts[1] == counts[2] == steady, "a call after the forced one retried: launches %r, steady %d" % (counts, steady)
        assert forced > steady, "the forced call did not retry: %d launches, steady %d" % (forced, steady)


def test_random_sweep_on_one_poisoned_context(monkeypatch):
    """The 96 seeded random cases of test_gpu_parity's sweep in sequence on one fresh context whose allocations start
    as all ones: many buffer growths, graph keys and table switches, each file exact."""
    from test_gpu_parity import _random_cases, _sweep_image
    monkeypatch.setenv("JPGB_POISON_ALLOC", "1")
    failures = []
    with _context() as dev:
        for i, color, w, h, cfg, kind in _random_cases():
            img = _sweep_image(i, color, w, h, kind)
            got = make_encoder(cfg, dev).encode(img, w, h, CT[color][1])
            want = oracle_encode(img, w, h, color, cfg)
            if got != want:
                failures.append("case %d: %s %dx%d %r (%s): %s" % (i, color, w, h, {k: v for k, v in cfg.items() if k != "qtables"}, kind, _diff(got, want)))
    assert not failures, "\n".join(failures)


# ---- coefficient reuse between the strip histogram and the optimized strip encode, as ranks run it ------------------
REUSE_CASES = {
    "optimized_420": ("rgb", 1270, 1001, dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=40), 4),
    "optimized_progressive": ("rgb", 1270, 1001, dict(quality=70, sampling=(2, 1), optimize_huffman=True, progressive_scans=5, restart_interval=6), 4),
    "optimized_cmyk_1_2": ("cmyk", 1270, 1001, dict(quality=90, sampling=(1, 2), optimize_huffman=True, restart_interval=10), 5),
}


def _strip_inputs(color, w, h, cfg, max_strips):
    import torch
    img = _photo(w, h, BPP[color], 23)
    strips = make_encoder(cfg).plan_strips(w, h, CT[color][1], max_strips)
    assert 3 <= len(strips) <= 5
    flat = np.ascontiguousarray(img).reshape(h, -1)
    d_px = [torch.from_numpy(flat[r0:r0 + rows].copy()).cuda() for r0, rows in strips]
    copies = [t.clone() for t in d_px]  # the same pixels at another address
    torch.cuda.synchronize()
    return img, strips, d_px, copies


def _rank_histogram(dev, cfg, color, w, h, strips, i, d):
    r0, rows = strips[i]
    return make_encoder(cfg, dev).strip_histogram_device(d.data_ptr(), i, len(strips), r0, rows, w, h, CT[color][1])


def _rank_encode(dev, cfg, color, w, h, strips, i, d, hist_total):
    """One strip's encode on `dev`: (pieces, launch count, stage times or None)."""
    from jpeg_encoder_b200 import sharding
    r0, rows = strips[i]
    d_bytes, offs = make_encoder(cfg, dev).encode_strip_device(d.data_ptr(), i, len(strips), r0, rows, w, h, CT[color][1], hist_total=hist_total)
    launches = dev.last_launch_count()
    return sharding.split_pieces(dev.download(d_bytes, offs[-1]), offs), launches, dev.last_timing()


def _merge(cfg, color, w, h, results):
    hists = [r[0] for r in results]
    edges = [e for r in results for e in r[1]]
    return make_encoder(cfg).merge_strip_histograms([sum(col) for col in zip(*hists)], edges, w, h, CT[color][1])


@pytest.mark.parametrize("name", sorted(REUSE_CASES))
def test_strip_encode_reuses_the_histogram_coefficients(name):
    """One context per strip, as the ranks of a sharded encode: each computes its strip's histogram, the histograms are
    merged on the host, and each context encodes its strip on the same pointer, so the encode takes the coefficients
    the histogram left instead of running the colour+DCT kernel again. Contexts B have the same history except that
    their histogram ran on a copy of the pixels at another address: they must recompute, one launch more. Both
    assembled files equal the whole-image oracle file."""
    import jpeg_encoder_b200 as je
    from jpeg_encoder_b200 import sharding
    color, w, h, cfg, max_strips = REUSE_CASES[name]
    img, strips, d_px, copies = _strip_inputs(color, w, h, cfg, max_strips)
    want = _want(("reuse", name), img, w, h, color, cfg)
    ctx_a = [je.Device(0) for _ in strips]
    ctx_b = [je.Device(0) for _ in strips]
    try:
        hist_a = [_rank_histogram(ctx_a[i], cfg, color, w, h, strips, i, d_px[i]) for i in range(len(strips))]
        hist_b = [_rank_histogram(ctx_b[i], cfg, color, w, h, strips, i, copies[i]) for i in range(len(strips))]
        assert hist_a == hist_b
        total = _merge(cfg, color, w, h, hist_a)
        enc_a = [_rank_encode(ctx_a[i], cfg, color, w, h, strips, i, d_px[i], total) for i in range(len(strips))]
        enc_b = [_rank_encode(ctx_b[i], cfg, color, w, h, strips, i, d_px[i], total) for i in range(len(strips))]
    finally:
        for dev in ctx_a + ctx_b:
            dev.close()
    la, lb = [r[1] for r in enc_a], [r[1] for r in enc_b]
    print("%s: %d strips, launches with reuse %r, without %r" % (name, len(strips), la, lb))
    got_a = sharding.assemble_pieces([r[0] for r in enc_a])
    got_b = sharding.assemble_pieces([r[0] for r in enc_b])
    assert got_a == want, "with reuse: " + _diff(got_a, want)
    assert got_b == want, "without reuse: " + _diff(got_b, want)
    assert [b - a for a, b in zip(la, lb)] == [1] * len(strips), (la, lb)


@pytest.mark.parametrize("timing", [False, True], ids=["graphs", "timing"])
def test_strip_coefficient_reuse_is_invalidated(timing):
    """Per strip, four fresh contexts with the same histogram results and the same strip encode:
    A: histogram, encode (reuses); B: histogram on a copy at another address, encode (recomputes);
    C: histogram, an unrelated encode on the same context, encode (recomputes: the coefficients were overwritten);
    D: histogram of the same pointer with other settings, encode (recomputes: the coefficients were quantized differently).
    All four files are exact; B, C and D take one launch more than A. With timing on (no graph replay) the reusing
    encode still reports the colour+DCT stage, which ran in its histogram call."""
    import jpeg_encoder_b200 as je
    from jpeg_encoder_b200 import sharding
    color, w, h, cfg, max_strips = REUSE_CASES["optimized_420"]
    other_cfg = dict(cfg, quality=60)
    img, strips, d_px, copies = _strip_inputs(color, w, h, cfg, max_strips)
    want = _want(("reuse", "optimized_420"), img, w, h, color, cfg)
    unrelated = np.random.default_rng(5).integers(0, 256, (222, 333, 3), dtype=np.uint8)  # noise: C's sizes stay generous
    unrelated_cfg = dict(quality=75, sampling=(2, 1), progressive_scans=3)
    unrelated_want = _want(("unrelated",), unrelated, 333, 222, "rgb", unrelated_cfg)
    n = len(strips)
    ctx = {k: [je.Device(0) for _ in strips] for k in "ABCD"}
    try:
        for devs in ctx.values():
            for dev in devs:
                dev.set_timing(timing)
        hists = {}
        for i in range(n):
            hists[("A", i)] = _rank_histogram(ctx["A"][i], cfg, color, w, h, strips, i, d_px[i])
            hists[("B", i)] = _rank_histogram(ctx["B"][i], cfg, color, w, h, strips, i, copies[i])
            hists[("C", i)] = _rank_histogram(ctx["C"][i], cfg, color, w, h, strips, i, d_px[i])
            _rank_histogram(ctx["D"][i], other_cfg, color, w, h, strips, i, d_px[i])
            got = make_encoder(unrelated_cfg, ctx["C"][i]).encode(unrelated, 333, 222, je.ColorType.Rgb)
            assert got == unrelated_want
        for k in "BC":
            assert [hists[(k, i)] for i in range(n)] == [hists[("A", i)] for i in range(n)]
        total = _merge(cfg, color, w, h, [hists[("A", i)] for i in range(n)])
        res = {k: [_rank_encode(ctx[k][i], cfg, color, w, h, strips, i, d_px[i], total) for i in range(n)] for k in "ABCD"}
    finally:
        for devs in ctx.values():
            for dev in devs:
                dev.close()
    counts = {k: [r[1] for r in v] for k, v in res.items()}
    print("timing %s: launches %r" % (timing, counts))
    for k, v in res.items():
        got = sharding.assemble_pieces([r[0] for r in v])
        assert got == want, "%s: %s" % (k, _diff(got, want))
        if timing:
            assert all(r[2] is not None and r[2]["colour_dct_quant"] > 0 for r in v), (k, [r[2] for r in v])
    for k in "BCD":
        assert [b - a for a, b in zip(counts["A"], counts[k])] == [1] * n, (k, counts)


# ---- one large packed image: uploaded in slices of whole MCU rows, the colour+DCT kernel runs per slice -------------
SLICE_MIN = 48 << 20  # a single packed image of at least this many bytes is uploaded in slices (api.cu)

SLICE_CASES = [
    ("rgb_2_4_partial_last_row", "rgb", 4099, 5650, dict(quality=90, sampling=(2, 4))),
    ("rgb_1_4", "rgb", 4099, 4105, dict(quality=85, sampling=(1, 4))),
    ("bgra_4_2", "bgra", 3001, 4203, dict(quality=80, sampling=(4, 2))),
    ("cmyk_1_4", "cmyk", 3001, 4203, dict(quality=90, sampling=(1, 4))),
    ("rgb_2_2_optimized_restart7", "rgb", 4099, 4097, dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=7)),
    ("luma_progressive5_restart3", "luma", 7001, 7203, dict(quality=92, sampling=(1, 1), progressive_scans=5, restart_interval=3)),
    ("threshold_exactly_48MiB", "luma", 6144, 8192, dict(quality=90, sampling=(1, 1))),
    ("threshold_one_row_fewer", "luma", 6144, 8191, dict(quality=90, sampling=(1, 1))),
]


def _slice_plan(color, w, h, cfg):
    """(number of slices, MCU rows per slice, MCU rows, MCU height in pixels) as the sliced upload cuts the image."""
    lay = make_encoder(cfg).coef_layout(w, h, CT[color][1])
    mcu_px = 8 * max(lay.comp_v[c] for c in range(lay.n_components))
    rows_per_slice = max(1, (32 << 20) // (w * BPP[color] * mcu_px))
    rows_per_slice = (rows_per_slice + 3) & ~3
    return (lay.mcu_rows + rows_per_slice - 1) // rows_per_slice, rows_per_slice, lay.mcu_rows, mcu_px


def test_slice_cases_cover_the_edges():
    """The geometry of SLICE_CASES (host only): every case but the lower threshold is sliced, at least twice; widths
    and heights off multiples of 16 except where the exact threshold needs them; one last slice is a single partial
    MCU row."""
    last_single_partial = False
    for name, color, w, h, cfg in SLICE_CASES:
        n, rps, mcu_rows, mcu_px = _slice_plan(color, w, h, cfg)
        size = w * h * BPP[color]
        if name.startswith("threshold"):
            assert size == SLICE_MIN if name.endswith("48MiB") else size == SLICE_MIN - w * BPP[color]
            continue
        assert size >= SLICE_MIN and n >= 2 and w % 16 and h % 16, name
        last_single_partial |= mcu_rows - (n - 1) * rps == 1 and h % mcu_px != 0
    assert last_single_partial


@pytest.mark.parametrize("name,color,w,h,cfg", SLICE_CASES, ids=[c[0] for c in SLICE_CASES])
def test_sliced_upload_of_one_large_image(name, color, w, h, cfg):
    """Encoder.encode of one large packed image, twice on a fresh context, against the oracle. The second call runs
    with learnt sizes; its launch count is that of the device-resident encode of the same image (second call on
    another fresh context) plus one colour+DCT launch for every slice after the first: that shows the image went
    through the sliced path exactly when it is at least 48 MiB."""
    import torch
    from test_gpu_parity import _torch_frame
    img = _torch_frame(w, h, BPP[color], seed=5)
    size = w * h * BPP[color]
    n_slices = _slice_plan(color, w, h, cfg)[0] if size >= SLICE_MIN else 1
    want = _want(("slice", name), img, w, h, color, cfg)
    ct = CT[color][1]
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        for k in range(2):
            got = enc.encode(img, w, h, ct)
            assert got == want, "host call %d: %s" % (k + 1, _diff(got, want))
        sliced = dev.last_launch_count()
    stride = (size + 255) & ~255
    d_in = torch.zeros(stride, dtype=torch.uint8, device="cuda")
    d_in[:size].copy_(torch.from_numpy(img.reshape(-1)))
    torch.cuda.synchronize()
    with _context() as dev:
        enc = make_encoder(cfg, dev)
        for k in range(2):
            d_files, offs = enc.encode_batch_device(d_in.data_ptr(), stride, 1, w, h, ct)
            got = dev.download(d_files, offs[-1])
            assert got == want, "device call %d: %s" % (k + 1, _diff(got, want))
        whole = dev.last_launch_count()
    del d_in
    torch.cuda.empty_cache()
    print("%s: %d slices, launches %d (device-resident %d)" % (name, n_slices, sliced, whole))
    assert sliced == whole + n_slices - 1, (sliced, whole, n_slices)


# ---- one context, a long mixed sequence ------------------------------------------------------------------------------
SEQ_SIZES = [(97, 75), (321, 243), (800, 601), (1283, 719)]
SEQ_CONFIGS = [  # default and optimized tables alternate as the sequence cycles through them
    ("rgb", dict(quality=90, sampling=(2, 2))),
    ("rgb", dict(quality=80, sampling=(2, 2), optimize_huffman=True, restart_interval=9)),
    ("rgb", dict(quality=85, sampling=(2, 1), progressive_scans=4, restart_interval=12)),
    ("rgb", dict(quality=75, sampling=(1, 1), optimize_huffman=True, restart_interval=5)),
    ("cmyk", dict(quality=88, sampling=(4, 1), restart_interval=8)),
]


def _sequence():
    """~40 calls: (kind, config index, size index). Kinds: host encode, planes, host batch, device batch, strips, and
    a pair of host encodes whose APP segments differ in their bytes but not in their length."""
    rng = np.random.default_rng(20261020)
    kinds = ["encode"] * 8 + ["planes"] * 6 + ["batch"] * 5 + ["device"] * 5 + ["strips"] * 6 + ["app_pair"] * 5
    kinds = [kinds[i] for i in rng.permutation(len(kinds))]
    return [(kind, i % len(SEQ_CONFIGS), int(rng.integers(len(SEQ_SIZES)))) for i, kind in enumerate(kinds)]


@pytest.mark.parametrize("poison", [False, True], ids=["plain", "poisoned"])
def test_long_mixed_sequence_on_one_context(poison, monkeypatch):
    """One context runs ~40 calls: more settings than the four cached graphs, so slots are evicted and revisited;
    default and optimized tables alternate; packed and planar input, host batches, device batches and strips
    interleave; sizes grow and shrink, so buffers are reallocated and graphs keyed on the old ones must miss; and a
    repeated call differs only in the bytes of a same-length APP segment, so its graph key is equal and the header must
    still be uploaded again. Every file is exact."""
    import torch
    import jpeg_encoder_b200 as je
    if poison:
        monkeypatch.setenv("JPGB_POISON_ALLOC", "1")
    failures, calls = [], 0
    with _context() as dev:
        for step, (kind, ci, si) in enumerate(_sequence()):
            color, cfg = SEQ_CONFIGS[ci]
            w, h = SEQ_SIZES[si]
            ch, ct = BPP[color], CT[color][1]
            results = []  # (what, got, want)
            if kind == "encode":
                img = _photo(w, h, ch, step % 3)
                results.append(("", make_encoder(cfg, dev).encode(img, w, h, ct), _want(("seq", step % 3), img, w, h, color, cfg)))
            elif kind == "app_pair":
                img = _photo(w, h, ch, 7)
                for k in range(2):
                    c = dict(cfg, app_segments=[(15, bytes([step, k]) * 20)])
                    results.append(("app %d" % k, make_encoder(c, dev).encode(img, w, h, ct), _want(("seq", 7), img, w, h, color, c)))
            elif kind == "planes":
                jct = je.JpegColorType.Cmyk if color == "cmyk" else je.JpegColorType.Ycbcr
                planes = [_photo(w, h, 1, 50 + c) for c in range(jct.get_num_components())]
                packed = np.stack(planes, -1)
                ref, rc = (255 - packed, "cmyk") if color == "cmyk" else (packed, "ycbcr")
                results.append(("", make_encoder(cfg, dev).encode_planes(planes, w, h, jct), _want(("seqplanes",), ref, w, h, rc, cfg)))
            elif kind == "batch":
                frames = [_photo(w, h, ch, 20 + k) for k in range(3)]
                outs = make_encoder(cfg, dev).encode_batch(frames, w, h, ct)
                results += [("file %d" % k, o, _want(("seq", 20 + k), f, w, h, color, cfg)) for k, (o, f) in enumerate(zip(outs, frames))]
            elif kind == "device":
                frames = [_photo(w, h, ch, 30 + k) for k in range(2 + step % 2)]
                stride = (w * h * ch + 255) & ~255
                d_in = torch.zeros(len(frames) * stride, dtype=torch.uint8, device="cuda")
                for k, f in enumerate(frames):
                    d_in[k * stride:k * stride + f.size].copy_(torch.from_numpy(f.reshape(-1)))
                torch.cuda.synchronize()
                d_files, offs = make_encoder(cfg, dev).encode_batch_device(d_in.data_ptr(), stride, len(frames), w, h, ct)
                blob = dev.download(d_files, offs[-1])
                results += [("file %d" % k, bytes(blob[offs[k]:offs[k + 1]]), _want(("seq", 30 + k), f, w, h, color, cfg)) for k, f in enumerate(frames)]
            else:
                if not cfg.get("restart_interval"):  # strips need restart intervals
                    color, cfg = SEQ_CONFIGS[1]
                img = _photo(w, h, BPP[color], 9)
                got, _, _ = _encode_strips(dev, img, w, h, color, cfg, 3)
                results.append(("", got, _want(("seq", 9), img, w, h, color, cfg)))
            calls += 1 if kind != "app_pair" else 2
            for what, got, want in results:
                if got != want:
                    failures.append("step %d %s %s %dx%d %r %s: %s" % (step, kind, color, w, h, cfg, what, _diff(got, want)))
    assert calls >= 40
    assert not failures, "\n".join(failures)
