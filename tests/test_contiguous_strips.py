"""One image in strips without restart intervals: the strip planner and the join arithmetic on the CPU, and on the GPU
every file byte-identical to the oracle's whole-image encode and to one jpgb_encode_batch_device call."""
import ctypes as C
import os
import random

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import images
import jpeg_encoder_b200 as je
from cases import BPP, CT, make_encoder, oracle_encode
from jpeg_encoder_b200 import sharding


def _enc(restart=0, sampling=je.SamplingFactor.F_2_2, progressive=None, optimize=False):
    e = je.Encoder(90)
    e.set_sampling_factor(sampling)
    e.set_restart_interval(restart)
    if progressive:
        e.set_progressive_scans(progressive)
    e.set_optimized_huffman_tables(optimize)
    return e


# ---- the planner (host only) ----------------------------------------------------------------------
@pytest.mark.parametrize("w,h,sampling,max_strips", [(1920, 1080, je.SamplingFactor.F_2_2, 8), (509, 397, je.SamplingFactor.F_2_2, 8),
                                                     (640, 24, je.SamplingFactor.F_1_1, 8), (100, 100, je.SamplingFactor.F_2_4, 3),
                                                     (16384, 16384, je.SamplingFactor.F_2_2, 8), (7, 7, je.SamplingFactor.F_4_1, 5),
                                                     (65535, 65535, je.SamplingFactor.F_1_1, 1000)])
def test_plan_contiguous_strips_invariants(w, h, sampling, max_strips):
    e = _enc(sampling=sampling)
    mcu_px = 8 * sampling.get_sampling_factors()[1]
    mcu_rows = (h + mcu_px - 1) // mcu_px
    strips = e.plan_contiguous_strips(w, h, je.ColorType.Rgb, max_strips)
    assert len(strips) == min(max_strips, mcu_rows)
    assert strips[0][0] == 0 and sum(n for _, n in strips) == h
    assert all(a[0] + a[1] == b[0] for a, b in zip(strips, strips[1:]))
    assert all(r % mcu_px == 0 for r, _ in strips)                  # whole MCU rows
    assert all(n % mcu_px == 0 for _, n in strips[:-1])
    mcu = [(n + mcu_px - 1) // mcu_px for _, n in strips]
    assert max(mcu) - min(mcu) <= 1                                   # sizes within one MCU row


def test_plan_contiguous_strips_refuses_restart_intervals():
    with pytest.raises(je.EncodingError):
        _enc(restart=64).plan_contiguous_strips(1920, 1080, je.ColorType.Rgb, 8)
    # the restart-aligned planner keeps refusing restart 0
    with pytest.raises(je.EncodingError):
        _enc().plan_strips(1920, 1080, je.ColorType.Rgb, 8)
    assert len(_enc(optimize=True, progressive=4).plan_contiguous_strips(1920, 1080, je.ColorType.Rgb, 8)) == 8


def test_plan_contiguous_strips_survives_arbitrary_params():
    """Whatever bytes a caller puts into jpgb_params: the same verdict as the other host entries, BAD_PARAMS when a
    restart interval is set, and strips that cover the image otherwise."""
    from jpeg_encoder_b200.encoder import _Params, _Strip
    lib = je.load_library()
    rnd = random.Random(11)
    seen = set()
    for _ in range(4000):
        p = _Params()
        raw = (C.c_uint8 * C.sizeof(p)).from_buffer(p)
        for i in range(C.sizeof(p)):
            raw[i] = rnd.getrandbits(8) if rnd.random() < 0.5 else rnd.choice([0, 1, 2, 4, 0x11, 0x22, 0x41, 9, 255])
        p.n_app, p.apps = 0, None
        if rnd.random() < 0.7:
            p.color_type = rnd.randrange(0, 11)
            p.sampling = rnd.choice([0x11, 0x12, 0x21, 0x22, 0x41, 0x42, 0x14, 0x24, 0x44, 0x00, 0xA2])
            p.progressive_scans = rnd.choice([0, 1, 2, 4, 64, 65])
            p.qtable_kind[0], p.qtable_kind[1] = rnd.randrange(0, 12), rnd.randrange(0, 12)
        if rnd.random() < 0.5:
            p.restart_interval = 0
        ns = C.c_uint32()
        arr, k = (_Strip * 9)(), C.c_uint32()
        r1 = lib.jpgb_scan_count(C.byref(p), C.byref(ns))
        r2 = lib.jpgb_plan_contiguous_strips(C.byref(p), 9, arr, C.byref(k))
        assert r2 == r1 or (r1 == 0 and r2 == 5 and p.restart_interval != 0)
        if r2 == 0:
            assert p.restart_interval == 0 and 1 <= k.value <= 9
            assert arr[0].first_row == 0 and sum(arr[i].rows for i in range(k.value)) == p.height
        seen.add(r2)
    assert seen == {0, 2, 5}


# ---- the join arithmetic (csrc/gather.cu, csrc/entropy.cu), restated and checked against plain bit concatenation ----
def _bits_to_words(bitstr, first_bit, n_words):
    """bit string placed at first_bit of a zeroed stream of n_words 32-bit big-endian words -> list of ints"""
    v = int(bitstr, 2) << (n_words * 32 - first_bit - len(bitstr)) if bitstr else 0
    return [(v >> (32 * (n_words - 1 - i))) & 0xFFFFFFFF for i in range(n_words)]


def _join_stream(pieces, leads_bytes):
    """What rank 0's stream holds after every rank stored its owned words and side words and rank 0 wrote leads, zeroed
    the shared words, ORed the side words and the pad bits: built the way the kernels build it."""
    world, n = len(pieces), len(pieces[0])
    table = [[len(pieces[r][k]) for k in range(n)] for r in range(world)]
    dest, _, total = sharding.join_destinations(table, [len(l) for l in leads_bytes])
    n_words = (total + 3) // 4 + 1
    stream = [random.getrandbits(32) for _ in range(n_words)]  # whatever the target held before
    side = []
    for r in range(world):  # ranks: owned words stored, shared words to the side table
        for k in range(n):
            words = _bits_to_words(pieces[r][k], dest[r][k], n_words)
            owned, shared = sharding.join_words(dest[r][k], table[r][k])
            for w in owned:
                stream[w] = words[w]
            side += [(w, words[w]) for w in shared]
    # rank 0: leads byte-wise, shared words zeroed (only their data bytes), side words and pad bits ORed, EOI
    b = bytearray(b"".join(w.to_bytes(4, "big") for w in stream))
    at = 0
    for k in range(n):
        b[at:at + len(leads_bytes[k])] = leads_bytes[k]
        at += len(leads_bytes[k])
        end_bit = at * 8 + sum(table[r][k] for r in range(world))
        data1 = (end_bit + 7) // 8
        bounds = [dest[r][k] for r in range(world)] + [end_bit]
        for q in bounds:
            if q % 32:
                w = q // 32
                for x in range(max(w * 4, at), min(w * 4 + 4, data1)):
                    b[x] = 0
        pad = -(end_bit - at * 8) % 8
        if pad:
            b[data1 - 1] |= (1 << pad) - 1
        at = data1
    for w, v in side:
        for i in range(4):
            b[4 * w + i] |= (v >> (24 - 8 * i)) & 0xFF
    b[at:at + 2] = b"\xff\xd9"
    return bytes(b[:total])


def _concat_stream(pieces, leads_bytes):
    out = b""
    for k in range(len(pieces[0])):
        bits = "".join(pieces[r][k] for r in range(len(pieces)))
        bits += "1" * (-len(bits) % 8)
        out += leads_bytes[k] + int(bits, 2).to_bytes(len(bits) // 8, "big") if bits else leads_bytes[k]
    return out + b"\xff\xd9"


def test_join_arithmetic_equals_bit_concatenation():
    rnd = random.Random(5)
    random.seed(6)
    for world, n_scans in ((1, 1), (2, 3), (3, 1), (8, 12), (5, 7)):
        for _ in range(20):
            pieces = [["".join(rnd.choice("01") for _ in range(rnd.choice([0, 1, 7, 8, 31, 32, 33, 64, rnd.randint(1, 300)])))
                       for _ in range(n_scans)] for _ in range(world)]
            leads = [bytes(rnd.getrandbits(8) for _ in range(rnd.randint(1, 40) if k else rnd.randint(100, 700))) for k in range(n_scans)]
            assert _join_stream(pieces, leads) == _concat_stream(pieces, leads)


def test_join_source_offsets_are_16_byte_pieces():
    dest, src, total = sharding.join_destinations([[1, 128, 129, 0, 5]], [10, 2, 2, 2, 2])
    assert src == [[0, 16, 32, 64, 64]]
    assert dest[0][0] == 80 and dest[0][1] == (10 + 1 + 2) * 8 and total == 10 + 1 + 2 + 16 + 2 + 17 + 2 + 0 + 2 + 1 + 2


def _join_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rnd = random.Random(100 + rank)
    mine = ["".join(rnd.choice("01") for _ in range(rnd.randint(1, 200))) for _ in range(4)]
    edges = sharding.exchange_edge_dc([rank * 100 + i for i in range(8)], torch.device("cpu"))
    assert edges == [r * 100 + i for r in range(world) for i in range(8)]
    t = torch.tensor([len(b) for b in mine], dtype=torch.int64)
    table = torch.empty(world * 4, dtype=torch.int64)
    dist.all_gather_into_tensor(table, t)
    table = table.view(world, 4).tolist()
    leads = [600, 10, 10, 10]
    dest, _, total = sharding.join_destinations(table, leads)
    words = {}
    for k in range(4):
        n_words = (total + 3) // 4 + 1
        ws = _bits_to_words(mine[k], dest[rank][k], n_words)
        owned, shared = sharding.join_words(dest[rank][k], table[rank][k])
        words[k] = ([(w, ws[w]) for w in owned], [(w, ws[w]) for w in shared])
    q.put((rank, mine, words, total))
    dist.destroy_process_group()


def test_join_positions_gloo_world2():
    """Each rank works out its pieces' positions from the all-gathered table alone; together their owned and shared
    words make the concatenated bit strings."""
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_join_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    got.sort()
    totals = {g[3] for g in got}
    assert len(totals) == 1
    total = totals.pop()
    n_words = (total + 3) // 4 + 1
    stream = [0] * n_words
    for _, _, words, _ in got:
        for k in words:
            for w, v in words[k][0]:
                assert stream[w] == 0
                stream[w] = v
            for w, v in words[k][1]:
                stream[w] |= v
    b = b"".join(w.to_bytes(4, "big") for w in stream)
    pieces = [g[1] for g in got]
    at = 600
    for k in range(4):
        bits = "".join(pieces[r][k] for r in range(world))
        val = int.from_bytes(b, "big") >> (len(b) * 8 - at * 8 - len(bits)) & ((1 << len(bits)) - 1)
        assert val == int(bits, 2)
        at = (at * 8 + len(bits) + 7) // 8 + 10


# ---- on the GPU ------------------------------------------------------------------------------------
def _contiguous_join(img, w, h, color, cfg, max_strips, device=None, want_stream=False):
    """Every rank's role on one GPU, one after the other: prepare every strip, gather the edge DCs (and histograms),
    encode every strip to learn the bit table, then encode each again and place it as rank i, then finish as rank 0."""
    enc = make_encoder(cfg, device)
    dev = enc._dev()
    ct = CT[color][1]
    strips = enc.plan_contiguous_strips(w, h, ct, max_strips)
    n = len(strips)
    flat = np.ascontiguousarray(img).reshape(h, -1)
    d_px = [torch.from_numpy(flat[r0:r0 + rows].copy()).cuda() for r0, rows in strips]
    torch.cuda.synchronize()
    hists, edges = [], []
    for i, (r0, rows) in enumerate(strips):
        hi, ed = enc.contiguous_strip_prepare_device(d_px[i].data_ptr(), i, n, r0, rows, w, h, ct)
        hists.append(hi)
        edges += ed
    hist_total = None
    if cfg.get("optimize_huffman"):
        hist_total = enc.merge_strip_histograms([sum(col) for col in zip(*hists)], edges, w, h, ct)
    table = []
    for i, (r0, rows) in enumerate(strips):
        enc.encode_contiguous_strip_device(d_px[i].data_ptr(), i, n, r0, rows, w, h, ct, edges, hist_total=hist_total)
        d_bits, n_scans = enc.piece_bits_device()
        table.append(list(np.frombuffer(dev.download(d_bits, n_scans * 8), dtype=np.int64)))
    cap = w * h * BPP[color] + (1 << 20)
    target, handle = C.c_void_p(), (C.c_uint8 * 64)()
    assert dev.lib.jpgb_gather_target_create(dev.handle, cap, C.byref(target), handle) == 0, dev.last_error()
    d_table = torch.tensor([v for row in table for v in row], dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    try:
        for i, (r0, rows) in enumerate(strips):
            enc.encode_contiguous_strip_device(d_px[i].data_ptr(), i, n, r0, rows, w, h, ct, edges, hist_total=hist_total)
            enc.join_place_bits(target.value, cap, d_table.data_ptr(), n, i)
        d_file, length = enc.join_finish_device(target.value, cap, d_table.data_ptr(), n, w, h, ct, hist_total=hist_total)
        got = dev.download(d_file, length)
        stream = None
        if want_stream:
            side = ((n * len(table[0]) * 2 * 16) + 127) // 128 * 128
            stream = dev.download(target.value + side, cap - side)
    finally:
        assert dev.lib.jpgb_gather_target_close(dev.handle, target, 0) == 0
    return got, n, table, stream


def _batch_device(img, w, h, color, cfg):
    enc = make_encoder(cfg)
    dev = enc._dev()
    d = torch.from_numpy(np.ascontiguousarray(img).reshape(-1)).cuda()
    torch.cuda.synchronize()
    d_files, offs = enc.encode_batch_device(d.data_ptr(), d.numel(), 1, w, h, CT[color][1])
    return dev.download(d_files, offs[1])


def _img(color, w, h, seed=21):
    return images.photo_like(w, h, BPP[color], seed=seed)


CASES = [
    ("rgb_420", "rgb", 640, 480, dict(quality=85, sampling=(2, 2)), 5),
    ("rgb_422", "rgb", 512, 256, dict(quality=90, sampling=(2, 1)), 4),
    ("rgb_444", "rgb", 384, 200, dict(quality=95, sampling=(1, 1)), 6),
    ("sequential_411", "rgb", 512, 256, dict(quality=75, sampling=(4, 1)), 4),
    ("luma", "luma", 384, 512, dict(quality=95), 8),
    ("cmyk", "cmyk", 256, 320, dict(quality=90, sampling=(2, 2)), 5),
    ("cmyk_as_ycck", "cmyk_as_ycck", 320, 256, dict(quality=90, sampling=(1, 2)), 4),
    ("progressive_2", "rgb", 512, 400, dict(quality=85, sampling=(2, 2), progressive_scans=2), 4),
    ("progressive_4", "rgb", 512, 400, dict(quality=85, sampling=(2, 2), progressive_scans=4), 8),
    ("progressive_64", "rgb", 256, 256, dict(quality=90, sampling=(2, 2), progressive_scans=64), 3),
    ("optimized", "rgb", 512, 400, dict(quality=85, sampling=(2, 2), optimize_huffman=True), 4),
    ("optimized_progressive", "rgb", 384, 384, dict(quality=70, sampling=(2, 1), optimize_huffman=True, progressive_scans=5), 8),
    ("optimized_luma", "luma", 256, 256, dict(quality=80, optimize_huffman=True), 3),
    ("odd_size", "rgb", 509, 397, dict(quality=85, sampling=(2, 2), progressive_scans=4), 8),
    ("one_mcu_row_strips", "rgb", 200, 64, dict(quality=90, sampling=(2, 2)), 4),
    ("more_strips_than_rows", "luma", 96, 40, dict(quality=90), 64),
    ("one_strip", "rgb", 320, 240, dict(quality=90, sampling=(2, 2)), 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,color,w,h,cfg,max_strips", CASES, ids=[c[0] for c in CASES])
def test_contiguous_strips_equal_the_whole_image(name, color, w, h, cfg, max_strips):
    img = _img(color, w, h)
    got, n, _, _ = _contiguous_join(img, w, h, color, cfg, max_strips)
    mcu_px = 8 * (cfg.get("sampling") or (1, 1))[1] if color != "luma" else 8
    assert n == min(max_strips, (h + mcu_px - 1) // mcu_px)
    want = oracle_encode(img, w, h, color, cfg)
    assert got == want
    assert got == _batch_device(img, w, h, color, cfg)


@pytest.mark.gpu
def test_join_with_a_stuffed_ff_across_a_bit_boundary():
    """High-quality noise in 64 one-MCU-row strips of 64 scans: at some join whose bit position is not a byte boundary,
    the byte that straddles it is 0xFF (stuffed as FF 00 on the root)."""
    w, h, color = 512, 512, "luma"
    cfg = dict(quality=100, progressive_scans=64)
    img = np.random.default_rng(3).integers(0, 256, (h, w), dtype=np.uint8)
    got, n, table, stream = _contiguous_join(img, w, h, color, cfg, 64, want_stream=True)
    assert n == 64
    assert got == oracle_encode(img, w, h, color, cfg)
    enc = make_encoder(cfg)
    leads = [len(enc.build_header(w, h, je.ColorType.Luma))] + [10] * (len(table[0]) - 1)  # single-component SOS
    dest, _, _ = sharding.join_destinations(table, leads)
    straddling = [(r, k) for r in range(1, n) for k in range(len(table[0])) if dest[r][k] % 8 and stream[dest[r][k] // 8] == 0xFF]
    assert straddling, "no 0xFF byte straddles a join: the case is not exercised"


@pytest.mark.gpu
def test_category_11_dc_jump_across_a_join():
    w, h, color = 64, 64, "luma"
    img = np.zeros((h, w), np.uint8)
    img[32:] = 255
    cfg = dict(quality=100)
    got, n, _, _ = _contiguous_join(img, w, h, color, cfg, 2)
    assert n == 2
    assert got == oracle_encode(img, w, h, color, cfg)


@pytest.mark.gpu
def test_config5_without_restarts_full_size_8_strips_one_gpu():
    """16384 x 16384 RGB progressive 4:2:0 with restart interval 0 in 8 strips: the whole image's file."""
    from test_gpu_parity import _torch_frame
    w = h = 16384
    cfg = dict(quality=90, sampling=(2, 2), progressive_scans=4)
    img = _torch_frame(w, h, 3, seed=7)
    got, n, _, _ = _contiguous_join(img, w, h, "rgb", cfg, 8)
    assert n == 8
    want = oracle_encode(img, w, h, "rgb", cfg)
    assert len(got) == len(want) and got == want


@pytest.mark.gpu
@pytest.mark.parametrize("env", [("JPGB_TIGHT_CAPS", "pool,stream,out"), ("JPGB_POISON_ALLOC", "1")])
def test_one_context_alternates_strip_paths_and_batches(env, monkeypatch):
    """One context: restart-aligned strips, contiguous strips and a device batch, twice over; every file stays right
    (no stale DC predictor from a replayed graph, no coefficients taken across paths)."""
    monkeypatch.setenv(*env)
    dev = je.Device(0)
    try:
        w, h, color = 512, 384, "rgb"
        img = _img(color, w, h, seed=9)
        cfg0 = dict(quality=85, sampling=(2, 2), progressive_scans=4)
        cfg_r = dict(cfg0, restart_interval=32)
        cfg_o = dict(quality=85, sampling=(2, 2), optimize_huffman=True)
        want0, want_r, want_o = (oracle_encode(img, w, h, color, c) for c in (cfg0, cfg_r, cfg_o))
        for _ in range(2):
            assert _contiguous_join(img, w, h, color, cfg0, 4, device=dev)[0] == want0
            d = torch.from_numpy(np.ascontiguousarray(img).reshape(-1)).cuda()
            torch.cuda.synchronize()
            enc = make_encoder(cfg0, dev)
            d_files, offs = enc.encode_batch_device(d.data_ptr(), d.numel(), 1, w, h, CT[color][1])
            assert dev.download(d_files, offs[1]) == want0
            assert _contiguous_join(img, w, h, color, cfg_o, 3, device=dev)[0] == want_o
            assert _restart_aligned_strips(img, w, h, color, cfg_r, 4, dev) == want_r
            assert _contiguous_join(img, w, h, color, cfg0, 6, device=dev)[0] == want0
    finally:
        dev.close()


def _restart_aligned_strips(img, w, h, color, cfg, max_strips, dev):
    enc = make_encoder(cfg, dev)
    ct = CT[color][1]
    strips = enc.plan_strips(w, h, ct, max_strips)
    assert len(strips) > 1
    flat = np.ascontiguousarray(img).reshape(h, -1)
    pieces = []
    for i, (r0, rows) in enumerate(strips):
        d = torch.from_numpy(flat[r0:r0 + rows].copy()).cuda()
        torch.cuda.synchronize()
        d_bytes, offs = enc.encode_strip_device(d.data_ptr(), i, len(strips), r0, rows, w, h, ct)
        pieces.append(sharding.split_pieces(dev.download(d_bytes, offs[-1]), offs))
    return sharding.assemble_pieces(pieces)


def _nccl_worker(rank, world, port, w, h, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        dev_t = torch.device("cuda", rank)
        stream = torch.cuda.Stream(device=dev_t)
        torch.cuda.set_stream(stream)
        device = je.Device(rank, cuda_stream=stream.cuda_stream)
        cfg = dict(quality=90, sampling=(2, 2), progressive_scans=4)
        enc = make_encoder(cfg, device)
        img = images.photo_like(w, h, 3, seed=4)
        strips = enc.plan_contiguous_strips(w, h, je.ColorType.Rgb, world)
        r0, rows = strips[rank]
        d_px = torch.from_numpy(np.ascontiguousarray(img).reshape(h, -1)[r0:r0 + rows].copy()).to(dev_t)
        _, edge = enc.contiguous_strip_prepare_device(d_px.data_ptr(), rank, world, r0, rows, w, h, je.ColorType.Rgb)
        edges = sharding.exchange_edge_dc(edge, dev_t)
        pg = sharding.PeerGather(device, w * h * 3 + (1 << 20), rank, world, dev_t)
        enc.encode_contiguous_strip_device(d_px.data_ptr(), rank, world, r0, rows, w, h, je.ColorType.Rgb, edges)
        pg.gather_bits(enc)
        pg.barrier()
        if rank == 0:
            got = bytes(pg.finish_bits(enc, w, h, je.ColorType.Rgb).cpu().numpy().tobytes())
            q.put(got == oracle_encode(img, w, h, "rgb", cfg))
        torch.cuda.synchronize()
        dist.barrier()
        pg.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2 if torch.cuda.is_available() else True, reason="needs two GPUs")
def test_contiguous_strips_nccl_world2():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, port, 640, 480, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        assert q.get(timeout=300) is True
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.kill()
                p.join()
    assert all(p.exitcode == 0 for p in procs)
