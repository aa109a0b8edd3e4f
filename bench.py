#!/usr/bin/env python
"""bench.py -- megapixels/s of the JPEG encode hot path on N B200s (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c1|c2|c4a|c4b|c5] [--impl reference]
                    [--dump-outputs DIR]

A step = one pass of the whole encode path (colour -> DCT -> quant -> entropy -> stuffed JFIF bytes)
over one batch of synthetic frames. Default workload: BASELINE config 3, a batch of 1920x1080 RGB
frames, q=90, 4:2:0, standard Huffman tables: a FIXED batch of 1024 frames sharded by image over the ranks
(strong scaling, no data-path collective; the weak variant -- 1024 frames on every GPU -- is reported beside it
under `weak` at N > 1). The same line carries `c5`: BASELINE config 5, one 16384^2 progressive image cut into
restart-aligned strips, one per GPU, pieces gathered to rank 0 over NVLink -- the only path with a data collective --
parity-gated against the oracle. `value` is measured with inputs resident in HBM; `e2e` goes
through the host-buffer C ABI (pinned host pixels in, host JPEG bytes out, copies inside the timed
region). `roofline` is the colour+DCT+quant kernel against the measured HBM peak. `cpu_baseline`
is the CPU restatement of the reference (oracle/) on the host cores: a reported baseline, not the
target. `--impl reference` times only that CPU restatement (the Rust crate cannot be built here:
no Rust toolchain in the image).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (width, height, color, cfg, default batch per GPU, description)
    "c1": (1920, 1080, "rgb", dict(quality=90, sampling=(2, 2)), 1, "1 x 1920x1080 RGB q90 4:2:0 baseline (BASELINE config 1)"),
    "c2": (4096, 4096, "rgb", dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=64), 1,
           "1 x 4096x4096 RGB q85 4:2:0 optimized Huffman, restart 64 (BASELINE config 2)"),
    "c3": (1920, 1080, "rgb", dict(quality=90, sampling=(2, 2)), 1024,
           "batch of 1920x1080 RGB q90 4:2:0 baseline frames, sharded by image (BASELINE config 3)"),
    "c3o": (1920, 1080, "rgb", dict(quality=90, sampling=(2, 2), optimize_huffman=True), 1024,
            "batch of 1920x1080 RGB q90 4:2:0 frames with per-image optimized Huffman tables (histogram + Annex K.2 on the device)"),
    # formats outside the BASELINE configurations (SURVEY 8f rank 4): verbatim / inverted byte formats on the warp kernel,
    # a factor-4 sampling and 4:4:4
    "x_ycbcr": (1920, 1080, "ycbcr", dict(quality=90, sampling=(2, 2)), 256, "batch of 1920x1080 YCbCr (verbatim) q90 4:2:0 baseline frames"),
    "x_cmyk": (4096, 4096, "cmyk", dict(quality=90, sampling=(2, 2)), 16, "batch of 4096x4096 CMYK (inverted) q90, K at 2x2, baseline frames"),
    "x_ycck": (4096, 4096, "ycck", dict(quality=90, sampling=(1, 1)), 16, "batch of 4096x4096 YCCK (verbatim) q90 4:4:4 baseline frames"),
    "x_rgb411": (1920, 1080, "rgb", dict(quality=90, sampling=(4, 1)), 256, "batch of 1920x1080 RGB q90 4:1:1 (factor 4: sequential scans)"),
    "x_rgb444": (1920, 1080, "rgb", dict(quality=90, sampling=(1, 1)), 256, "batch of 1920x1080 RGB q90 4:4:4 baseline frames (the crate's default sampling for quality >= 90)"),
    "c4a": (8192, 8192, "luma", dict(quality=95, sampling=(1, 1), qtables="custom"), 1,
            "1 x 8192x8192 grayscale q95 custom tables (BASELINE config 4a)"),
    "c4b": (8192, 8192, "cmyk_as_ycck", dict(quality=95, sampling=(1, 1), qtables="custom"), 1,
            "1 x 8192x8192 CMYK->YCCK q95 4:4:4 custom tables (BASELINE config 4b)"),
    "c5": (16384, 16384, "rgb", dict(quality=90, sampling=(2, 2), progressive_scans=4, restart_interval=2048), 1,
           "1 x 16384x16384 RGB progressive (4 scans per component, spectral selection) 4:2:0, restart 2048, "
           "split by restart-aligned strips across the GPUs, pieces gathered to rank 0 (BASELINE config 5)"),
    "c5o": (16384, 16384, "rgb", dict(quality=85, sampling=(2, 2), optimize_huffman=True, restart_interval=2048), 1,
            "1 x 16384x16384 RGB 4:2:0 optimized Huffman tables, restart 2048, split by restart-aligned strips: symbol "
            "histograms all-reduced over NCCL, pieces gathered to rank 0 (SURVEY 8e, optimized variant of config 5)"),
}
BPP = {"luma": 1, "rgb": 3, "cmyk_as_ycck": 4, "ycbcr": 3, "cmyk": 4, "ycck": 4}
DISTINCT = 16  # distinct synthetic frames; the batch repeats them (inputs stay >> L2: 6.2 MB per frame)


def custom_table():
    """fixed non-preset table, all values 1..255 so the file still decodes (SURVEY.md 8d)"""
    return [min(255, 2 + ((i % 8) + (i // 8)) * 3 + (i * 7) % 5) for i in range(64)]


def resolve_cfg(cfg):
    cfg = dict(cfg)
    if cfg.get("qtables") == "custom":
        t = custom_table()
        cfg["qtables"] = (t, t)
    return cfg


def frames_for(width, height, color, n_distinct):
    import images
    return [images.synth_frame(width, height, BPP[color], seed=s) for s in range(n_distinct)]


DUMP_WINDOW = 1 << 15  # bytes per window of a sampled dump
DUMP_BUDGET = 8 << 20  # bytes of the timed path's stream per dump (x4 as float32); the config-5 leg of the default line adds half


def dump_outputs(out_dir, name, d_bytes, offsets, budget):
    """--dump-outputs: what a caller of the timed path receives from one step -- the JPEG files back to back in
    device memory (`d_bytes`, uint8) and the file offsets -- written as <name>_offsets.npy (float64, every file) and
    <name>_bytes.npy (float32). A stream longer than `budget` bytes is sampled: budget / DUMP_WINDOW windows of
    DUMP_WINDOW contiguous bytes at starts drawn from a fixed seed (<name>_window_starts.npy, float64), so two builds
    that produce the same stream dump the same arrays."""
    import torch
    n = int(offsets[-1])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + "_offsets.npy"), np.asarray(offsets, dtype=np.float64))
    if n <= budget:
        data = d_bytes[:n]
    else:
        starts = np.sort(np.random.default_rng(20261020).integers(0, n - DUMP_WINDOW + 1, budget // DUMP_WINDOW))
        np.save(os.path.join(out_dir, name + "_window_starts.npy"), starts.astype(np.float64))
        idx = torch.from_numpy(starts[:, None] + np.arange(DUMP_WINDOW)).to(d_bytes.device)
        data = d_bytes[idx]
    np.save(os.path.join(out_dir, name + "_bytes.npy"), data.cpu().numpy().astype(np.float32))


def stage_a_bytes(width, height, color, cfg):
    """Algorithmic bytes of the colour+DCT+quant kernel per image: w*h*bpp read + 128 B per block written
    (SURVEY.md 8d; block counts as src/encoder.rs:713-717)."""
    import jpeg_encoder_b200 as je
    from cases import CT, make_encoder
    lay = make_encoder(cfg).coef_layout(width, height, CT[color][1])
    return width * height * BPP[color] + 128 * int(lay.blocks_per_image)


# ---- CPU baseline (oracle) ------------------------------------------------------------------------
def cpu_encode_rate(frames, width, height, color, cfg, seconds, threads):
    """One encode per thread on `threads` host threads for about `seconds`; returns (MP/s, frames done)."""
    from cases import CT
    from oracle import oracle as orc
    orc.lib(native=True)  # built with -march=native on the machine that times it
    ct = CT[color][0]
    if orc.has_simd(native=True):  # AVX2 colour + fDCT where the reference's `simd` feature has its own; same bytes, checked here
        orc.set_simd(False, native=True)
        plain = orc.encode(frames[0], width, height, ct, native=True, **cfg)
        orc.set_simd(True, native=True)
        if orc.encode(frames[0], width, height, ct, native=True, **cfg) != plain:
            raise SystemExit("bench.py: the oracle's AVX2 path differs from its scalar path")
    done = [0] * threads
    stop = time.perf_counter() + seconds

    def work(i):
        k = i
        while True:
            orc.encode(frames[k % len(frames)], width, height, ct, native=True, **cfg)
            done[i] += 1
            k += threads
            if time.perf_counter() >= stop:
                break

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    n = sum(done)
    return n * width * height / 1e6 / dt, n


def usable_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# ---- clocks ---------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out = self.proc.communicate()[0]
        sm, mx, reasons = [], None, set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm_sorted = sorted(sm)
        # median of the samples taken under load = upper half of the distribution
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "how": "nvidia-smi every 50 ms from the warm-up through the timed steps plus ~1 s of the same work un-timed; median of the upper half"}


def bind_to_gpu_numa_node(local):
    """Host side of the end-to-end path: every rank's pinned staging memory and its copy threads should live on the
    NUMA node its GPU hangs off, or the uploads of 8 ranks fight over the socket interconnect. Binds this process to
    the CPUs of that node (first-touch then places the pinned pages there) and returns what it did for the JSON line."""
    info = {"bound": False}
    try:
        import torch
        props = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        info.update(pci=bdf, numa_node=node)
        if node < 0:
            return info
        cpulist = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info.update(bound=True, cpus=cpulist, n_cpus=len(allowed))
    except (OSError, ValueError, AttributeError) as e:
        info["error"] = str(e)[:120]
    return info


# ---- the product arm ------------------------------------------------------------------------------
def run_product(args):
    import torch
    import torch.distributed as dist
    import jpeg_encoder_b200 as je
    from cases import CT, make_encoder

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev_t = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"bound": False, "note": "single rank: not bound"}

    width, height, color, cfg, def_batch, desc = WORKLOADS[args.workload]
    cfg = resolve_cfg(cfg)
    if args.workload in ("c5", "c5o"):
        return run_strips(args, rank, world, local, dev_t)
    bpp = BPP[color]
    img_bytes = width * height * bpp
    # BASELINE config 3 is a FIXED batch sharded by image: rank r owns shard_batch(total, world, r) (strong scaling).
    # `--batch` overrides the total. The weak variant (the whole batch on every GPU) is reported beside it at N > 1.
    from jpeg_encoder_b200 import sharding
    total_frames = args.batch or def_batch
    lo, hi = sharding.shard_batch(total_frames, world, rank)
    batch = hi - lo
    if batch == 0:
        raise SystemExit("bench.py: fewer frames than ranks")
    weak_batch = total_frames if (world > 1 and args.workload == "c3" and not args.no_weak) else 0
    resident = max(batch, weak_batch)

    n_distinct = min(DISTINCT, total_frames)
    frames = frames_for(width, height, color, n_distinct)
    # frame i of the global batch is distinct frame i % n_distinct
    order_global = [i % n_distinct for i in range(total_frames)]
    order = order_global[lo:hi]
    order_weak = [(i + rank) % n_distinct for i in range(weak_batch)]

    # a stream of our own (the legacy default stream cannot be captured into the CUDA graph the library replays)
    stream = torch.cuda.Stream(device=dev_t)
    torch.cuda.set_stream(stream)
    device = je.Device(local, cuda_stream=stream.cuda_stream)
    enc = make_encoder(cfg, device)
    ct = CT[color][1]

    # inputs resident in HBM (image stride padded to 256 B)
    stride = (img_bytes + 255) & ~255
    d_in = torch.empty(resident * stride, dtype=torch.uint8, device=dev_t)
    d_distinct = [torch.from_numpy(f.reshape(-1)).to(dev_t) for f in frames]

    def fill(order_):
        for i, k in enumerate(order_):
            d_in[i * stride:i * stride + img_bytes].copy_(d_distinct[k])
        torch.cuda.synchronize()

    fill(order)

    # parity gate (un-timed): EVERY file of the device-resident batch -- the path that is timed below -- must equal
    # the oracle's bytes; the files are brought back once and compared one by one
    from cases import oracle_encode
    want = [oracle_encode(f, width, height, color, cfg) for f in frames]
    d_files, offs = enc.encode_batch_device(d_in.data_ptr(), stride, batch, width, height, ct)
    total = offs[-1]
    blob = device.download(d_files, total)
    for i in range(batch):
        if blob[offs[i]:offs[i + 1]] != want[order[i]]:
            raise SystemExit("bench.py: device-batch file %d differs from the oracle -- number would be invalid" % (lo + i))
    del blob
    check = sorted(set([0, batch // 2, batch - 1]))[:3]
    out_bytes_per_step = int(total)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    rank_ms = []

    def timed_device(n_frames, stage_timers=False, dump=False):
        """K timed steps of the device-resident path over the first n_frames resident frames: (ms per step max over
        ranks, per-stage ms, launches). With stage_timers the library brackets every stage with CUDA events (and
        launches kernel by kernel instead of replaying its CUDA graph): used for the breakdown, not for `value`.
        With dump and --dump-outputs, rank 0 writes the files of the last timed step."""
        device.set_timing(stage_timers)
        for _ in range(args.warmup):
            enc.encode_batch_device(d_in.data_ptr(), stride, n_frames, width, height, ct)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage_ms_, launches_ = {}, 0
        e0.record(stream)
        for _ in range(args.steps):
            d_files_, offs_ = enc.encode_batch_device(d_in.data_ptr(), stride, n_frames, width, height, ct)
            launches_ += device.last_launch_count()
            for k, v in (device.last_timing() or {}).items():
                stage_ms_[k] = stage_ms_.get(k, 0.0) + v
        e1.record(stream)
        barrier()
        if dump and args.dump_outputs and rank == 0:  # before the next call on the context reuses its output buffer
            dump_outputs(args.dump_outputs, "files", _as_tensor(d_files_, offs_[-1], dev_t), offs_, DUMP_BUDGET)
        ms_ = e0.elapsed_time(e1)
        if world > 1:
            t_ = torch.tensor([ms_], device=dev_t)
            all_ = [torch.zeros_like(t_) for _ in range(world)]
            dist.all_gather(all_, t_)
            rank_ms[:] = [float(x.item()) / args.steps for x in all_]  # every rank's own time: shows a straggler
            ms_ = max(float(x.item()) for x in all_)
        return ms_ / args.steps, stage_ms_, launches_

    # ---- device-resident timing ----
    # the clock sampler (an nvidia-smi process) is started before the warm-up: its start-up initialises NVML on every
    # GPU of the box and takes driver locks for tens of ms, which must not land inside the timed region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    ms_per_step, _, launches = timed_device(batch, dump=True)
    rank_ms_value = list(rank_ms)
    _, stage_ms, _ = timed_device(batch, stage_timers=True)  # second pass: per-stage breakdown and the roofline numerator
    device.set_timing(False)
    if rank == 0:
        # the timed region is tens of milliseconds: keep the same work running (un-timed) for about a
        # second so that the 50 ms clock samples are taken under this load
        t_obs = time.perf_counter()
        while time.perf_counter() - t_obs < 1.0:
            enc.encode_batch_device(d_in.data_ptr(), stride, batch, width, height, ct)
    clocks = sampler.stop() if rank == 0 else None
    barrier()
    mp_per_step = total_frames * width * height / 1e6  # whole job: all ranks' frames
    value = mp_per_step / (ms_per_step / 1e3)

    weak = None
    if weak_batch:
        fill(order_weak)
        w_ms, _, _ = timed_device(weak_batch)
        weak = {"frames_per_gpu": weak_batch, "ms_per_step": w_ms, "value": weak_batch * world * width * height / 1e6 / (w_ms / 1e3),
                "unit": "megapixels/s", "note": "every GPU encodes its own %d frames (per-GPU work fixed as N grows)" % weak_batch}
        fill(order)

    # ---- end to end through the host-buffer C ABI (pinned pixels in, host bytes out) ----
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    if batch * img_bytes < 200e6:
        e2e_steps = max(e2e_steps, 20)  # single-image calls take well under a millisecond: average more of them
    pinned = [torch.from_numpy(f.reshape(-1)).pin_memory() for f in frames]
    ptrs = (C.c_void_p * batch)(*[pinned[k].data_ptr() for k in order])
    files_c = C.c_void_p()
    offs_c = (C.c_uint64 * (batch + 1))()
    p = enc._params(width, height, ct)
    lib = device.lib

    def e2e_step():
        # the call a user makes: host pixels in, host JPEG files out (pinned, owned by the context)
        rc = lib.jpgb_encode_batch_pinned(device.handle, C.byref(p), ptrs, img_bytes, batch, C.byref(files_c), offs_c)
        if rc != 0:
            raise SystemExit("bench.py: jpgb_encode_batch_pinned failed: %s" % device.last_error())
        return int(offs_c[batch])

    n_out = e2e_step()
    first = C.string_at(files_c.value + offs_c[check[0]], offs_c[check[0] + 1] - offs_c[check[0]])
    if first != oracle_encode(frames[order[check[0]]], width, height, color, cfg):
        raise SystemExit("bench.py: host-batch bytes differ from the oracle")
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(e2e_steps):
        d2h = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev_t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = mp_per_step * e2e_steps / e2e_s

    # what the link alone can do: the same pinned frames copied to the device back to back, nothing else running
    # (explains the end-to-end number: it moves bpp bytes per pixel over PCIe)
    stage_d = torch.empty(min(batch, 64) * img_bytes, dtype=torch.uint8, device=dev_t)
    n_copy = min(batch, 256)

    def copy_all():
        for i in range(n_copy):
            k = i % min(batch, 64)
            stage_d[k * img_bytes:(k + 1) * img_bytes].copy_(pinned[order[i]], non_blocking=True)

    copy_all()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    copy_all()
    torch.cuda.synchronize()
    h2d_gbs = n_copy * img_bytes / (time.perf_counter() - t0) / 1e9
    del stage_d

    # the crate's own call shape: Encoder::encode(&[u8]) -> one image per call, PAGEABLE input (a plain Vec<u8>),
    # bytes handed to the sink. Measured beside the pinned batch figure (rank 0 reports its own rate).
    sink_bytes = [0]

    @C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)
    def sink_cb(_user, _buf, ln):  # a JfifWrite that only counts: the library hands over its pinned download buffer
        sink_bytes[0] = ln
        return 0

    def drop_in_rate(src_frames, n_calls):
        views = [np.ascontiguousarray(f).reshape(-1) for f in src_frames]

        def call(v):
            rc = lib.jpgb_encode_to_sink(device.handle, C.byref(p), v.ctypes.data, v.size, C.cast(sink_cb, C.c_void_p), None)
            if rc != 0:
                raise SystemExit("bench.py: jpgb_encode_to_sink failed: %s" % device.last_error())

        call(views[0])
        t0_ = time.perf_counter()
        for i in range(n_calls):
            call(views[i % len(views)])
        return n_calls * width * height / 1e6 / (time.perf_counter() - t0_)

    n_calls = 24 if img_bytes < 64e6 else 3
    drop_pageable = drop_in_rate(frames, n_calls)
    drop_pinned = drop_in_rate([t_.numpy() for t_ in pinned], n_calls)
    if enc.encode(frames[0], width, height, ct) != want[0]:
        raise SystemExit("bench.py: jpgb_encode bytes differ from the oracle")

    # ---- BASELINE config 5 inside the default line: one 16384^2 progressive image cut into restart-aligned strips,
    # one strip per GPU, pieces gathered to rank 0 (the only path with a data collective), parity-gated ----
    c5 = None
    if args.workload == "c3" and not args.no_c5:
        del d_in, d_distinct
        device.close()
        torch.cuda.empty_cache()
        c5_args = argparse.Namespace(**vars(args))
        c5_args.workload, c5_args.size, c5_args.skip_parity = "c5", args.c5_size, False
        c5_line = run_strips(c5_args, rank, world, local, dev_t, extra=True, dump_name="c5_file")
        if rank == 0:
            c5 = {k: c5_line[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "scaling", "gpu_launches", "stage_ms_per_step", "gather_ms_per_step")}
            c5.update(parity=True, workload=c5_line["config"]["workload"], strips=c5_line["config"]["strips"], bytes_out=c5_line["config"]["bytes_out"],
                      collective=c5_line["config"]["collective"], e2e=c5_line["e2e"], stage_a_frac_of_hbm_peak=c5_line["roofline"]["frac"])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (colour + DCT + quant) ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    a_bytes = stage_a_bytes(width, height, color, cfg) * batch
    a_ms = stage_ms.get("colour_dct_quant", 0.0) / args.steps
    achieved = a_bytes / (a_ms * 1e-3) / 1e9 if a_ms > 0 else None
    roofline = {"bound": "hbm", "kernel": "stage_a_warp_kernel (colour+decimate+fDCT+quant)", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": a_bytes, "ms_per_launch": a_ms,
                "share_of_step": a_ms / ms_per_step if ms_per_step else None}
    traffic_path = os.path.join(ROOT, "profiles", "stage_a_traffic.json")
    if os.path.exists(traffic_path):
        try:
            tr = json.load(open(traffic_path))
            if tr.get("workload") == args.workload:  # ncu --set full capture of the same kernel, per frame x frames per launch
                roofline["traffic"] = tr["dram_bytes_per_frame"] * batch
                roofline["traffic_source"] = tr.get("source")
        except (ValueError, OSError):
            pass

    # ---- CPU baseline on a bounded sample of the same workload ----
    cpu = None
    if not args.no_cpu and world == 1:  # rank 0 at N=1 only
        cores = usable_cores()
        v1, n1 = cpu_encode_rate(frames, width, height, color, cfg, args.cpu_seconds / 3.0, 1)
        vN, nN = cpu_encode_rate(frames, width, height, color, cfg, args.cpu_seconds, cores)
        cpu = {"value": vN, "unit": "megapixels/s", "cores": cores, "kind": "port",
               "sample": "%d encodes of the workload's frames, one encode per thread on %d threads (%.0f s); single thread: %d encodes"
                         % (nN, cores, args.cpu_seconds, n1),
               "single_thread_value": v1,
               "note": "C restatement of jpeg-encoder 0.7.0 (oracle/), gcc -O3 -march=native, AVX2 colour conversion and fDCT like the crate's simd feature "
                       "(quantizer and entropy coder scalar, as in the crate); the Rust crate cannot be built in this image"}

    line = {
        "metric": "megapixels/sec encoded, byte-identical to the reference restatement",
        "value": value, "unit": "megapixels/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8 in / i32 arithmetic / i16 coefficients", "data": "synthetic",
        "config": {"workload": desc, "workload_id": args.workload, "frames_total": total_frames, "frames_per_gpu": batch,
                   "sharding": "fixed batch of %d frames, rank r encodes frames shard_batch(total, N, r): no data-path collective" % total_frames,
                   "width": width, "height": height,
                   "settings": {k: (v if k != "qtables" else "custom u16[64] x2") for k, v in cfg.items()},
                   "distinct_frames": n_distinct, "bytes_out_per_step_per_gpu": out_bytes_per_step,
                   "l2": "inputs (%.1f MB per step per GPU) larger than L2, no flush" % (batch * img_bytes / 1e6)
                   if batch * img_bytes > 200e6 else "inputs smaller than L2 (%.1f MB): single-image latency case" % (batch * img_bytes / 1e6)},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "megapixels/s", "h2d_bytes_per_step": total_frames * img_bytes,
                "d2h_bytes_per_step": int(d2h) * world, "steps": e2e_steps, "api": "jpgb_encode_batch_pinned (pinned host pixels -> host JPEG files; chunked upload/encode/download overlap)",
                "host_placement": numa, "h2d_link_gbs_measured": h2d_gbs, "h2d_gbs_in_e2e": batch * img_bytes * e2e_steps / e2e_s / 1e9,
                "frac_of_link": (batch * img_bytes * e2e_steps / e2e_s / 1e9) / h2d_gbs,
                "note": "end to end is bound by the host->device link (bpp bytes per pixel over PCIe): frac_of_link = h2d_gbs_in_e2e / h2d_link_gbs_measured (rank 0)",
                "drop_in_call": {"api": "jpgb_encode_to_sink: one image per call, what Encoder::encode(&[u8]) binds (sink = the crate's JfifWrite::write_all)", "calls": n_calls, "unit": "megapixels/s",
                                 "pageable_input": drop_pageable, "pinned_input": drop_pinned,
                                 "note": "rank 0's own rate; pageable input is staged through the context's two pinned buffers (4 copy threads); one large image is uploaded in slices with the colour+DCT kernel running behind the link"}},
        "gpu_launches": launches,
        "stage_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    if weak:
        line["weak"] = weak
    if rank_ms_value:
        line["rank_ms_per_step"] = [round(x, 4) for x in rank_ms_value]
    if c5:
        line["c5"] = c5
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---- one very large image, strips across the GPUs (BASELINE config 5) ---------------------------
def run_strips(args, rank, world, local, dev_t, extra=False, dump_name="file"):
    import torch
    import torch.distributed as dist
    import images
    import jpeg_encoder_b200 as je
    from cases import CT, make_encoder, oracle_encode
    from jpeg_encoder_b200 import sharding

    width, height, color, cfg, _, desc = WORKLOADS[args.workload]
    if args.size:
        width = height = args.size
    ct = CT[color][1]
    bpp = BPP[color]
    stream = torch.cuda.Stream(device=dev_t)
    torch.cuda.set_stream(stream)
    device = je.Device(local, cuda_stream=stream.cuda_stream)
    enc = make_encoder(cfg, device)
    strips = enc.plan_strips(width, height, ct, world)
    if len(strips) != world:
        raise SystemExit("bench.py: image cannot be cut into %d restart-aligned strips (got %d)" % (world, len(strips)))
    r0, rows = strips[rank]
    seed = 7
    d_strip = images.synth_frame_torch(width, height, bpp, seed=seed, row0=r0, rows=rows, device=dev_t).reshape(-1)
    torch.cuda.synchronize()

    optimized = bool(cfg.get("optimize_huffman"))

    def encode_strip(d_ptr):
        hist_total = None
        if optimized:  # tables describe the whole image: all-reduce the strips' symbol histograms first
            hist, edge = enc.strip_histogram_device(d_ptr, rank, world, r0, rows, width, height, ct)
            if world > 1:
                hist, edge = sharding.exchange_strip_histograms(hist, edge, dev_t)
            hist_total = enc.merge_strip_histograms(hist, edge, width, height, ct)
        return enc.encode_strip_device(d_ptr, rank, world, r0, rows, width, height, ct, hist_total=hist_total)

    def encode_once():
        return encode_strip(d_strip.data_ptr())

    gather_events = []
    # the assembled file is at most the raw strip sizes; rank 0 owns the target, the other ranks map it over NVLink (CUDA IPC)
    pg = sharding.PeerGather(device, max(width * height * bpp // 2, 1 << 20), rank, world, dev_t) if world > 1 else None

    def step(gather=True, timed=False):
        d_bytes, offs = encode_once()
        launches = device.last_launch_count()
        tm = device.last_timing()
        out = None
        if world > 1 and gather:
            # device-placed gather: one NCCL all-gather of the piece offsets, then every rank's kernel stores its pieces at
            # their scan-major place inside rank 0's buffer through a peer pointer; one barrier
            if timed:
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(stream)
            pg.gather()
            pg.barrier()
            launches += 1
            if timed:
                g1.record(stream)
                gather_events.append((g0, g1))
            out = pg
        elif gather:
            out = _as_tensor(d_bytes, offs[-1], dev_t)
        return out, launches, tm

    def fetch(out):
        """rank 0: the assembled file as a device tensor"""
        return out.result() if world > 1 else out

    # parity gate (un-timed): the assembled file must equal the oracle's for the whole image
    out, _, _ = step()
    torch.cuda.synchronize()
    if rank == 0:
        got = bytes(fetch(out).cpu().numpy().tobytes())
        if not args.skip_parity:
            full = torch.cat([images.synth_frame_torch(width, height, bpp, seed=seed, row0=a, rows=b, device=dev_t).cpu()
                              for a, b in strips]).numpy()
            want = oracle_encode(full, width, height, color, cfg)
            if got != want:
                raise SystemExit("bench.py: assembled strips differ from the oracle (%d vs %d bytes)" % (len(got), len(want)))
            del full
        out_bytes = len(got)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    device.set_timing(False)
    sampler = ClockSampler(local)  # started before the warm-up, see run_batch
    if rank == 0 and not extra:
        sampler.start()
        time.sleep(0.3)
    for _ in range(args.warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    e0.record(stream)
    for _ in range(args.steps):
        out, l, _ = step(timed=True)
        launches += l
    e1.record(stream)
    barrier()
    if args.dump_outputs and rank == 0:  # the last timed step's file, before the next step overwrites it
        f = fetch(out)
        dump_outputs(args.dump_outputs, dump_name, f, [0, f.numel()], DUMP_BUDGET // 2 if extra else DUMP_BUDGET)
    # second pass with the library's per-stage events (kernel-by-kernel launches instead of the graph replay): breakdown only
    device.set_timing(True)
    stage_ms = {}
    for _ in range(args.steps):
        _, _, tm = step()
        for k, v in (tm or {}).items():
            stage_ms[k] = stage_ms.get(k, 0.0) + v
    device.set_timing(False)
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev_t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    gather_ms = sum(a.elapsed_time(b) for a, b in gather_events) / args.steps if gather_events else 0.0
    if world > 1:  # the slowest rank's gather (rank 0 receives, the others send)
        t = torch.tensor([gather_ms], device=dev_t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gather_ms = float(t.item())
    # keep the same work running (un-timed, same count on every rank) for about a second so that the
    # 50 ms clock samples are taken under this load
    if not extra:
        for _ in range(int(min(400, 1000.0 / max(ms_per_step, 1.0)))):
            step()
        barrier()
    clocks = sampler.stop() if (rank == 0 and not extra) else None
    mp = width * height / 1e6
    value = mp / (ms_per_step / 1e3)

    # end to end: pinned host strip -> device -> encode -> gather -> host file on rank 0
    h_strip = d_strip.cpu().pin_memory()
    d_stage = torch.empty_like(d_strip)
    h_file = torch.empty(max(width * height * bpp // 2, 1 << 20), dtype=torch.uint8).pin_memory() if rank == 0 else None
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(e2e_steps):
        d_stage.copy_(h_strip, non_blocking=True)
        d_bytes, offs = encode_strip(d_stage.data_ptr())
        if world > 1:
            pg.gather()
            pg.barrier()
            o = pg.result() if rank == 0 else None
        else:
            o = _as_tensor(d_bytes, offs[-1], dev_t)
        if rank == 0:
            d2h = o.numel()
            h_file[:d2h].copy_(o, non_blocking=True)  # the file lands in pinned host memory
        torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev_t)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    if pg:  # the peers unmap rank 0's buffer before rank 0 frees it
        torch.cuda.synchronize()
        if rank != 0:
            pg.close()
        dist.barrier()
        if rank == 0:
            pg.close()
    if rank != 0:
        if world > 1 and not extra:
            dist.destroy_process_group()
        return None
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = (float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)") if os.path.exists(peaks_path) \
        else (6650.0, "fallback (B200_PROFILING.md)")
    lay = enc.coef_layout(width, rows, ct)
    a_bytes = width * rows * bpp + 128 * int(lay.blocks_per_image)
    a_ms = stage_ms.get("colour_dct_quant", 0.0) / args.steps
    achieved = a_bytes / (a_ms * 1e-3) / 1e9 if a_ms > 0 else None
    line = {
        "metric": "megapixels/sec encoded, byte-identical to the reference restatement",
        "value": value, "unit": "megapixels/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8 in / i32 arithmetic / i16 coefficients", "data": "synthetic",
        "config": {"workload": desc, "workload_id": args.workload, "width": width, "height": height,
                   "strips": [[int(a), int(b)] for a, b in strips], "settings": cfg, "bytes_out": out_bytes,
                   "l2": "strip input %.0f MB per GPU, larger than L2" % (width * rows * bpp / 1e6),
                   "collective": ("all-reduce of the 4 x 257 symbol histogram + all_gather of edge DCs, then " if optimized else "")
                   + ("one NCCL all-gather of the piece offsets (device tensors), then every rank's kernel stores its pieces at their "
                      "scan-major place in rank 0's buffer through a CUDA-IPC peer pointer over NVLink, one barrier" if world > 1 else "none at N = 1")},
        "clocks": clocks,
        "e2e": {"value": mp * e2e_steps / e2e_s, "unit": "megapixels/s", "h2d_bytes_per_step": width * height * bpp,
                "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                "api": "pinned host strip -> jpgb_encode_strip_device -> device-placed gather -> host file on rank 0"},
        "gpu_launches": launches,
        "stage_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
        "gather_ms_per_step": gather_ms,
        "roofline": {"bound": "hbm", "kernel": "stage_a_warp_kernel (colour+decimate+fDCT+quant), rank 0's strip", "achieved": achieved,
                     "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": None,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": a_bytes, "ms_per_launch": a_ms},
        "cpu_baseline": None,
    }
    if extra:
        return line
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def _as_tensor(d_ptr, nbytes, dev_t):
    """Zero-copy torch view of context-owned device memory (valid until the next call on the context)."""
    import torch

    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(d_ptr), False), "version": 3}
    return torch.as_tensor(h, device=dev_t)


# ---- the reference arm: the CPU restatement on the host cores -------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    width, height, color, cfg, def_batch, desc = WORKLOADS[args.workload]
    cfg = resolve_cfg(cfg)
    n_distinct = min(DISTINCT, args.batch or def_batch)
    frames = frames_for(width, height, color, n_distinct)
    cores = usable_cores()
    per_step = max(1.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        cpu_encode_rate(frames, width, height, color, cfg, min(per_step, 2.0), cores)
    t0 = time.perf_counter()
    mp = 0.0
    n_enc = 0
    for _ in range(args.steps):
        v, n = cpu_encode_rate(frames, width, height, color, cfg, per_step, cores)
        n_enc += n
        mp += n * width * height / 1e6
    dt = time.perf_counter() - t0
    value = mp / dt
    sample = "%d encodes of the workload's frames per run, one encode per thread on %d threads, %.1f s per step" % (n_enc, cores, per_step)
    line = {
        "impl": "reference", "metric": "megapixels/sec encoded, byte-identical to the reference restatement",
        "value": value, "unit": "megapixels/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 in / i32 arithmetic / i16 coefficients", "data": "synthetic",
        "config": {"workload": desc, "workload_id": args.workload, "width": width, "height": height,
                   "settings": {k: (v if k != "qtables" else "custom u16[64] x2") for k, v in cfg.items()}},
        "cpu_baseline": {"value": value, "unit": "megapixels/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "C restatement of jpeg-encoder 0.7.0 (oracle/), gcc -O3 -march=native, AVX2 colour conversion and fDCT like the crate's simd feature "
                                 "(quantizer and entropy coder scalar, as in the crate); no Rust toolchain in the image"},
        "e2e": {"value": value, "unit": "megapixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU (default: the workload's)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--size", type=int, default=0, help="c5 only: square image size override (testing)")
    ap.add_argument("--c5-size", type=int, default=0, help="size override of the config-5 leg inside the default line (testing)")
    ap.add_argument("--no-c5", action="store_true", help="default workload only: skip the config-5 (strips + gather) leg")
    ap.add_argument("--no-weak", action="store_true", help="default workload only: skip the weak-scaling leg at N > 1")
    ap.add_argument("--skip-parity", action="store_true", help="c5 only: skip the whole-image oracle comparison")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed step as .npy files "
                    "(JPEG bytes as float32, a fixed sample of long streams; offsets as float64) for comparing builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
