"""Time one large image in strips without restart intervals across the GPUs of a box, next to the restart-aligned path.

    torchrun --nproc_per_node N tools/contiguous_strips_time.py [--steps 20] [--warmup 5] [--size 16384] [--json out.json]

Workloads (restart interval 0): 16384^2 RGB progressive (4 scans) 4:2:0, and 16384^2 RGB q90 4:2:0 interleaved. A step on
every rank: prepare its strip (stage A), all-gather the edge DCs, code its pieces, all-gather their bit lengths, store
them at their bit positions in rank 0's buffer, barrier; then rank 0 finishes the file (leads, pad, EOI, 0xFF
stuffing). Step time and rank 0's finish time are CUDA events on rank 0's stream, median over the steps. The same run
times the restart-2048 strip path (restart-aligned pieces, device-placed gather) and the one-GPU whole-image call
(jpgb_encode_batch_device), and checks rank 0's file against that one-GPU call byte for byte.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import images  # noqa: E402
import jpeg_encoder_b200 as je  # noqa: E402
from cases import make_encoder  # noqa: E402
from jpeg_encoder_b200 import sharding  # noqa: E402

WORKLOADS = {
    "progressive_420": dict(quality=90, sampling=(2, 2), progressive_scans=4),
    "interleaved_420_q90": dict(quality=90, sampling=(2, 2)),
}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                             timeout=30).stdout.strip()
        return out
    except Exception as e:  # the numbers are still reported, without the card
        return "unknown (%s)" % e


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2] if xs else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--size", type=int, default=16384)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev_t = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev_t)
    stream = torch.cuda.Stream(device=dev_t)
    torch.cuda.set_stream(stream)
    device = je.Device(local, cuda_stream=stream.cuda_stream)
    w = h = args.size
    ct = je.ColorType.Rgb
    results = {"world": world, "card": card() if rank == 0 else None, "size": w, "workloads": {}}
    for name, cfg in WORKLOADS.items():
        enc = make_encoder(cfg, device)
        strips = enc.plan_contiguous_strips(w, h, ct, world)
        assert len(strips) == world
        r0, rows = strips[rank]
        d_strip = images.synth_frame_torch(w, h, 3, seed=7, row0=r0, rows=rows, device=dev_t).reshape(-1).contiguous()
        torch.cuda.synchronize()
        pg = sharding.PeerGather(device, w * h * 3 // 2 + (1 << 24), rank, world, dev_t)
        ev = []

        def step(timed):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record(stream)
            _, edge = enc.contiguous_strip_prepare_device(d_strip.data_ptr(), rank, world, r0, rows, w, h, ct)
            edges = sharding.exchange_edge_dc(edge, dev_t) if world > 1 else edge
            enc.encode_contiguous_strip_device(d_strip.data_ptr(), rank, world, r0, rows, w, h, ct, edges)
            pg.gather_bits(enc)
            pg.barrier()
            e1.record(stream)
            f = pg.finish_bits(enc, w, h, ct) if rank == 0 else None
            e2.record(stream)
            if timed:
                ev.append((e0, e1, e2))
            return f

        out = step(False)
        got = bytes(out.cpu().numpy().tobytes()) if rank == 0 else None
        for _ in range(args.warmup):
            step(False)
        for _ in range(args.steps):
            step(True)
        torch.cuda.synchronize()
        res = {}
        if rank == 0:
            res["step_ms"] = median([a.elapsed_time(c) for a, _, c in ev])
            res["root_finish_ms"] = median([b.elapsed_time(c) for _, b, c in ev])
            res["file_bytes"] = len(got)
        pg.close()

        # the restart-aligned path, restart 2048, in the same run
        cfg_r = dict(cfg, restart_interval=2048)
        enc_r = make_encoder(cfg_r, device)
        strips_r = enc_r.plan_strips(w, h, ct, world)
        if len(strips_r) == world and strips_r[rank] == (r0, rows):
            pg_r = sharding.PeerGather(device, w * h * 3 // 2 + (1 << 24), rank, world, dev_t)
            ev_r = []
            for i in range(args.warmup + args.steps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                enc_r.encode_strip_device(d_strip.data_ptr(), rank, world, r0, rows, w, h, ct)
                if world > 1:
                    pg_r.gather()
                    pg_r.barrier()
                b.record(stream)
                if i >= args.warmup:
                    ev_r.append((a, b))
            torch.cuda.synchronize()
            if rank == 0:
                res["restart2048_step_ms"] = median([a.elapsed_time(b) for a, b in ev_r])
            pg_r.close()

        # the one-GPU whole-image call: the reference time and the parity check
        if world > 1:
            dist.barrier()
        if rank == 0:
            full = torch.cat([images.synth_frame_torch(w, h, 3, seed=7, row0=a, rows=b, device=dev_t) for a, b in strips]).reshape(-1).contiguous()
            torch.cuda.synchronize()
            ev1 = []
            for i in range(args.warmup + args.steps + 1):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                d_files, offs = enc.encode_batch_device(full.data_ptr(), full.numel(), 1, w, h, ct)
                b.record(stream)
                if i == 0:
                    res["parity_with_one_gpu"] = device.download(d_files, offs[1]) == got
                elif i > args.warmup:
                    ev1.append((a, b))
            torch.cuda.synchronize()
            res["one_gpu_whole_image_ms"] = median([a.elapsed_time(b) for a, b in ev1])
            del full
            torch.cuda.empty_cache()
        if world > 1:
            dist.barrier()
        results["workloads"][name] = res
    if rank == 0:
        line = json.dumps(results)
        print(line)
        if args.json:
            with open(args.json, "w") as f:
                f.write(line + "\n")
    device.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
