"""Strided device input against the packed entry, for the C3 batch (1024 x 1920x1080 RGB, q90 4:2:0; the inputs are
far larger than L2):

    (a) packed contiguous (jpgb_encode_batch_device)
    (b) NHWC rows in a 5,888-byte pitch
    (c) NCHW planar
    (d) a crop at x0 = 1 of a wider NHWC tensor (unaligned base: cp.async staging)
    (e) the alternative without strided input: .contiguous() of (b) / permute(0, 2, 3, 1).contiguous() of (c), then (a)

Per layout: stage A ms (per-stage events, set_timing) and its fraction of 6,541 GB/s for stage A's algorithmic bytes
(w*h*bpp + 128 B per block, bench.stage_a_bytes), and the whole call in ms (CUDA events on the context's stream around
the copy, if any, and the encode). The layouts are alternated round by round.

    python tools/strided_stage_time.py [rounds] [n]          (GPU box)
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import images  # noqa: E402
import jpeg_encoder_b200 as je  # noqa: E402
from cases import make_encoder, oracle_encode  # noqa: E402

PEAK_GBS = 6541.1  # measured HBM peak of the B200 (DESIGN.md section 4)


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 1024
    w, h, pitch, distinct = 1920, 1080, 5888, 8
    cfg = dict(quality=90, sampling=(2, 2))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print("GPU: %s | %s" % (torch.cuda.get_device_name(0), q.stdout.strip()), flush=True)

    frames = [images.synth_frame_torch(w, h, 3, seed=s) for s in range(distinct)]
    order = [i % distinct for i in range(n)]
    want = [oracle_encode(images.synth_frame(w, h, 3, seed=s), w, h, "rgb", cfg) for s in range(distinct)]
    packed = torch.stack([frames[k] for k in order])                          # (n, h, w, 3)
    pitched = torch.empty(n, h, pitch, dtype=torch.uint8, device="cuda")      # (b): NHWC in a pitch
    pitched[:, :, :w * 3].copy_(packed.view(n, h, w * 3))
    nhwc_pitched = torch.as_strided(pitched, (n, h, w, 3), (h * pitch, pitch, 3, 1))
    nchw = packed.permute(0, 3, 1, 2).contiguous()                            # (c)
    wide = torch.empty(n, h, w + 16, 3, dtype=torch.uint8, device="cuda")     # (d)
    wide[:, :, 1:1 + w].copy_(packed)
    crop = wide[:, :, 1:1 + w]
    torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    dev = je.Device(0, cuda_stream=stream.cuda_stream)
    enc = make_encoder(cfg, dev)
    rgb = je.ColorType.Rgb
    scratch = {}

    def contiguous_then_packed(src):
        def run():
            scratch["c"] = src().contiguous()  # on `stream`: the context's stream
            return enc.encode_batch_device(scratch["c"].data_ptr(), w * h * 3, n, w, h, rgb)
        return run

    cases = {
        "a_packed": lambda: enc.encode_batch_device(packed.data_ptr(), w * h * 3, n, w, h, rgb),
        "b_pitch5888": lambda: enc.encode_cuda_array(nhwc_pitched, rgb),
        "c_nchw": lambda: enc.encode_cuda_array(nchw, rgb, channels_first=True),
        "d_crop_x1": lambda: enc.encode_cuda_array(crop, rgb),
        "e_contig_of_b": contiguous_then_packed(lambda: nhwc_pitched),
        "e_contig_of_c": contiguous_then_packed(lambda: nchw.permute(0, 2, 3, 1)),
    }
    sa_bytes = bench.stage_a_bytes(w, h, "rgb", cfg) * n
    res = {k: {"stage_a": [], "call": []} for k in cases}
    with torch.cuda.stream(stream):
        for name, call in cases.items():  # warm-up and exactness of every layout
            for _ in range(2):
                d_files, offs = call()
            blob = dev.download(d_files, offs[-1])
            bad = [i for i in range(n) if bytes(blob[offs[i]:offs[i + 1]]) != want[order[i]]]
            assert not bad, "%s: files differ %r" % (name, bad[:8])
        for _ in range(rounds):
            for name, call in cases.items():
                dev.set_timing(True)
                call()
                res[name]["stage_a"].append(dev.last_timing()["colour_dct_quant"])
                dev.set_timing(False)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                call()
                e1.record(stream)
                e1.synchronize()
                res[name]["call"].append(e0.elapsed_time(e1))
    print("C3 batch: %d x %dx%d RGB q90 4:2:0, stage A algorithmic bytes %.3f GB, %d rounds alternated (median [min..max])" %
          (n, w, h, sa_bytes / 1e9, rounds))
    print("| layout | stage A ms | of %.0f GB/s | whole call ms |" % PEAK_GBS)
    print("|---|---|---|---|")
    for name, r in res.items():
        sa, call = np.array(r["stage_a"]), np.array(r["call"])
        frac = sa_bytes / (np.median(sa) * 1e-3) / (PEAK_GBS * 1e9)
        print("| %s | %.3f [%.3f..%.3f] | %.1f %% | %.3f [%.3f..%.3f] |" %
              (name, np.median(sa), sa.min(), sa.max(), 100 * frac, np.median(call), call.min(), call.max()), flush=True)
    a = np.median(res["a_packed"]["stage_a"])
    print("stage A ratios to (a): " + ", ".join("%s %.3f" % (k, np.median(r["stage_a"]) / a) for k, r in res.items()))
    dev.close()


if __name__ == "__main__":
    main()
