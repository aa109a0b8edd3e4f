"""Time subsampled YCbCr frames read from their planes against the full-resolution planar path, at C3 geometry
(1024 x 1920x1080 frames, q90 4:2:0 baseline).

  (a) I420 (three planes) and NV12 (luma + interleaved Cb/Cr) through Encoder.encode_cuda_ycbcr; and NV12's Cb and Cr
      each in a copy of the interleaved plane of its own (nv12_split), which takes one launch per channel, each staging
      the whole pair plane: what NV12 costs when Cb and Cr do not share a launch;
  (b) the same frames upsampled to full-resolution (N, 3, H, W) planes beforehand, encoded through the strided planar
      Ycbcr call (Encoder.encode_cuda_array with channels_first): what stage A reads when the caller upsamples;
  (c) the torch upsample (repeat_interleave into the planar tensor) followed by (b), end to end: what a user does
      without the frame entry;
  (d) one 8192 x 8192 I420 frame to 4:2:0 and to 4:4:4 (F_1_1, each plane sample feeding two block samples).
Calls are timed with device events, stage 0 (the colour+DCT launches) with the context's own events; medians over
warm steps. The batch is several GB, far beyond the 126 MB L2. Stage A's algorithmic bytes are the samples a frame
holds (w*h*1.5 at 4:2:0, w*h*3 at full resolution) plus 128 bytes per coded block; its rate is given as a share of
7.7 TB/s (the HBM3e bandwidth of one B200). Fails without a GPU.

    python tools/ycbcr_frames_time.py [--n 1024] [--iters 7] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

PEAK_BPS = 7.7e12


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # the name still comes from torch below
        return "nvidia-smi unavailable (%s)" % e


def blocks_420(w, h):
    """coded blocks of one frame at 4:2:0 in MCU order (the padded grids the interleaved scan stores)"""
    mx, my = -(-w // 16), -(-h // 16)
    return mx * my * 6


def blocks_444(w, h):
    return 3 * (-(-w // 8)) * (-(-h // 8))


def timed(fn, dev, iters):
    import torch
    fn()
    torch.cuda.synchronize()
    ms, st0 = [], []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
        st0.append(dev.last_timing()["colour_dct_quant"])
    return float(np.median(ms)), float(np.median(st0))


def main():
    import torch
    import images
    import jpeg_encoder_b200 as je
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=7)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    w, h, n = 1920, 1080, a.n
    info = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": gpu_info(), "n": n, "width": w, "height": h}
    print(json.dumps(info), flush=True)
    dev = je.Device(0)
    dev.set_timing(True)
    enc = je.Encoder(90, device=dev)
    enc.set_sampling_factor(je.SamplingFactor.from_factors(2, 2))

    distinct = 8
    full = torch.stack([torch.from_numpy(images.synth_frame(w, h, 3, seed=s)) for s in range(distinct)]).cuda()  # (8, H, W, 3)
    idx = torch.arange(n, device="cuda") % distinct
    y = full[..., 0][idx].contiguous()
    cb = full[:, ::2, ::2, 1][idx].contiguous()
    cr = full[:, ::2, ::2, 2][idx].contiguous()
    nv12 = torch.cat([y, torch.stack([cb, cr], -1).reshape(n, h // 2, w)], 1).contiguous()  # (N, H * 3 // 2, W)
    uv = nv12[:, h:].view(n, h // 2, w // 2, 2)
    uv_cb, uv_cr = uv.clone(), uv.clone()  # Cb read from one copy, Cr from the other: no shared pairs
    planar = torch.empty((n, 3, h, w), dtype=torch.uint8, device="cuda")

    def upsample():
        planar[:, 0].copy_(y)
        planar[:, 1].copy_(cb.repeat_interleave(2, 1).repeat_interleave(2, 2)[:, :h, :w])
        planar[:, 2].copy_(cr.repeat_interleave(2, 1).repeat_interleave(2, 2)[:, :h, :w])

    upsample()
    torch.cuda.synchronize()
    out = {}

    def files_of(call):
        d, offs = call()
        return dev.download(d, offs[-1])

    # the four inputs give the same files
    same = files_of(lambda: enc.encode_cuda_ycbcr(y, cb, cr)) == files_of(lambda: enc.encode_cuda_ycbcr(nv12[:, :h], uv[..., 0], uv[..., 1])) \
        == files_of(lambda: enc.encode_cuda_ycbcr(nv12[:, :h], uv_cb[..., 0], uv_cr[..., 1])) \
        == files_of(lambda: enc.encode_cuda_array(planar, je.ColorType.Ycbcr, channels_first=True))
    info["files_identical"] = bool(same)
    cases = {
        "i420": lambda: enc.encode_cuda_ycbcr(y, cb, cr),
        "nv12": lambda: enc.encode_cuda_ycbcr(nv12[:, :h], uv[..., 0], uv[..., 1]),
        "nv12_split": lambda: enc.encode_cuda_ycbcr(nv12[:, :h], uv_cb[..., 0], uv_cr[..., 1]),
        "full_res_planar": lambda: enc.encode_cuda_array(planar, je.ColorType.Ycbcr, channels_first=True),
        "torch_upsample_then_planar": lambda: (upsample(), enc.encode_cuda_array(planar, je.ColorType.Ycbcr, channels_first=True)),
    }
    blk = n * blocks_420(w, h) * 128
    for name, fn in cases.items():
        ms, st0 = timed(fn, dev, a.iters)
        src = n * w * h * (3 if name == "full_res_planar" else 1.5)
        r = {"case": name, "call_ms": ms, "stage0_ms": st0, "stage_a_bytes": src + blk,
             "stage_a_share_of_7.7TBps": (src + blk) / (st0 * 1e-3) / PEAK_BPS}
        if name == "torch_upsample_then_planar":
            del r["stage_a_bytes"], r["stage_a_share_of_7.7TBps"]
        print(json.dumps(r), flush=True)
        out[name] = r
    del y, cb, cr, nv12, uv, uv_cb, uv_cr, planar, full
    torch.cuda.empty_cache()

    # one large frame: 4:2:0 (step-1 plane reads) and 4:4:4 (half-sample steps)
    W = 8192
    big = torch.from_numpy(images.synth_frame(W, W, 3, seed=9)).cuda()
    by, bcb, bcr = big[..., 0].contiguous(), big[::2, ::2, 1].contiguous(), big[::2, ::2, 2].contiguous()
    for samp, nblk in (((2, 2), blocks_420(W, W)), ((1, 1), blocks_444(W, W))):
        e = je.Encoder(95 if samp == (1, 1) else 90, device=dev)
        e.set_sampling_factor(je.SamplingFactor.from_factors(*samp))
        ms, st0 = timed(lambda: e.encode_cuda_ycbcr(by, bcb, bcr), dev, a.iters)
        src, wr = W * W * 1.5, nblk * 128
        r = {"case": "8192_i420_to_%d%d" % samp, "call_ms": ms, "stage0_ms": st0, "stage_a_bytes": src + wr,
             "stage_a_share_of_7.7TBps": (src + wr) / (st0 * 1e-3) / PEAK_BPS}
        print(json.dumps(r), flush=True)
        out[r["case"]] = r
    dev.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"info": info, "rows": out}, f, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
