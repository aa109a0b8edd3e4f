"""Time the fused sample-type path against converting first, at C3 geometry (1024 x 1920x1080 RGB, q90 4:2:0).

For each sample type (float32, float16, bfloat16, uint16) and layout (NHWC, NCHW):
  (a) fused: Encoder.encode_cuda_samples, stage A converting while it stages;
  (b) two-step: torch's x.float() * scale + offset, rounded, clamped and cast to uint8 (the multiply and add as two
      ops), then Encoder.encode_cuda_array on the uint8 tensor in the same layout.
Both are timed with device events around whole calls. Stage 0 (colour+DCT, the stage A launch) comes from the
context's own events. Stage A's algorithmic bytes are the input read plus the int16 coefficients written; its rate is
given as a share of 7.7 TB/s (the HBM3e bandwidth of one B200). The pixels are photo-like frames scaled into the
value range. Fails without a GPU.

    python tools/sample_types_time.py [--n 1024] [--iters 5] [--out results.json]
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
TYPES = {"f32": ("float32", (0.0, 1.0)), "f16": ("float16", (0.0, 1.0)), "bf16": ("bfloat16", (-1.0, 1.0)), "u16": ("uint16", (0.0, 65535.0))}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:  # the name still comes from torch below
        return "nvidia-smi unavailable (%s)" % e


def main():
    import torch
    import images
    import jpeg_encoder_b200 as je
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    w, h, n = 1920, 1080, a.n
    info = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": gpu_info(), "n": n, "width": w, "height": h}
    print(json.dumps(info))
    dev = je.Device(0)
    dev.set_timing(True)
    enc = je.Encoder(90, device=dev)
    enc.set_sampling_factor(je.SamplingFactor.from_factors(2, 2))
    distinct = 8
    base = torch.stack([torch.from_numpy(images.synth_frame(w, h, 3, seed=s)) for s in range(distinct)]).cuda()
    idx = torch.arange(n, device="cuda") % distinct
    coef_bytes = n * (w * h + 2 * (w // 2) * (h // 2)) * 2  # int16 coefficients of Y + Cb + Cr at 4:2:0
    rows = []
    for st, (dtype, (lo, hi)) in TYPES.items():
        scale, offset = je.sample_scale_offset(je.SampleType[st.upper()], (lo, hi))
        for layout in ("nhwc", "nchw"):
            cf = layout == "nchw"
            u = base.permute(0, 3, 1, 2) if cf else base
            x = (u.float() * ((hi - lo) / 255.0) + lo)[idx]
            x = (x.round() if st == "u16" else x).to(getattr(torch, dtype)).contiguous()
            torch.cuda.synchronize()

            def fused():
                enc.encode_cuda_samples(x, je.ColorType.Rgb, channels_first=cf, value_range=(lo, hi))

            def two_step():
                y = torch.mul(x.float(), scale)
                y = torch.add(y, offset)
                u8 = y.round_().clamp_(0, 255).to(torch.uint8)
                enc.encode_cuda_array(u8, je.ColorType.Rgb, channels_first=cf)

            res = {"type": st, "layout": layout}
            for name, fn in (("fused", fused), ("two_step", two_step)):
                fn()
                torch.cuda.synchronize()
                ms, st0 = [], []
                for _ in range(a.iters):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn()
                    e1.record()
                    torch.cuda.synchronize()
                    ms.append(e0.elapsed_time(e1))
                    st0.append(dev.last_timing()["colour_dct_quant"])
                res[name + "_call_ms"] = float(np.median(ms))
                res[name + "_stage0_ms"] = float(np.median(st0))
            in_bytes = x.numel() * x.element_size()
            res["stage_a_bytes"] = in_bytes + coef_bytes
            res["fused_stage_a_share_of_7.7TBps"] = (in_bytes + coef_bytes) / (res["fused_stage0_ms"] * 1e-3) / PEAK_BPS
            res["u8_stage_a_share_of_7.7TBps"] = (n * w * h * 3 + coef_bytes) / (res["two_step_stage0_ms"] * 1e-3) / PEAK_BPS
            res["fused_faster"] = res["fused_call_ms"] < res["two_step_call_ms"]
            print(json.dumps(res))
            rows.append(res)
            del x
            torch.cuda.empty_cache()
    dev.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"info": info, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
