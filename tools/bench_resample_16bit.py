"""resample2d family: fp32 planar NCHW (the reference's layout) against bf16 channels_last, fwd+bwd, on seeded inputs.

    python tools/bench_resample_16bit.py [--out FILE.json] [--steps N]

Workloads:
  f4_relu3_1 / f4_relu2_1   Resample2dCosine(4, 1, sigma=2) fwd + bwd with the gradient to the flow only, at the two
                            PerceptualCorrectness shapes bench.py's f4 key uses (16x256x64^2, 16x128x128^2), blocky
                            (nearest-upsampled) flow
  cfg3_ks4                  Resample2d(4, 1, sigma=2) fwd + bwd (both gradients), B=32 C=128 512x512, smooth flow
Per arm: milliseconds per fwd+bwd (CUDA events over --steps calls after warm-up), the algorithmic bytes (each input read
once, each output written once, at the arm's storage width) and the share of the 7.7 TB/s HBM roofline they give.  The
two arms' outputs are compared at the timed sizes.  Prints and writes one JSON object.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_BPS = 7.7e12


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the number still stands with the card name
        q = f"unavailable ({e})"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def timed(fn, steps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def rel_diff(a, b):
    a, b = a.float(), b.float()
    return (a - b).abs().max().item() / max(1e-30, b.abs().max().item())


def blocky_flow(B, H, W, g):
    return torch.nn.functional.interpolate(torch.randn(B, 2, H // 8, W // 8, generator=g) * 3, size=(H, W))


def smooth_flow(B, H, W, g):
    ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
    f = torch.stack([2.5 * torch.sin(ys / 23.0 + xs / 31.0), 1.7 * torch.cos(xs / 29.0 - ys / 17.0)])
    return f.unsqueeze(0).repeat(B, 1, 1, 1) + 0.1 * torch.randn(B, 2, H, W, generator=g)


def f4(F_, B, C, H, W, steps, dev):
    g = torch.Generator().manual_seed(C * 7 + H)
    in2 = torch.cat([blocky_flow(B, H, W, g), torch.full((B, 1, H, W), 2.0)], 1).to(dev)
    x32 = torch.randn(B, C, H, W, generator=g).to(dev)
    t32 = torch.randn(B, C, H, W, generator=g).to(dev)
    gcos = torch.randn(B, H, W, generator=g).to(dev)
    cl = torch.channels_last
    x16, t16 = x32.bfloat16().contiguous(memory_format=cl), t32.bfloat16().contiguous(memory_format=cl)
    res, outs = {}, {}
    for arm, x, t, es in (("fp32_nchw", x32, t32, 4), ("bf16_channels_last", x16, t16, 2)):
        def step():
            cos, stats = F_.resample2d_cosine_fwd(x, in2, t, 4, 1, 1e-8)
            _, g2, _ = F_.resample2d_cosine_bwd(x, in2, t, stats, gcos, 4, 1, 1e-8)
            return cos, g2
        ms = timed(step, steps)
        outs[arm] = step()
        px = B * H * W
        # fwd: in1, target, in2 read; cos + stats written.  bwd: in1, target, in2, stats, grad_cos read; grad_in2 written
        nbytes = 2 * (2 * px * C * es + 12 * px) + 16 * px + (12 + 4) * px + 12 * px
        res[arm] = {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "hbm_roofline_fraction": round(nbytes / HBM_BPS / (ms * 1e-3), 4)}
    res["speedup_fp32_over_bf16"] = round(res["fp32_nchw"]["ms"] / res["bf16_channels_last"]["ms"], 3)
    res["max_rel_diff_bf16_vs_fp32"] = {"cos": rel_diff(outs["bf16_channels_last"][0], outs["fp32_nchw"][0]),
                                        "grad_flow": rel_diff(outs["bf16_channels_last"][1], outs["fp32_nchw"][1])}
    res["shape"] = f"B={B} C={C} {H}x{W}, ks 4 dilation 1 sigma 2, blocky flow, gradient to the flow only"
    return res


def cfg3(F_, steps, dev):
    B, C, H, W = 32, 128, 512, 512
    g = torch.Generator().manual_seed(3)
    in2 = torch.cat([smooth_flow(B, H, W, g), torch.full((B, 1, H, W), 2.0)], 1).to(dev)
    gd = torch.Generator(device=dev).manual_seed(3)                  # 4.3 GB tensors: drawn on the device
    x32 = torch.randn(B, C, H, W, generator=gd, device=dev)
    go32 = torch.randn(B, C, H, W, generator=gd, device=dev)
    cl = torch.channels_last
    x16, go16 = x32.bfloat16().contiguous(memory_format=cl), go32.bfloat16().contiguous(memory_format=cl)
    res, outs = {}, {}
    for arm, x, go, es in (("fp32_nchw", x32, go32, 4), ("bf16_channels_last", x16, go16, 2)):
        def step():
            out = F_.resample2d_fwd(x, in2, 4, 1)
            g1, g2 = F_.resample2d_bwd(x, in2, go, 4, 1)
            return out, g1, g2
        ms = timed(step, steps, warm=2)
        outs[arm] = step()
        px, el = B * H * W, B * C * H * W
        # fwd: in1 + in2 read, out written.  bwd: in1, grad_out, in2 read; grad_in1 (arm's storage) + grad_in2 written
        nbytes = (2 * el * es + 12 * px) + (3 * el * es + 24 * px)
        res[arm] = {"ms": round(ms, 3), "algorithmic_bytes": nbytes, "hbm_roofline_fraction": round(nbytes / HBM_BPS / (ms * 1e-3), 4)}
    res["speedup_fp32_over_bf16"] = round(res["fp32_nchw"]["ms"] / res["bf16_channels_last"]["ms"], 3)
    names = ("out", "grad_input1", "grad_flow_sigma")
    res["max_rel_diff_bf16_vs_fp32"] = {n: rel_diff(a, b) for n, a, b in zip(names, outs["bf16_channels_last"], outs["fp32_nchw"])}
    res["shape"] = f"B={B} C={C} {H}x{W}, ks 4 dilation 1 sigma 2, smooth flow, both gradients"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--skip-cfg3", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_resample_16bit.py needs a GPU: nothing measured")
    import gfla_b200
    F_ = gfla_b200.functional
    dev = torch.device("cuda:0")
    r = {"card": card(), "steps": a.steps,
         "note": ("f4 feature tensors are 33.5 MB (bf16) / 67 MB (fp32) each, so an arm's working set is about "
                  "the size of the 126 MB L2 and partly served from it; cfg3 tensors (2.1 / 4.3 GB) are not"),
         "f4_relu3_1": f4(F_, 16, 256, 64, 64, a.steps, dev),
         "f4_relu2_1": f4(F_, 16, 128, 128, 128, a.steps, dev)}
    if not a.skip_cfg3:
        r["cfg3_ks4"] = cfg3(F_, max(3, a.steps // 4), dev)
    line = json.dumps(r, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
