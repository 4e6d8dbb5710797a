#!/usr/bin/env python
"""bench.py -- the warping hot path on B200, measured the way BASELINE.json asks.

    python bench.py [--gpus N] [--steps K] [--warmup W]          our CUDA path
    python bench.py --impl reference [...]                        the reference's CPU path
    python bench.py --dump-outputs DIR [...]                      also write what the last timed step returned, DIR/<name>.npy

Workload (BASELINE.json configs[1], the configuration the metric is quoted on):
fused block_extractor + local_attn_reshape + softmax ("ExtractorAttn tail",
model/networks/base_function.py:804-810), forward + backward, per GPU
B=16, C=256, 256x256, k=5, bf16 data / fp32 flow, synthetic smooth flow.
One step = one forward + one backward over that batch.  Weak scaling: every rank
owns its own B=16 batch shard (the path has no cross-sample dependence, so there is
no data-path collective; see gfla_b200/sharding.py).

Printed JSON (one line, rank 0):
  value      Mpixels/s (B*H*W output pixels, fwd+bwd) with inputs resident in HBM,
             whole job (sum over ranks / max-over-ranks device time)
  e2e        same metric through the public autograd API with HOST (pinned) buffers:
             H2D of source/flow/logits/grad_out and D2H of out + the three gradients
             inside the timed region
  roofline   dominant kernel of the step: algorithmic bytes / CUDA-event duration vs
             the measured HBM peak (MEASURED_PEAKS.json); roofline_fwd: the fused forward
  cpu_baseline  the reference's own kernel bodies on the host cores (oracle/_ref),
             bounded sample, rank 0 / N=1 only
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "warp-layer Mpixels/s (fwd+bwd) @256^2 C=256 k=5"
UNIT = "Mpixels/s"
CFG = dict(B=16, C=256, H=256, W=256, k=5)


# ----------------------------------------------------------------------------- helpers
def algorithmic_bytes(B, C, H, W, k, elt=2):
    """SURVEY.md 8(d) / BASELINE.md section 2, bf16 data + fp32 flow.
    fwd: read source, write out (C*elt each), read flow (2*4), read logits (k*k*elt)
    bwd: read grad_out, source (C*elt each), flow, logits; write grad_source (C*elt), grad_flow (8), grad_logits"""
    px = B * H * W
    fwd = 2 * C * elt + 8 + k * k * elt
    bwd = 3 * C * elt + 8 + k * k * elt + 8 + k * k * elt
    return px * fwd, px * bwd


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "samples": len(rows), "power_w_max": max(float(r[3]) for r in rows)}


def make_inputs(torch, dev, B, C, H, W, k, seed, flow_kind="smooth"):
    g = torch.Generator(device="cpu").manual_seed(seed)
    src = torch.randn(B, C, H, W, generator=g).bfloat16()
    if flow_kind == "smooth":   # bilinear x16 up-sampling of U(-8,8) noise (SURVEY.md 8d)
        coarse = torch.rand(B, 2, H // 16, W // 16, generator=g) * 16 - 8
        flow = torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True).contiguous()
    else:
        flow = torch.rand(B, 2, H, W, generator=g) * 16 - 8
    logits = torch.randn(B, k * k, H, W, generator=g).bfloat16()
    gout = torch.randn(B, C, H, W, generator=g).bfloat16()
    return src, flow.float(), logits, gout


# ----------------------------------------------------------------------------- CPU reference leg
REF_ROWS = 64      # fixed strip of the 256x256 map that one reference step processes (bounded sample)


def host_flow(np, torch, rng, kind, rows, W):
    """the same two flow families as the GPU arm (make_inputs): smooth = x16 bilinear up-sampling of U(-8,8), iid = U(-8,8)"""
    if kind == "smooth":
        coarse = torch.from_numpy(rng.uniform(-8, 8, (1, 2, max(rows // 16, 2), W // 16)))
        return torch.nn.functional.interpolate(coarse, size=(rows, W), mode="bilinear", align_corners=True).numpy().astype(np.float32)
    return rng.uniform(-8, 8, (1, 2, rows, W)).astype(np.float32)


def cpu_reference_run(steps, warmup, flow_kind="smooth", rows=REF_ROWS):
    """Times the reference's CPU implementation of the path (its own kernel bodies compiled
    for the host + torch CPU ops for softmax/mul/avg_pool, oracle/ref_pipeline.py) on a bounded
    sample of the cfg2 workload: B=1, full C=256, k=5, a FIXED strip of `rows` rows x 256 columns, fp32
    (the reference has no bf16), the same flow family as the GPU arm.  Thread count is set explicitly
    (torchrun exports OMP_NUM_THREADS=1): the host build's atomics (`#pragma omp atomic` standing in for
    atomicAdd) collide C*k*k-fold on grad_flow, so more threads are not always faster (128 threads across two sockets
    measured 5x SLOWER than 64 on one) -- a short probe picks the best of {1, 8, 32, half, all} cores and `cores` states what
    the timed steps used.
    Returns the cpu_baseline dict and per-step seconds."""
    import numpy as np
    import torch
    import oracle.oracle as orc
    from oracle.ref_pipeline import local_attn_fwd_bwd
    ncpu = max(1, len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    if orc.have_ref():
        lib, kind = orc.Ref(), "reference"
    else:
        orc.build(ref=False)
        lib, kind = orc.Oracle(), "port"
    torch.set_num_threads(ncpu)
    C, W, k = CFG["C"], CFG["W"], CFG["k"]
    rng = np.random.default_rng(0)
    src = rng.standard_normal((1, C, CFG["H"], W)).astype(np.float32)
    flow = host_flow(np, torch, rng, flow_kind, rows, W)
    logits = rng.standard_normal((1, k * k, rows, W)).astype(np.float32)
    g = rng.standard_normal((1, C, rows, W)).astype(np.float32)

    def run(r=rows):
        t = time.perf_counter()
        c = np.ascontiguousarray
        local_attn_fwd_bwd(lib, src, c(flow[:, :, :r]), c(logits[:, :, :r]), c(g[:, :, :r]), k)
        return time.perf_counter() - t

    cores = 1
    if kind == "reference":
        probe = {}
        for n in sorted({n for n in (1, 8, 32, ncpu // 2, ncpu) if 1 <= n <= ncpu}):
            lib.set_threads(n)
            run(8)                                       # page-in / thread-pool warm-up
            probe[n] = run(8)
        cores = min(probe, key=probe.get)
        lib.set_threads(cores)
    for _ in range(warmup):
        run()
    times = [run() for _ in range(steps)]
    sec = sum(times) / len(times)
    mpx = rows * W / sec / 1e6
    return {"value": mpx, "unit": UNIT, "cores": cores, "host_cores": ncpu, "kind": kind,
            "sample": f"B=1 C={C} k={k} fp32, fixed strip of {rows} rows x {W} cols of the 256x256 map, {flow_kind} flow, fwd+bwd, "
                      f"{steps} steps (+{warmup} warm-up), unfused reference pipeline; threads = best of {{1, 8, 32, {ncpu // 2}, {ncpu}}} on an 8-row probe"}, sec


def bind_to_gpu_numa_node(torch, local_rank):
    """pin this process (and so its pinned host buffers, first-touch) to the NUMA node the GPU hangs off"""
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        devid = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devid:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


DUMP_SAMPLE = 1 << 21      # elements kept of a larger output: the four outputs of the cfg2 step take 32 MB in float32


def sample_outputs(torch, named):
    """{name: float32 numpy array} of the step's outputs, in logical [B,C,H,W] order whatever the storage; an output with
    more than DUMP_SAMPLE elements is reduced to the same DUMP_SAMPLE seeded positions (sorted) on every run"""
    res = {}
    for name, t in named.items():
        flat = t.detach().reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            g = torch.Generator(device="cpu").manual_seed(0)
            idx = torch.randint(0, flat.numel(), (DUMP_SAMPLE,), generator=g).sort().values
            flat = flat[idx.to(flat.device)]
        res[name] = flat.float().cpu().numpy()
    return res


def _time(torch, fn, warm, n):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def extras(torch, F_, dev, args, peak, peak_kind):
    """Extra keys of the N=1 line (each bounded to a fraction of a second of GPU time):
      iid_flow        the same cfg2 step with iid U(-8,8) flow (SURVEY.md 8d: adversarial for the tiling)
      cfg3            BASELINE config 3: resample2d fwd+bwd, B=32 C=128 512x512 fp32, kernel_size 2 (module default) and 4
                      (what training uses), each with its own HBM roofline (1036 / 1560 algorithmic B per pixel, SURVEY.md 8d)
      f4_resample_cosine   the fused resample2d -> cosine op vs the unfused modules (SURVEY row f4), fwd+bwd
      reference_cuda  the reference's own CUDA kernels recompiled for sm_100a (oracle/_ref/libgfla_ref_cuda.so), running the
                      unfused ExtractorAttn tail in fp32 on 2 samples of the cfg2 shape -- the same-box GPU baseline"""
    out = {}
    B, C, H, W, k = (CFG[x] for x in "BCHWk")
    cl = torch.channels_last
    try:
        src, flow, logits, gout = (t.to(dev) for t in make_inputs(torch, dev, B, C, H, W, k, seed=4321, flow_kind="iid"))
        src, gout = src.contiguous(memory_format=cl), gout.contiguous(memory_format=cl)
        f_ms = _time(torch, lambda: F_.local_attn_fwd(src, flow, logits, k), 3, 10)
        b_ms = _time(torch, lambda: F_.local_attn_bwd(src, flow, logits, gout, k), 3, 10)
        fb, bb = algorithmic_bytes(B, C, H, W, k)
        out["iid_flow"] = {"value": B * H * W / ((f_ms + b_ms) * 1e-3) / 1e6, "unit": UNIT, "fwd_ms": f_ms, "bwd_ms": b_ms,
                           "fwd_frac": fb / (f_ms * 1e-3) / 1e9 / peak, "bwd_frac": bb / (b_ms * 1e-3) / 1e9 / peak, "steps": 10}
        del src, flow, logits, gout
    except Exception as exc:
        out["iid_flow"] = {"error": repr(exc)[:200]}
    try:
        Bc, Cc, Hc, Wc = 32, 128, 512, 512
        g = torch.Generator(device="cpu").manual_seed(5)
        coarse = torch.rand(Bc, 2, Hc // 16, Wc // 16, generator=g) * 16 - 8
        flow = torch.nn.functional.interpolate(coarse, size=(Hc, Wc), mode="bilinear", align_corners=True).to(dev)
        x = torch.randn(Bc, Cc, Hc, Wc, device=dev)
        go = torch.randn(Bc, Cc, Hc, Wc, device=dev)
        px = Bc * Hc * Wc
        c3 = {}
        for ks, sigma in ((2, 5.0), (4, 2.0)):
            in2 = torch.cat([flow, torch.full((Bc, 1, Hc, Wc), sigma, device=dev)], 1).contiguous()
            f_ms = _time(torch, lambda: F_.resample2d_fwd(x, in2, ks, 1), 2, 5)
            b_ms = _time(torch, lambda: F_.resample2d_bwd(x, in2, go, ks, 1), 2, 5)
            fwd_b, bwd_b = px * (2 * Cc * 4 + 12), px * (3 * Cc * 4 + 24)
            c3[f"ks{ks}"] = {"value": px / ((f_ms + b_ms) * 1e-3) / 1e6, "unit": UNIT, "fwd_ms": f_ms, "bwd_ms": b_ms, "sigma": sigma,
                            "roofline": {"bound": "hbm", "achieved": (fwd_b + bwd_b) / ((f_ms + b_ms) * 1e-3) / 1e9, "peak": peak,
                                         "peak_source": peak_kind, "unit": "GB/s", "frac": (fwd_b + bwd_b) / ((f_ms + b_ms) * 1e-3) / 1e9 / peak,
                                         "frac_fwd": fwd_b / (f_ms * 1e-3) / 1e9 / peak, "frac_bwd": bwd_b / (b_ms * 1e-3) / 1e9 / peak}}
            del in2
        c3["workload"] = "cfg3: resample2d fwd+bwd, B=32 C=128 512x512 fp32, smooth flow, dilation 1"
        out["cfg3"] = c3
        del x, go, flow
    except Exception as exc:
        out["cfg3"] = {"error": repr(exc)[:200]}
    torch.cuda.empty_cache()
    try:
        # f4: PerceptualCorrectness' resample -> cosine step at the VGG relu3_1 / relu2_1 shapes of a 256x256 batch of 16
        # (external_function.py:275-279): ONE fused kernel each way vs Resample2d + F.cosine_similarity through autograd;
        # gradient to the flow only, like the loss
        import gfla_b200
        f4 = {}
        for name, (Bf, Cf, Hf) in (("relu3_1", (16, 256, 64)), ("relu2_1", (16, 128, 128))):
            gen = torch.Generator(device="cpu").manual_seed(Hf)
            xs = torch.randn(Bf, Cf, Hf, Hf, generator=gen).to(dev)
            tg = torch.randn(Bf, Cf, Hf, Hf, generator=gen).to(dev)
            coarse = torch.rand(Bf, 2, Hf // 8, Hf // 8, generator=gen) * 8 - 4
            fl = torch.nn.functional.interpolate(coarse, size=(Hf, Hf)).to(dev).requires_grad_()     # nearest, like the loss (:254)
            fused_m, plain_m = gfla_b200.Resample2dCosine(4, 1, sigma=2), gfla_b200.Resample2d(4, 1, sigma=2)
            go = torch.randn(Bf, Hf, Hf, device=dev)

            def fused():
                fl.grad = None
                fused_m(xs, fl, tg).backward(go)

            def unfused():
                fl.grad = None
                torch.nn.functional.cosine_similarity(plain_m(xs, fl), tg, dim=1, eps=1e-8).backward(go)
            t_f, t_u = _time(torch, fused, 3, 10), _time(torch, unfused, 3, 10)
            alg = Bf * Hf * Hf * (2 * 2 * Cf * 4 + 60)            # source + target read once each way, per-pixel planes
            f4[name] = {"shape": [Bf, Cf, Hf, Hf], "fused_ms": t_f, "unfused_ms": t_u, "speedup": t_u / t_f,
                        "roofline_frac": alg / (t_f * 1e-3) / 1e9 / peak}
            del xs, tg, fl, go
        f4["workload"] = "resample2d(ks 4, sigma 2) -> cosine_similarity fwd+bwd (grad to the flow), fp32, blocky (nearest-upsampled) flow"
        out["f4_resample_cosine"] = f4
    except Exception as exc:
        out["f4_resample_cosine"] = {"error": repr(exc)[:200]}
    torch.cuda.empty_cache()
    try:
        import oracle.ref_cuda as rc
        if not rc.available():
            raise FileNotFoundError("oracle/_ref/libgfla_ref_cuda.so not built")
        nb = 2
        src, flow, logits, gout = (t.to(dev) for t in make_inputs(torch, dev, nb, C, H, W, k, seed=77, flow_kind=args.flow))
        s32, l32, g32 = src.float(), logits.float(), gout.float()
        ms = _time(torch, lambda: rc.local_attn_fwd_bwd(s32, flow, l32, g32, k, chunk=1), 1, 2)
        out["reference_cuda"] = {"value": nb * H * W / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_sample": ms / nb, "dtype": "f32",
                                 "kind": "reference CUDA kernels (block_extractor / local_attn_reshape) recompiled for sm_100a + torch softmax/mul/avg_pool",
                                 "sample": f"{nb} samples of the cfg2 shape (C={C} {H}x{W} k={k}), fwd+bwd, one sample per launch (the reference's int n limit)"}
    except Exception as exc:
        out["reference_cuda"] = {"unavailable": repr(exc)[:200]}
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--flow", default="smooth", choices=["smooth", "iid"])
    ap.add_argument("--algo", default="auto", choices=["auto", "gather", "tile"])
    ap.add_argument("--layout", default="nhwc", choices=["nhwc", "nchw"],
                    help="storage of the [B,C,H,W] feature tensors: channels_last (default, the tile kernels' fast layout) or contiguous NCHW")
    ap.add_argument("--e2e-chunks", type=int, default=4, help="e2e leg: number of batch chunks per step")
    ap.add_argument("--e2e-streams", type=int, default=2, help="e2e leg: CUDA streams the chunks alternate between")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4", "cfg5"],
                    help="cfg2 (default, the BASELINE metric): fused warp layer fwd+bwd; cfg4 / cfg5: the reference's Pose / Face generator on these ops (bench_models.py)")
    ap.add_argument("--model-dtype", default="bf16", choices=["bf16", "fp32"], help="cfg4/cfg5: parameter / activation dtype")
    ap.add_argument("--arms", default="fused,literal,refcuda", help="cfg4/cfg5: comma list, first = the reported value")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra keys (iid flow, cfg3 resample2d, reference CUDA kernels)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (out, grad_source, grad_flow, grad_logits of rank 0) as "
                         f"DIR/<name>.npy in float32; an output above {DUMP_SAMPLE} elements is a fixed seeded sample of it")
    args = ap.parse_args()
    if args.dump_outputs is not None:
        if args.workload != "cfg2" or args.impl != "ours":
            ap.error("--dump-outputs covers the default workload on the GPU (--workload cfg2 --impl ours)")
        os.makedirs(args.dump_outputs, exist_ok=True)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, C, H, W, k = (CFG[x] for x in "BCHWk")
    config = {"workload": f"cfg2: fused block_extractor+local_attn_reshape+softmax fwd+bwd, per-GPU B={B} C={C} "
                          f"{H}x{W} k={k}, bf16 data / fp32 flow ({args.flow} flow)",
              "per_gpu_batch": B, "global_batch": B * world, "C": C, "H": H, "W": W, "k": k,
              "flow": args.flow, "layout": "channels_last (NHWC storage)" if args.layout == "nhwc" else "contiguous NCHW",
              "sharding": f"batch x{world} (no data-path collective)",
              "l2": "inputs (>=1 GiB per step) exceed the 126 MB L2; no explicit flush"}

    if args.workload != "cfg2":
        if args.impl == "reference":
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the reference has no CPU path for its generators "
                                  "(block_extractor.py:23-24 raises on CPU tensors); its CUDA kernels run as the `refcuda` arm of "
                                  f"`bench.py --workload {args.workload}`"}), flush=True)
            return 0
        import bench_models
        return bench_models.run(args)

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        steps, warmup = max(1, args.steps), max(0, args.warmup)
        cb, sec = cpu_reference_run(steps, warmup, flow_kind=args.flow)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": steps, "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    import gfla_b200
    from gfla_b200 import functional as F_
    from gfla_b200 import _lib
    from gfla_b200.sharding import reduce_max_time

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa_node(torch, local_rank)      # before any pinned allocation (e2e host buffers)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.lib().gfla_device_check(), "device check")
    steps, warmup = max(1, args.steps), max(3, args.warmup)

    src_h, flow_h, logits_h, gout_h = make_inputs(torch, dev, B, C, H, W, k, seed=1234 + rank, flow_kind=args.flow)
    if args.layout == "nhwc":   # torch.channels_last: same logical [B,C,H,W] tensors, pixel-major storage
        src_h = src_h.contiguous(memory_format=torch.channels_last)
        gout_h = gout_h.contiguous(memory_format=torch.channels_last)
    src, flow, logits, gout = (t.to(dev) for t in (src_h, flow_h, logits_h, gout_h))

    def step(record=None):
        if record is not None:
            record[0].record()
        out = F_.local_attn_fwd(src, flow, logits, k, algo=args.algo)
        if record is not None:
            record[1].record()
        grads = F_.local_attn_bwd(src, flow, logits, gout, k)
        if record is not None:
            record[2].record()
        return out, grads

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    for _ in range(warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    barrier()
    t_wall0 = time.time()
    launches0 = _lib.lib().gfla_debug_launch_count()
    last = None
    for i in range(steps):
        last = None            # the previous step's outputs are freed before the next step, as if they were discarded
        last = step(ev[i])
    launches = int(_lib.lib().gfla_debug_launch_count() - launches0)   # kernels of libgfla_warp.so launched in the timed region
    barrier()
    t_wall1 = time.time()
    dump = None
    if args.dump_outputs is not None and rank == 0:
        out, (gs, gf, gl) = last
        dump = sample_outputs(torch, {"out": out, "grad_source": gs, "grad_flow": gf, "grad_logits": gl})
        del out, gs, gf, gl
    del last
    total_ms = ev[0][0].elapsed_time(ev[-1][2])
    fwd_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
    bwd_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
    total_ms = reduce_max_time(total_ms, dev)
    ms_per_step = total_ms / steps
    value = world * B * H * W / (ms_per_step * 1e-3) / 1e6

    # ---- the same step with planar (contiguous NCHW) feature tensors, for callers that keep the reference's layout:
    #      forward = NCHW variant of the tile kernel, backward = re-layout + channels-last tile kernels + re-layout
    nchw = None
    if args.layout == "nhwc":
        src_p, gout_p = src.contiguous(), gout.contiguous()
        def step_planar():
            F_.local_attn_fwd(src_p, flow, logits, k, algo=args.algo)
            F_.local_attn_bwd(src_p, flow, logits, gout_p, k)
        for _ in range(3):
            step_planar()
        barrier()
        a_, b__ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p_steps = steps
        a_.record()
        for _ in range(p_steps):
            step_planar()
        b__.record()
        barrier()
        p_ms = reduce_max_time(a_.elapsed_time(b__), dev) / p_steps
        nchw = {"value": world * B * H * W / (p_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": p_ms, "steps": p_steps,
                "note": "contiguous NCHW feature tensors (the reference's layout), same workload"}
        del src_p, gout_p

    # ---- e2e: public autograd API, host buffers, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        pin = lambda t: t.pin_memory()
        hs, hf, hl, hg = pin(src_h), pin(flow_h), pin(logits_h), pin(gout_h)
        ho = torch.empty_like(hs).pin_memory()
        hgs, hgf, hgl = torch.empty_like(hs).pin_memory(), torch.empty_like(hf).pin_memory(), torch.empty_like(hl).pin_memory()
        h2d = sum(t.numel() * t.element_size() for t in (hs, hf, hl, hg))
        d2h = sum(t.numel() * t.element_size() for t in (ho, hgs, hgf, hgl))

        # The batch is processed in chunks (default 4 of 4 samples) alternating between streams (default 2), so the H2D of chunk i+1 overlaps the
        # kernels and the D2H of chunk i (PCIe is full duplex; every byte is still copied inside the timed region, through
        # the public autograd API, once per step).  The two streams are joined to the timing stream once in front of the
        # first step and once behind the last one -- consecutive steps pipeline like consecutive chunks (a chunk always
        # returns to the stream that handled the same host slices in the previous step, so host buffers are reused in order).
        # Host buffers are pinned on the GPU's own NUMA node (see above).
        per = max(1, B // max(1, args.e2e_chunks))
        chunks = [(b0, min(B, b0 + per)) for b0 in range(0, B, per)]
        side = [torch.cuda.Stream(device=dev) for _ in range(max(1, min(args.e2e_streams, len(chunks))))]
        assert len(chunks) % len(side) == 0, "chunks must be a multiple of streams (a host slice always returns to the same stream)"

        def e2e_steps_run(n):
            main = torch.cuda.current_stream(dev)
            for st in side:
                st.wait_stream(main)
            for _ in range(n):
                for ci, (b0, b1) in enumerate(chunks):
                    with torch.cuda.stream(side[ci % len(side)]):
                        s = hs[b0:b1].to(dev, non_blocking=True).requires_grad_()
                        f = hf[b0:b1].to(dev, non_blocking=True).requires_grad_()
                        l = hl[b0:b1].to(dev, non_blocking=True).requires_grad_()
                        g = hg[b0:b1].to(dev, non_blocking=True)
                        out = gfla_b200.local_attention(s, f, l, k)          # the call a user makes
                        out.backward(g)
                        ho[b0:b1].copy_(out.detach(), non_blocking=True)
                        hgs[b0:b1].copy_(s.grad, non_blocking=True)
                        hgf[b0:b1].copy_(f.grad, non_blocking=True)
                        hgl[b0:b1].copy_(l.grad, non_blocking=True)
            for st in side:
                main.wait_stream(st)

        e2e_steps = steps
        e2e_steps_run(2)
        barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e2e_steps_run(e2e_steps)
        b_.record()
        barrier()
        e2e_ms = reduce_max_time(a.elapsed_time(b_), dev) / e2e_steps
        e2e = {"value": world * B * H * W / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps, "numa_node": numa_node,
               "chunks": len(chunks), "streams": len(side), "pipelined_across_steps": True}
    if rank == 0:
        sampler.stop()
    if dump is not None:
        import numpy as np
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_kind = measured_peak_gbs()
    fwd_bytes, bwd_bytes = algorithmic_bytes(B, C, H, W, k)

    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures
    # (profiles/traffic.json; cold-cache single launch at this exact workload), or null
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        traffic = {}

    def roof(nbytes, ms, kernel, tkey=None):
        ach = nbytes / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": kernel, "achieved": ach, "peak": peak, "peak_source": peak_kind, "unit": "GB/s",
                "frac": ach / peak, "traffic": traffic.get(tkey) if args.layout == "nhwc" and args.flow == "smooth" else None,
                "algorithmic_bytes": nbytes, "launch_ms": ms}

    rf_fwd = roof(fwd_bytes, fwd_ms, "k_local_attn_fwd_strip (fused forward)", "fwd")
    fused_bwd = os.environ.get("GFLA_BWD_FUSED", "1") != "0"
    rf_bwd = roof(bwd_bytes, bwd_ms, "k_local_attn_bwd_fused (fused backward, zero fill of grad_source inside the kernel)" if fused_bwd
                  else "k_local_attn_bwd_gs_tc + k_local_attn_bwd_q_tc + grad_source memset", "bwd")
    rf_fwd["share_of_step"], rf_bwd["share_of_step"] = fwd_ms / ms_per_step, bwd_ms / ms_per_step
    # The step is two launches: the fused forward (~1/3 of the time) and the fused backward (~2/3; ncu launch list:
    # profiles/r2_bench_launches.md).  `roofline` describes the DOMINANT one by measured share; both are always reported.
    dominant = dict(rf_bwd if bwd_ms >= fwd_ms else rf_fwd)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "config": config,
            "roofline": dominant, "roofline_fwd": rf_fwd, "roofline_bwd": rf_bwd,
            "step_roofline_frac": (fwd_bytes + bwd_bytes) / (ms_per_step * 1e-3) / 1e9 / peak,
            "clocks": sampler.summary(t_wall0, t_wall1),
            "planar_nchw": nchw,
            "gpu_launches": launches,    # counted by the library (gfla_debug_launch_count) across the timed region
            "e2e": e2e}
    if world == 1 and not args.no_extras:
        line.update(extras(torch, F_, dev, args, peak, peak_kind))
    if world == 1 and not args.no_cpu_baseline:
        try:
            cb, _ = cpu_reference_run(steps=2, warmup=0, flow_kind=args.flow)
            line["cpu_baseline"] = cb
        except Exception as exc:  # the baseline leg must never take the bench line down
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": repr(exc)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
