#!/usr/bin/env python
"""Generate the golden vectors in tests/golden/*.npz.

Run in the BUILD container only (needs /root/reference to build oracle/_ref):

    python tests/golden/make_golden.py

Ground truth = the reference's own CUDA kernel bodies compiled for the host
(``oracle/_ref/libgfla_ref.so``, one thread, see oracle/Makefile) and, for the
``ExtractorAttn`` tail, those bodies composed with stock torch CPU ops exactly
as ``model/networks/base_function.py:804-810`` composes them (Softmax(dim=1),
broadcast multiply, ``avg_pool2d(k, k)``), differentiated by torch autograd
with the reference backward bodies plugged in as custom Functions -- the same
structure as ``block_extractor.py:5-42`` / ``local_attn_reshape.py:5-37``.

The reference ships no golden files; the only results its own tests pin are two
layout identities (``test_block_extractor.py:55``, ``test_local_attn_reshape.py:29-43``)
and two double-precision gradchecks (``test_block_extractor.py:74-78``,
``test_local_attn_reshape.py:66-70``).  Both identities are stored here as
cases; the gradcheck shapes are reproduced in tests/.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle.oracle as orc  # noqa: E402
from conftest import FixedFeatures, golden_grad_out, perceptual_inputs, sample_index, sha256  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def smooth_flow(rng, B, H, W, amp, cell=4):
    """bilinear up-sampling of coarse U(-amp, amp) noise (SURVEY.md 8d 'smooth')."""
    coarse = torch.from_numpy(rng.uniform(-amp, amp, (B, 2, max(H // cell, 2), max(W // cell, 2))))
    return torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True).numpy()


def main():
    orc.build(ref=True)
    R = orc.Ref(threads=1)
    rng = np.random.default_rng(20260923)

    # ------------------------------------------------------------------ block_extractor
    be = {}
    cases = [
        # name, dtype, B, C, Hs, Ws, Hf, Wf, k, flow kind
        ("cfg1", np.float32, 1, 8, 32, 32, 32, 32, 3, "iid8"),          # BASELINE.json configs[0]
        ("k4_border", np.float32, 2, 3, 9, 7, 9, 7, 4, "border"),       # even k: offsets -2..1; taps cross every border
        ("k5_smooth", np.float32, 2, 5, 16, 16, 16, 16, 5, "smooth"),
        ("src_gt_flow", np.float32, 1, 2, 12, 14, 10, 12, 3, "const"),  # external_function.py:61-66 usage
        ("zero_flow", np.float32, 2, 3, 8, 8, 8, 8, 3, "zero"),         # test_block_extractor.py:46-55
        ("gradcheck_shape", np.float64, 4, 6, 14, 10, 14, 10, 3, "rand1.8"),  # test_block_extractor.py:74-78
        ("k2", np.float64, 1, 2, 6, 5, 6, 5, 2, "iid8"),
    ]
    for seed, (name, dt, B, C, Hs, Ws, Hf, Wf, k, kind) in enumerate(cases):
        src = rng.standard_normal((B, C, Hs, Ws)).astype(dt)
        if kind == "iid8":
            flow = rng.uniform(-8, 8, (B, 2, Hf, Wf))
        elif kind == "border":
            flow = rng.uniform(-1.5 * Wf, 1.5 * Wf, (B, 2, Hf, Wf))
        elif kind == "smooth":
            flow = smooth_flow(rng, B, Hf, Wf, 6.0)
        elif kind == "const":
            flow = np.full((B, 2, Hf, Wf), float(k // 2))
        elif kind == "zero":
            flow = np.zeros((B, 2, Hf, Wf))
        elif kind == "rand1.8":
            flow = rng.uniform(0, 1, (B, 2, Hf, Wf)) * 1.8
        flow = np.ascontiguousarray(flow.astype(dt))
        out = R.block_extract_fwd(src, flow, k)
        # out and grad_out are k*k times the size of the source, so neither is stored: out is compared bit for bit and
        # its digest stands in for it; grad_out comes from a stored seed (conftest.load_golden rebuilds it)
        rng.standard_normal(out.shape)      # an unused draw that keeps the later sections' inputs as committed
        gout = golden_grad_out(seed, out.shape, dt)
        gs, gf = R.block_extract_bwd(src, flow, gout, k)
        for key, v in dict(source=src, flow=flow, out_sha256=np.str_(sha256(out)), grad_out_seed=np.int64(seed),
                           grad_out_shape=np.array(out.shape, np.int64), grad_source=gs, grad_flow=gf, k=np.int32(k)).items():
            be[f"{name}/{key}"] = v
    np.savez_compressed(os.path.join(OUT, "block_extractor.npz"), **be)

    # ------------------------------------------------------------------ local_attn_reshape
    lr = {}
    x = np.arange(9, dtype=np.float32).reshape(1, 9, 1, 1).repeat(2, 0).repeat(10, 2).repeat(10, 3)
    x = np.ascontiguousarray(x)                       # test_local_attn_reshape.py:29-31
    lr["layout/in"], lr["layout/out"], lr["layout/k"] = x, R.attn_reshape_fwd(x, 3), np.int32(3)
    for name, dt, B, H, W, k in [("k3", np.float64, 4, 14, 10, 3), ("k5", np.float32, 2, 6, 7, 5), ("k4", np.float32, 1, 3, 5, 4)]:
        x = rng.standard_normal((B, k * k, H, W)).astype(dt)
        out = R.attn_reshape_fwd(x, k)
        g = rng.standard_normal(out.shape).astype(dt)
        lr[f"{name}/in"], lr[f"{name}/out"], lr[f"{name}/grad_out"] = x, out, g
        lr[f"{name}/grad_in"], lr[f"{name}/k"] = R.attn_reshape_bwd(x, g, k), np.int32(k)
    np.savez_compressed(os.path.join(OUT, "local_attn_reshape.npz"), **lr)

    # ------------------------------------------------------------------ resample2d
    rs = {}
    cases = [
        # name, dtype, B, C, Hi, Wi, H, W, ks, dil, sigma, flow amp
        ("ks2_default", np.float32, 2, 4, 12, 10, 12, 10, 2, 1, 5.0, 3.0),   # Resample2d() defaults, resample2d.py:43
        ("ks4_sigma2", np.float32, 2, 3, 10, 12, 10, 12, 4, 1, 2.0, 3.0),    # external_function.py:233
        ("ks4_border", np.float32, 1, 2, 8, 8, 8, 8, 4, 1, 2.0, 14.0),       # x+dx < 0: int() vs floor() quirk (:137-138)
        ("ks4_dil2", np.float64, 1, 2, 9, 9, 9, 9, 4, 2, 2.0, 3.0),
        ("in_ne_out", np.float32, 1, 3, 14, 9, 7, 11, 2, 1, 5.0, 3.0),
        ("sigma0", np.float32, 1, 2, 6, 6, 6, 6, 2, 1, 0.0, 2.0),            # SAFE_DIV EPS branch (:14-15)
    ]
    for name, dt, B, C, Hi, Wi, H, W, ks, dil, sigma, amp in cases:
        in1 = rng.standard_normal((B, C, Hi, Wi)).astype(dt)
        flow = rng.uniform(-amp, amp, (B, 2, H, W)).astype(dt)
        in2 = np.ascontiguousarray(np.concatenate([flow, np.full((B, 1, H, W), sigma, dt)], 1))  # resample2d.py:51-52
        out = R.resample2d_fwd(in1, in2, ks, dil)
        g = rng.standard_normal(out.shape).astype(dt)
        g1, g2 = R.resample2d_bwd(in1, in2, g, ks, dil)
        for key, v in dict(in1=in1, in2=in2, out=out, grad_out=g, grad_in1=g1, grad_in2=g2,
                           ks=np.int32(ks), dil=np.int32(dil)).items():
            rs[f"{name}/{key}"] = v
    np.savez_compressed(os.path.join(OUT, "resample2d.npz"), **rs)

    # ------------------------------------------------------------------ ExtractorAttn tail (fused op)
    from oracle.ref_pipeline import local_attn_fwd_bwd

    la = {}
    cases = [
        ("k3", np.float32, 2, 6, 10, 9, 3, "smooth"),
        ("k5", np.float32, 1, 8, 12, 12, 5, "iid8"),
        ("k5_border", np.float32, 1, 3, 7, 8, 5, "border"),
        ("k4_f64", np.float64, 1, 4, 6, 6, 4, "iid8"),
        ("k3_f64", np.float64, 2, 5, 9, 8, 3, "smooth"),
    ]
    for name, dt, B, C, H, W, k, kind in cases:
        src = rng.standard_normal((B, C, H, W)).astype(dt)
        if kind == "iid8":
            flow = rng.uniform(-8, 8, (B, 2, H, W))
        elif kind == "border":
            flow = rng.uniform(-1.5 * W, 1.5 * W, (B, 2, H, W))
        else:
            flow = smooth_flow(rng, B, H, W, 4.0)
        flow = np.ascontiguousarray(flow.astype(dt))
        logits = (2.0 * rng.standard_normal((B, k * k, H, W))).astype(dt)
        g = rng.standard_normal((B, C, H, W)).astype(dt)
        out, probs, gs, gf, gl = local_attn_fwd_bwd(R, src, flow, logits, g, k)   # base_function.py:804-810
        for key, v in dict(source=src, flow=flow, logits=logits, out=out, probs=probs, grad_out=g, grad_source=gs,
                           grad_flow=gf, grad_logits=gl, k=np.int32(k)).items():
            la[f"{name}/{key}"] = v
    np.savez_compressed(os.path.join(OUT, "local_attn.npz"), **la)

    oracle_vs_ref(R)
    reference_fullsize(R)
    reference_losses(R)
    reference_perceptual(R)

    for f in sorted(os.listdir(OUT)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


def oracle_vs_ref(R):
    """digests of the reference's outputs on tests/test_oracle_vs_ref.py's inputs (one thread, like the oracle)"""
    import test_oracle_vs_ref as T

    ref = {}

    def keep(name, outputs):
        for key, a in outputs.items():
            ref[f"{name}/{key}"] = np.str_(sha256(a))

    for dt in (np.float32, np.float64):
        for shape in T.BLOCK_SHAPES:
            keep(T.case_name("block_extractor", np.dtype(dt).name, *shape), T.block_outputs(R, dt, shape))
        for cfg in T.RESAMPLE_CFGS:
            keep(T.case_name("resample2d", np.dtype(dt).name, *cfg), T.resample_outputs(R, dt, cfg))
    for k in T.RESHAPE_KS:
        keep(T.case_name("reshape", k), T.reshape_outputs(R, k))
    np.savez_compressed(os.path.join(OUT, "oracle_vs_ref.npz"), **ref)


def reference_fullsize(R):
    """tests/test_gpu_refcuda.py's full-size cases (BASELINE configs 2 and 3): the reference's outputs at the fixed
    sample of positions, plus each output's largest magnitude (the tests' relative tolerances scale with it).  All host
    threads: the order of the atomic adds into grad_flow, and so its last bits (~1e-6 relative), vary from run to run."""
    import test_gpu_refcuda as T
    from oracle.ref_pipeline import local_attn_fwd_bwd

    R.set_threads(os.cpu_count() or 1)
    host = lambda *ts: [np.ascontiguousarray(t.numpy()) for t in ts]
    ref = {}

    def keep(case, **arrays):
        for name, a in arrays.items():
            ref[f"{case}/{name}"] = a.reshape(-1)[sample_index(a.size)].astype(np.float32)
            ref[f"{case}/{name}_absmax"] = np.float64(np.abs(a).max())

    for case in ("tile_smooth", "tile_iid", "planar", "fp32", "host"):
        inputs, k = T.cfg2_case(case, device="cpu")
        per_sample = [local_attn_fwd_bwd(R, *host(*(t[b:b + 1] for t in inputs)), k) for b in range(inputs[0].shape[0])]
        out, _, gs, gf, gl = (np.concatenate(parts) for parts in zip(*per_sample))
        keep(case, out=out, grad_source=gs, grad_flow=gf, grad_logits=gl)
    (src, flow, go), k = T.block_extractor_case(device="cpu")
    src, flow, go = host(src, flow, go)
    out = R.block_extract_fwd(src, flow, k)
    keep("block_extractor", out=out)
    del out
    gs, gf = R.block_extract_bwd(src, flow, go, k)
    keep("block_extractor", grad_source=gs, grad_flow=gf)
    for ks, sigma in ((2, 5.0), (4, 2.0)):
        (x, in2, go), _ = T.resample2d_case(ks, sigma, device="cpu")
        x, in2, go = host(x, in2, go)
        g1, g2 = R.resample2d_bwd(x, in2, go, ks, 1)
        keep(f"resample2d_ks{ks}", out=R.resample2d_fwd(x, in2, ks, 1), grad_in1=g1, grad_in2=g2)
    R.set_threads(1)
    np.savez_compressed(os.path.join(OUT, "reference_fullsize.npz"), **ref)


def reference_external_function():
    """the reference's model/networks/external_function.py on this package's ops (compat.install), importable here"""
    import types
    import gfla_b200
    from baseline import snapshot
    snapshot.snapshot()
    gfla_b200.compat.install(reference_root=snapshot.root())
    util = types.ModuleType("util")                   # external_function.py:8 (visualisation helpers, not needed here)
    util.util = types.ModuleType("util.util")
    sys.modules.setdefault("util", util)
    sys.modules.setdefault("util.util", util.util)
    from model.networks import external_function as ef
    return ef


def reference_losses(R):
    """what the reference's own AffineRegularizationLoss / MultiAffineRegularizationLoss classes compute
    (tests/test_reference_integration.py): the kernel per kz, flow2grid of a seeded flow, the layer order and kernel
    sizes; and (tests/test_gpu_models.py) the loss and its flow gradient on a seeded flow, with the two custom ops of
    the class on the reference's kernel bodies"""
    from oracle.ref_pipeline import make_functions
    ExtractFn, ReshapeFn = make_functions(R)

    class HostBlockExtractor(torch.nn.Module):
        def __init__(self, kz):
            super().__init__()
            self.kz = kz

        def forward(self, source, flow_field):
            return ExtractFn.apply(source.contiguous(), flow_field.contiguous(), self.kz)

    class HostLocalAttnReshape(torch.nn.Module):
        def forward(self, inputs, kernel_size):
            return ReshapeFn.apply(inputs.contiguous(), kernel_size)

    ef = reference_external_function()
    out = {}
    for kz in (3, 4, 5):
        loss = ef.AffineRegularizationLoss(kz)
        flow = torch.randn(2, 2, 9, 11, generator=torch.Generator().manual_seed(kz))
        out[f"kz{kz}/kernel"] = loss.kernel.numpy()
        out[f"kz{kz}/flow"], out[f"kz{kz}/grid"] = flow.numpy(), loss.flow2grid(flow).numpy()
        if kz != 4:
            loss.extractor, loss.reshape = HostBlockExtractor(kz), HostLocalAttnReshape()
            flow = (torch.randn(2, 2, 32, 32, generator=torch.Generator().manual_seed(kz)) * 3).requires_grad_()
            value = loss(flow)
            value.backward()
            out[f"kz{kz}/loss"], out[f"kz{kz}/loss_grad"] = np.float64(value.item()), flow.grad.numpy()
    m = ef.MultiAffineRegularizationLoss({"2": 5, "3": 3})
    out["multi/layers"] = np.array([int(x) for x in m.layers], np.int64)
    out["multi/kz"] = np.array([m.method_dic[x].kz for x in m.layers], np.int64)
    np.savez_compressed(os.path.join(OUT, "reference_losses.npz"), **out)


def reference_perceptual(R):
    """the reference's PerceptualCorrectness on conftest.perceptual_inputs with conftest.FixedFeatures as its feature
    extractor: loss and flow gradients, without and with the mask, through its grid_sample branch ("bilinear",
    tests/test_losses.py) and through its Resample2d(4, 1, sigma=2) branch ("resample", tests/test_gpu_resample_cosine.py),
    whose op runs on the reference's kernel bodies on the host"""
    import torchvision
    ef = reference_external_function()

    class HostResample2dFn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, in1, in2):
            ctx.save_for_backward(in1, in2)
            return torch.from_numpy(R.resample2d_fwd(in1.detach().numpy(), in2.detach().numpy(), 4, 1))

        @staticmethod
        def backward(ctx, g):
            in1, in2 = ctx.saved_tensors
            g1, g2 = R.resample2d_bwd(in1.detach().numpy(), in2.detach().numpy(), np.ascontiguousarray(g.numpy()), 4, 1)
            return torch.from_numpy(g1), torch.from_numpy(g2)

    class HostResample2d(torch.nn.Module):      # resample2d.py:43-51: sigma appended as a third flow channel
        def forward(self, input1, input2):
            b, _, h, w = input2.shape
            return HostResample2dFn.apply(input1.contiguous(), torch.cat([input2, torch.full((b, 1, h, w), 2.0)], 1).contiguous())

    vgg19 = torchvision.models.vgg19
    torchvision.models.vgg19 = lambda pretrained=False, **kw: vgg19(weights=None)     # built, then replaced: no weights needed
    try:
        loss = ef.PerceptualCorrectness()
    finally:
        torchvision.models.vgg19 = vgg19
    loss.vgg, loss.resample = FixedFeatures(), HostResample2d()
    target, source, mask, flows = perceptual_inputs()
    out = {}
    for branch in ("bilinear", "resample"):
        for name, m in (("nomask", None), ("mask", mask)):
            fs = [f.clone().requires_grad_() for f in flows]
            value = loss(target, source, fs, [2, 3], m, branch == "bilinear")
            value.backward()
            out[f"{branch}_{name}/loss"] = np.float64(value.item())
            for i, f in enumerate(fs):
                out[f"{branch}_{name}/grad{i}"] = f.grad.numpy()
    np.savez_compressed(os.path.join(OUT, "reference_perceptual.npz"), **out)


if __name__ == "__main__":
    main()
