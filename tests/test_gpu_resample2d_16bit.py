"""GPU (-m gpu): resample2d and the fused resample2d -> cosine op on bf16 / fp16 feature maps (channels-last kernels).

Oracle: the library's own fp32 planar path run on the 16-bit inputs widened to fp32 (tests/test_gpu_resample_cosine.py and
tests/test_gpu_parity.py pin that path to the CPU oracle).  The 16-bit kernels use the same taps and weights; what may
differ is the order of the sums over channels and the rounding at 16-bit stores, so:
  * forward output within 1 ulp (16-bit format) of the fp32 output rounded to the format;
  * cos, stats within 1e-5 of the largest magnitude; grad_input2 within 1e-4 of the largest magnitude;
  * grad_target, grad_input1 (fp32 scatter, narrowed) within 1 ulp + 1e-5 x the largest magnitude -- the cosine op's grad_input1
    also carries grad_val's 16-bit rounding (one relative ulp of each scattered contribution).
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EPS = 1e-8
MANT = {torch.bfloat16: 7, torch.float16: 10}
DTYPES = [torch.bfloat16, torch.float16]


@pytest.fixture(scope="module")
def F_():
    import gfla_b200
    from gfla_b200 import _lib
    _lib.check(_lib.lib().gfla_device_check(), "device check")
    return gfla_b200.functional


def ulp(ref16):
    """one unit in the last place of each element of a 16-bit tensor, in fp32"""
    dt = ref16.dtype
    a = ref16.float().abs()
    tiny = torch.finfo(dt).tiny
    e = torch.floor(torch.log2(torch.clamp(a, min=tiny)))
    return torch.exp2(e - MANT[dt])


def within_ulp(ours, ref32, rel=0.0, scale=None, extra=None):
    """|ours - ref32.to(dtype)| <= 1 ulp + rel * scale (+ extra), elementwise"""
    ref16 = ref32.to(ours.dtype)
    s = ref32.abs().max().item() if scale is None else scale
    tol = ulp(ref16) + rel * s + (0 if extra is None else extra)
    err = (ours.float() - ref16.float()).abs()
    bad = err > tol
    assert not bad.any(), f"{int(bad.sum())} elements off, worst {float((err - tol).max())}"


def _flow(kind, B, H, W, g):
    if kind == "smooth":
        ys, xs = torch.meshgrid(torch.arange(H, dtype=torch.float32), torch.arange(W, dtype=torch.float32), indexing="ij")
        f = torch.stack([2.5 * torch.sin(ys / 3.0 + xs / 7.0), 1.7 * torch.cos(xs / 5.0 - ys / 4.0)]).unsqueeze(0).repeat(B, 1, 1, 1)
        return f + 0.05 * torch.randn(B, 2, H, W, generator=g)
    if kind == "blocky":                      # nearest-upsampled: one integer shift per 4x4 block plus a shared fraction
        return torch.nn.functional.interpolate(torch.randn(B, 2, (H + 3) // 4, (W + 3) // 4, generator=g) * 3, size=(H, W))
    if kind == "border":                      # taps leave the image on every side (clamping)
        return (torch.rand(B, 2, H, W, generator=g) * 2 - 1) * 14
    if kind == "negx":                        # x + dx < 0: int() and floor() disagree (grad input1's fraction)
        xs = torch.arange(W, dtype=torch.float32).view(1, 1, W)
        dx = -xs - 0.25 - 1.5 * torch.rand(B, H, W, generator=g)
        dy = torch.randn(B, H, W, generator=g)
        return torch.stack([dx, dy], 1)
    raise ValueError(kind)


# (ks, dilation, C, flow): every value of each parameter appears
CASES = [(2, 1, 8, "smooth"), (4, 1, 64, "blocky"), (4, 2, 100, "border"), (6, 1, 512, "negx"), (6, 2, 8, "border"),
         (2, 2, 100, "negx"), (4, 1, 512, "smooth"), (8, 1, 64, "border")]
B, H, W, HI, WI = 2, 13, 35, 16, 40            # ragged 32 x 4 tiles; source larger than the flow grid


def _inputs(case, dtype, seed):
    ks, dil, C, kind = case
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, HI, WI, generator=g).to(dtype)
    tg = torch.randn(B, C, H, W, generator=g).to(dtype)
    sigma = 2.0 if ks >= 4 else 5.0
    in2 = torch.cat([_flow(kind, B, H, W, g), torch.full((B, 1, H, W), sigma)], 1).contiguous()
    go = torch.randn(B, C, H, W, generator=g).to(dtype)
    gcos = torch.randn(B, H, W, generator=g)
    return [t.to(DEV) for t in (x, in2, tg, go, gcos)]


def _fmt(t, cl):
    return t.contiguous(memory_format=torch.channels_last) if cl else t.contiguous()


@pytest.mark.parametrize("cl", [True, False], ids=["channels_last", "nchw"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("case", CASES, ids=[f"ks{c[0]}-dil{c[1]}-C{c[2]}-{c[3]}" for c in CASES])
def test_resample2d_16bit_vs_fp32_path(F_, case, dtype, cl):
    ks, dil, C, _ = case
    x, in2, _, go, _ = _inputs(case, dtype, seed=ks * 100 + dil * 10 + C)
    out = F_.resample2d_fwd(_fmt(x, cl), in2, ks, dil)
    assert out.dtype == dtype and out.shape == (B, C, H, W)
    assert out.is_contiguous(memory_format=torch.channels_last) if cl else out.is_contiguous()
    ref = F_.resample2d_fwd(x.float().contiguous(), in2, ks, dil)
    within_ulp(out, ref, scale=0.0)

    g1, g2 = F_.resample2d_bwd(_fmt(x, cl), in2, _fmt(go, cl), ks, dil)
    r1, r2 = F_.resample2d_bwd(x.float().contiguous(), in2, go.float().contiguous(), ks, dil)
    assert g1.dtype == dtype and g2.dtype == torch.float32
    assert g1.is_contiguous(memory_format=torch.channels_last) if cl else g1.is_contiguous()
    assert r1.abs().max().item() > 0
    within_ulp(g1, r1, rel=1e-5)
    s2 = r2.abs().max().item()
    assert (g2 - r2).abs().max().item() <= 1e-4 * s2


@pytest.mark.parametrize("cl", [True, False], ids=["channels_last", "nchw"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("case", CASES, ids=[f"ks{c[0]}-dil{c[1]}-C{c[2]}-{c[3]}" for c in CASES])
def test_resample2d_cosine_16bit_vs_fp32_path(F_, case, dtype, cl):
    ks, dil, C, _ = case
    x, in2, tg, _, gcos = _inputs(case, dtype, seed=ks * 100 + dil * 10 + C + 1)
    cos, stats = F_.resample2d_cosine_fwd(_fmt(x, cl), in2, _fmt(tg, cl), ks, dil, EPS)
    x32, tg32 = x.float().contiguous(), tg.float().contiguous()
    rcos, rstats = F_.resample2d_cosine_fwd(x32, in2, tg32, ks, dil, EPS)
    assert cos.dtype == stats.dtype == torch.float32
    assert (cos - rcos).abs().max().item() <= 1e-5 * max(1e-30, rcos.abs().max().item())
    assert (stats - rstats).abs().max().item() <= 1e-5 * rstats.abs().max().item()

    g1, g2, gt = F_.resample2d_cosine_bwd(_fmt(x, cl), in2, _fmt(tg, cl), stats, gcos, ks, dil, EPS, need_input1=True, need_target=True)
    r1, r2, rt = F_.resample2d_cosine_bwd(x32, in2, tg32, rstats, gcos, ks, dil, EPS, need_input1=True, need_target=True)
    assert g1.dtype == gt.dtype == dtype and g2.dtype == torch.float32
    for t in (g1, gt):
        assert t.is_contiguous(memory_format=torch.channels_last) if cl else t.is_contiguous()
    assert (g2 - r2).abs().max().item() <= 1e-4 * r2.abs().max().item()
    within_ulp(gt, rt, rel=1e-5)
    # grad_val (d/d warped) is stored in 16 bits before the scatter: bound by one relative ulp of the scattered magnitudes
    v32 = F_.resample2d_fwd(x32, in2, ks, dil)
    nv, nt = rstats[:, 1:2], rstats[:, 2:3]
    a, b = nv.clamp(min=EPS), nt.clamp(min=EPS)
    k1 = gcos.unsqueeze(1) / (a * b)
    k2v = torch.where(nv > EPS, gcos.unsqueeze(1) * rstats[:, 0:1] / (a * a * b * nv), torch.zeros_like(nv))
    gv_abs = (k1 * tg32 - k2v * v32).abs()
    s1 = F_.resample2d_bwd(x32, in2, gv_abs.contiguous(), ks, dil)[0]
    within_ulp(g1, r1, rel=1e-5, extra=2.0 ** -MANT[dtype] * s1)
    # the flow-only backward gives the same grad_input2
    n1, n2, n3 = F_.resample2d_cosine_bwd(_fmt(x, cl), in2, _fmt(tg, cl), stats, gcos, ks, dil, EPS)
    assert n1 is None and n3 is None and torch.equal(n2, g2)


@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "fp16"])
@pytest.mark.parametrize("cl", [True, False], ids=["channels_last", "nchw"])
def test_modules_through_autograd(dtype, cl):
    import gfla_b200
    g = torch.Generator().manual_seed(3)
    x = _fmt(torch.randn(2, 64, 24, 40, generator=g).to(dtype), cl).to(DEV).requires_grad_()
    tg = _fmt(torch.randn(2, 64, 20, 36, generator=g).to(dtype), cl).to(DEV).requires_grad_()
    flow = (torch.randn(2, 2, 20, 36, generator=g) * 3).to(dtype).to(DEV).requires_grad_()
    out = gfla_b200.Resample2d(4, 1, sigma=2)(x, flow)
    assert out.dtype == dtype and out.shape == (2, 64, 20, 36)
    assert out.is_contiguous(memory_format=torch.channels_last) if cl else out.is_contiguous()
    out.backward(torch.randn_like(out))
    assert x.grad.dtype == dtype and flow.grad.dtype == dtype
    assert x.grad.shape == x.shape and torch.isfinite(x.grad.float()).all() and torch.isfinite(flow.grad.float()).all()
    x.grad = flow.grad = None
    cos = gfla_b200.Resample2dCosine(4, 1, sigma=2)(x, flow, tg)
    assert cos.dtype == torch.float32 and cos.shape == (2, 20, 36)
    cos.sum().backward()
    assert x.grad.dtype == tg.grad.dtype == flow.grad.dtype == dtype
    for t in (x, tg):
        assert t.grad.is_contiguous(memory_format=torch.channels_last) if cl else t.grad.is_contiguous()
    # the same module with an fp32 source and a 16-bit flow: input2 is built in the source's dtype
    f2 = flow.detach().clone().requires_grad_()
    f3 = flow.detach().float().requires_grad_()
    xs = x.detach().float().contiguous()
    o2, o3 = gfla_b200.Resample2d(4, 1, sigma=2)(xs, f2), gfla_b200.Resample2d(4, 1, sigma=2)(xs, f3)
    assert o2.dtype == torch.float32 and torch.equal(o2, o3)
    o2.sum().backward()
    o3.sum().backward()
    assert f2.grad.dtype == dtype and torch.equal(f2.grad, f3.grad.to(dtype))


def _tf32_off():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    return old


def test_perceptual_correctness_fp32_features_bf16_flows():
    """fp32 VGG, bf16 generator flows (the INTEGRATION.md recipe before the VGG is cast): same loss and flow gradient as the
    call with flow.float()"""
    import gfla_b200
    from conftest import FixedFeatures, perceptual_inputs
    loss_fn = gfla_b200.PerceptualCorrectness(vgg=FixedFeatures()).to(DEV).eval()
    target, source, mask, flows = perceptual_inputs(DEV)
    old = _tf32_off()
    try:
        f16 = [f.bfloat16().requires_grad_() for f in flows]
        f32 = [f.bfloat16().float().requires_grad_() for f in flows]
        l16 = loss_fn(target, source, f16, [2, 3], mask)
        l32 = loss_fn(target, source, f32, [2, 3], mask)
        assert float(l16) == float(l32)
        l16.backward()
        l32.backward()
        for a, b in zip(f16, f32):
            assert a.grad.dtype == torch.bfloat16
            assert torch.equal(a.grad, b.grad.to(torch.bfloat16))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def test_perceptual_correctness_bf16_channels_last_features():
    """the whole recipe in bf16 channels_last: the loss within 1e-2 (relative) of the fp32 loss, flow gradients within 2e-2 of the
    largest magnitude.  The loss is mean(exp(-achieved / best)) - exp(-1), a small difference of two terms near exp(-1): its relative
    error is taken against the mean before the floor is subtracted, which is what the bf16 features perturb"""
    import gfla_b200
    from conftest import FixedFeatures, perceptual_inputs
    target, source, mask, flows = perceptual_inputs(DEV)
    old = _tf32_off()
    try:
        ref_fn = gfla_b200.PerceptualCorrectness(vgg=FixedFeatures()).to(DEV).eval()
        fr = [f.clone().requires_grad_() for f in flows]
        lr = ref_fn(target, source, fr, [2, 3], mask)
        lr.backward()
        fn = gfla_b200.PerceptualCorrectness(vgg=FixedFeatures().bfloat16()).to(DEV).eval()
        cl = torch.channels_last
        fb = [f.bfloat16().requires_grad_() for f in flows]
        lb = fn(target.bfloat16().contiguous(memory_format=cl), source.bfloat16().contiguous(memory_format=cl), fb, [2, 3],
                mask.bfloat16())
        assert abs(float(lb) - float(lr)) <= 1e-2 * (abs(float(lr)) + math.exp(-1.0))
        lb.backward()
        for a, b in zip(fb, fr):
            s = b.grad.abs().max().item()
            assert s > 0
            assert (a.grad.float() - b.grad).abs().max().item() <= 2e-2 * s
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def test_bf16_channels_last_launches_nhwc_kernels_only(F_):
    from torch.profiler import ProfilerActivity, profile
    g = torch.Generator().manual_seed(5)
    cl = torch.channels_last
    x = torch.randn(2, 128, 32, 48, generator=g).bfloat16().to(DEV).contiguous(memory_format=cl)
    tg = torch.randn(2, 128, 32, 48, generator=g).bfloat16().to(DEV).contiguous(memory_format=cl)
    in2 = torch.cat([torch.randn(2, 2, 32, 48, generator=g) * 3, torch.full((2, 1, 32, 48), 2.0)], 1).to(DEV)
    gcos = torch.randn(2, 32, 48, generator=g).to(DEV)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = F_.resample2d_fwd(x, in2, 4, 1)
        F_.resample2d_bwd(x, in2, out, 4, 1)
        cos, stats = F_.resample2d_cosine_fwd(x, in2, tg, 4, 1, EPS)
        F_.resample2d_cosine_bwd(x, in2, tg, stats, gcos, 4, 1, EPS)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    for k in ("k_resample2d_nhwc_fwd", "k_resample2d_nhwc_bwd_in1", "k_resample2d_nhwc_bwd_in2", "k_resample2d_nhwc_cos_fwd",
              "k_resample2d_nhwc_cos_bwd"):
        assert any(k in n for n in names), (k, names)
    planar = [n for n in names if "k_resample2d_" in n and "nhwc" not in n]
    moves = [n for n in names if any(s in n.lower() for s in ("transpose", "relayout", "copy", "contiguous"))]
    assert not planar and not moves, names
