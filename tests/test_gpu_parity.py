"""GPU (-m gpu): the CUDA library, called through the C ABI, against
  (1) the committed golden vectors (produced by the reference's own kernel bodies),
  (2) the CPU oracle on fresh seeded inputs,
  (3) size-independent properties at BASELINE.json's full sizes.
Tolerances (north_star): fp32 <= 1e-4, bf16 <= 1e-2; integer tap selection bit-identical,
which the fp32/fp64 forward of block_extractor / local_attn_reshape / resample2d shows by
being BIT-EXACT against the oracle (those kernels are built without FMA contraction)."""
import numpy as np
import pytest
import torch

from conftest import load_golden, sha256

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def cu(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def host(t):
    a = t.detach().float().cpu().numpy() if t.dtype in (torch.bfloat16, torch.float16) else t.detach().cpu().numpy()
    return np.ascontiguousarray(a)      # channels_last tensors come back with NHWC strides


@pytest.fixture(scope="module")
def F_():
    import gfla_b200
    from gfla_b200 import _lib
    _lib.check(_lib.lib().gfla_device_check(), "device check")
    return gfla_b200.functional


def tol(dt, f32, f64):
    return f32 if dt == np.float32 else f64


# ----------------------------------------------------------------------------- golden vectors
@pytest.mark.parametrize("case", sorted(load_golden("block_extractor")))
def test_block_extractor_golden(F_, case):
    g = load_golden("block_extractor")[case]
    k = int(g["k"])
    out = F_.block_extract_fwd(cu(g["source"]), cu(g["flow"]), k)
    assert sha256(host(out)) == str(g["out_sha256"]), "forward must be bit-exact (same taps, same arithmetic)"
    gs, gf = F_.block_extract_bwd(cu(g["source"]), cu(g["flow"]), cu(g["grad_out"]), k)
    t = tol(g["source"].dtype, 1e-5, 1e-12)
    np.testing.assert_allclose(host(gs), g["grad_source"], rtol=t, atol=t)
    np.testing.assert_allclose(host(gf), g["grad_flow"], rtol=10 * t, atol=10 * t * max(1.0, np.abs(g["grad_flow"]).max()))


@pytest.mark.parametrize("case", sorted(load_golden("local_attn_reshape")))
def test_local_attn_reshape_golden(F_, case):
    g = load_golden("local_attn_reshape")[case]
    k = int(g["k"])
    out = F_.attn_reshape_fwd(cu(g["in"]), k)
    assert np.array_equal(host(out), g["out"])
    if case == "layout":
        assert np.array_equal(host(out)[0, 0, :3, :3], np.arange(9, dtype=np.float32).reshape(3, 3))
    else:
        assert np.array_equal(host(F_.attn_reshape_bwd(cu(g["grad_out"]), k)), g["grad_in"])


@pytest.mark.parametrize("case", sorted(load_golden("resample2d")))
def test_resample2d_golden(F_, case):
    g = load_golden("resample2d")[case]
    ks, dil = int(g["ks"]), int(g["dil"])
    t = tol(g["in1"].dtype, 1e-6, 1e-14)     # exp() may differ in the last ulp between libm and CUDA
    out = F_.resample2d_fwd(cu(g["in1"]), cu(g["in2"]), ks, dil)
    np.testing.assert_allclose(host(out), g["out"], rtol=t, atol=t)
    g1, g2 = F_.resample2d_bwd(cu(g["in1"]), cu(g["in2"]), cu(g["grad_out"]), ks, dil)
    t = tol(g["in1"].dtype, 1e-5, 1e-12)
    np.testing.assert_allclose(host(g1), g["grad_in1"], rtol=t, atol=t)
    if case == "sigma0":
        # degenerate SAFE_DIV(., 0) branch: the reference divides 0-weights by 1e-8; only finiteness
        # and the forward are contractually meaningful here
        assert np.isfinite(host(g2)).all() == np.isfinite(g["grad_in2"]).all()
    else:
        scale = max(1.0, np.abs(g["grad_in2"]).max())
        np.testing.assert_allclose(host(g2), g["grad_in2"], rtol=1e-4 if g["in1"].dtype == np.float32 else 1e-10,
                                   atol=(1e-4 if g["in1"].dtype == np.float32 else 1e-10) * scale)


@pytest.mark.parametrize("algo", ["gather"])
@pytest.mark.parametrize("case", sorted(load_golden("local_attn")))
def test_local_attn_golden(F_, case, algo):
    g = load_golden("local_attn")[case]
    k = int(g["k"])
    t = tol(g["source"].dtype, 1e-5, 1e-12)
    s, f, l = cu(g["source"]), cu(g["flow"]), cu(g["logits"])
    out, probs = F_.local_attn_fwd(s, f, l, k, return_probs=True, algo=algo)
    np.testing.assert_allclose(host(probs), g["probs"], rtol=t, atol=t)
    np.testing.assert_allclose(host(out), g["out"], rtol=t, atol=t)
    gs, gf, gl = F_.local_attn_bwd(s, f, l, cu(g["grad_out"]), k)
    np.testing.assert_allclose(host(gs), g["grad_source"], rtol=10 * t, atol=10 * t)
    np.testing.assert_allclose(host(gf), g["grad_flow"], rtol=100 * t, atol=100 * t)
    np.testing.assert_allclose(host(gl), g["grad_logits"], rtol=100 * t, atol=10 * t)


# ----------------------------------------------------------------------------- vs the oracle, fresh inputs
def _flow(rng, kind, B, H, W):
    if kind == "iid":
        return rng.uniform(-8, 8, (B, 2, H, W))
    if kind == "border":
        return rng.uniform(-1.5 * W, 1.5 * W, (B, 2, H, W))
    if kind == "zero":
        return np.zeros((B, 2, H, W))
    if kind == "int":      # exactly integral displacements: frac == 0 everywhere
        return rng.integers(-3, 4, (B, 2, H, W)).astype(np.float64)
    coarse = torch.from_numpy(rng.uniform(-8, 8, (B, 2, max(H // 8, 2), max(W // 8, 2))))
    return torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True).numpy()


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 7])
@pytest.mark.parametrize("kind", ["iid", "border", "smooth", "int"])
def test_block_extractor_vs_oracle(F_, oracle_lib, dt, k, kind):
    rng = np.random.default_rng(k * 100 + len(kind))
    B, C, Hs, Ws, H, W = 2, 5, 19, 23, 17, 21
    s = rng.standard_normal((B, C, Hs, Ws)).astype(dt)
    f = _flow(rng, kind, B, H, W).astype(dt)
    out = F_.block_extract_fwd(cu(s), cu(f), k)
    assert np.array_equal(host(out), oracle_lib.block_extract_fwd(s, f, k))
    g = rng.standard_normal(out.shape).astype(dt)
    gs, gf = F_.block_extract_bwd(cu(s), cu(f), cu(g), k)
    ogs, ogf = oracle_lib.block_extract_bwd(s, f, g, k)
    t = tol(dt, 2e-5, 1e-12)   # float atomics: summation order differs; scale by the largest accumulated sum
    np.testing.assert_allclose(host(gs), ogs, rtol=t, atol=t * max(1.0, np.abs(ogs).max()))
    np.testing.assert_allclose(host(gf), ogf, rtol=t, atol=t * max(1.0, np.abs(ogf).max()))


def test_block_extractor_accumulate_contract(F_, oracle_lib):
    """legacy contract: backward ADDS into the caller's buffers (block_extractor.py:35-40)"""
    rng = np.random.default_rng(5)
    s = rng.standard_normal((1, 3, 9, 9)).astype(np.float32)
    f = rng.uniform(-3, 3, (1, 2, 9, 9)).astype(np.float32)
    g = rng.standard_normal((1, 3, 27, 27)).astype(np.float32)
    gs0, gf0 = torch.full((1, 3, 9, 9), 2.0, device=DEV), torch.full((1, 2, 9, 9), -1.0, device=DEV)
    F_.block_extract_bwd(cu(s), cu(f), cu(g), 3, gs0, gf0)
    ogs, ogf = oracle_lib.block_extract_bwd(s, f, g, 3)
    np.testing.assert_allclose(host(gs0), ogs + 2.0, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(host(gf0), ogf - 1.0, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("cfg", [(2, 1, 5.0), (4, 1, 2.0), (4, 2, 2.0), (6, 1, 3.0), (8, 1, 2.5)])
def test_resample2d_vs_oracle(F_, oracle_lib, dt, cfg):
    ks, dil, sigma = cfg
    rng = np.random.default_rng(ks * 10 + dil)
    B, C, Hi, Wi, H, W = 2, 6, 15, 18, 13, 16
    a = rng.standard_normal((B, C, Hi, Wi)).astype(dt)
    in2 = np.concatenate([rng.uniform(-6, 6, (B, 2, H, W)), np.full((B, 1, H, W), sigma)], 1).astype(dt)
    out = F_.resample2d_fwd(cu(a), cu(in2), ks, dil)
    t = tol(dt, 1e-6, 1e-14)
    np.testing.assert_allclose(host(out), oracle_lib.resample2d_fwd(a, in2, ks, dil), rtol=t, atol=t)
    g = rng.standard_normal(out.shape).astype(dt)
    g1, g2 = F_.resample2d_bwd(cu(a), cu(in2), cu(g), ks, dil)
    o1, o2 = oracle_lib.resample2d_bwd(a, in2, g, ks, dil)
    t = tol(dt, 1e-5, 1e-12)
    np.testing.assert_allclose(host(g1), o1, rtol=t, atol=t)
    t = tol(dt, 1e-4, 1e-10)
    np.testing.assert_allclose(host(g2), o2, rtol=t, atol=t * max(1.0, np.abs(o2).max()))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("kind", ["iid", "border", "smooth", "int", "zero"])
def test_local_attn_vs_oracle(F_, oracle_lib, dt, k, kind):
    rng = np.random.default_rng(k * 7 + len(kind))
    B, C, H, W = 2, 6, 14, 17
    s = rng.standard_normal((B, C, H, W)).astype(dt)
    f = _flow(rng, kind, B, H, W).astype(dt)
    l = (2 * rng.standard_normal((B, k * k, H, W))).astype(dt)
    t = tol(dt, 1e-5, 1e-12)
    out = F_.local_attn_fwd(cu(s), cu(f), cu(l), k, algo="gather")
    np.testing.assert_allclose(host(out), oracle_lib.local_attn_fwd(s, f, l, k), rtol=t, atol=t)
    g = rng.standard_normal(out.shape).astype(dt)
    gs, gf, gl = F_.local_attn_bwd(cu(s), cu(f), cu(l), cu(g), k)
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(s, f, l, g, k)
    np.testing.assert_allclose(host(gs), ogs, rtol=10 * t, atol=10 * t)
    np.testing.assert_allclose(host(gf), ogf, rtol=100 * t, atol=100 * t)
    np.testing.assert_allclose(host(gl), ogl, rtol=100 * t, atol=10 * t)


@pytest.mark.parametrize("flow_dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("k", [3, 5])
def test_local_attn_bf16_vs_oracle(F_, oracle_lib, k, flow_dt):
    """bf16 storage: oracle = the fp32 reference arithmetic on the bf16-rounded inputs, tolerance 1e-2"""
    torch.manual_seed(k)
    B, C, H, W = 2, 32, 24, 20
    s = torch.randn(B, C, H, W, device=DEV).bfloat16()
    f = ((torch.rand(B, 2, H, W, device=DEV) * 12) - 6).to(flow_dt)
    l = torch.randn(B, k * k, H, W, device=DEV).bfloat16()
    out = F_.local_attn_fwd(s, f, l, k, algo="gather")
    ref = oracle_lib.local_attn_fwd(host(s), host(f) if flow_dt != torch.float32 else f.cpu().numpy(), host(l), k)
    np.testing.assert_allclose(host(out), ref, rtol=0, atol=1e-2)
    g = torch.randn_like(out)
    gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k)
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), host(f) if flow_dt != torch.float32 else f.cpu().numpy(),
                                              host(l), host(g), k)
    np.testing.assert_allclose(host(gs), ogs, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gl), ogl, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gf), ogf, rtol=2e-2, atol=2e-2 * np.abs(ogf).max())


# ----------------------------------------------------------------------------- autograd surface (reference tests)
def test_gradcheck_block_extractor_double():
    """model/networks/block_extractor/test_block_extractor.py:74-78"""
    import gfla_b200
    torch.manual_seed(0)
    extractor = gfla_b200.BlockExtractor(3)
    source = torch.rand(4, 6, 14, 10, dtype=torch.float64, device=DEV, requires_grad=True)
    flow = (torch.rand(4, 2, 14, 10, dtype=torch.float64, device=DEV) * 1.8).requires_grad_()
    assert torch.autograd.gradcheck(extractor, (source, flow), nondet_tol=1e-10)


def test_gradcheck_local_attn_reshape_double():
    """model/networks/local_attn_reshape/test_local_attn_reshape.py:66-70 (k = 3)"""
    import gfla_b200
    torch.manual_seed(0)
    m = gfla_b200.LocalAttnReshape()
    source = torch.rand(4, 9, 14, 10, dtype=torch.float64, device=DEV, requires_grad=True)
    assert torch.autograd.gradcheck(lambda t: m(t, 3), (source,))


def test_gradcheck_local_attention_double():
    import gfla_b200
    torch.manual_seed(1)
    s = torch.rand(2, 3, 7, 6, dtype=torch.float64, device=DEV, requires_grad=True)
    f = (torch.rand(2, 2, 7, 6, dtype=torch.float64, device=DEV) * 3.3 - 1.4).requires_grad_()
    l = torch.randn(2, 9, 7, 6, dtype=torch.float64, device=DEV, requires_grad=True)
    assert torch.autograd.gradcheck(lambda a, b, c: gfla_b200.local_attention(a, b, c, 3), (s, f, l), nondet_tol=1e-10)


def test_resample2d_module_autograd(oracle_lib):
    import gfla_b200
    torch.manual_seed(2)
    m = gfla_b200.Resample2d(4, 1, sigma=2)          # what PerceptualCorrectness uses, external_function.py:233
    x = torch.randn(2, 5, 12, 12, device=DEV, requires_grad=True)
    flow = (torch.rand(2, 2, 12, 12, device=DEV) * 4 - 2).requires_grad_()
    out = m(x, flow)
    g = torch.randn_like(out)
    out.backward(g)
    in2 = np.concatenate([host(flow), np.full((2, 1, 12, 12), 2.0, np.float32)], 1)
    np.testing.assert_allclose(host(out), oracle_lib.resample2d_fwd(host(x), in2, 4, 1), rtol=1e-6, atol=1e-6)
    o1, o2 = oracle_lib.resample2d_bwd(host(x), in2, host(g), 4, 1)
    np.testing.assert_allclose(host(x.grad), o1, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(host(flow.grad), o2[:, :2], rtol=1e-4, atol=1e-4)   # sigma plane is dropped by cat


def test_extractor_attn_module_matches_literal_composition():
    """our ExtractorAttn (fused tail) == the reference's literal op sequence (base_function.py:804-810)
    built from our own unfused ops + torch, same weights; forward, hook and all gradients."""
    import gfla_b200
    torch.manual_seed(3)
    C, k, B, H, W = 8, 3, 2, 12, 10
    m = gfla_b200.ExtractorAttn(C, k, softmax=True).to(DEV)
    src = torch.randn(B, C, H, W, device=DEV, requires_grad=True)
    tgt = torch.randn(B, C, H, W, device=DEV, requires_grad=True)
    flow = (torch.rand(B, 2, H, W, device=DEV) * 6 - 3).requires_grad_()
    out = m(src, tgt, flow)
    g = torch.randn_like(out)
    grads = torch.autograd.grad(out, (src, tgt, flow) + tuple(m.parameters()), g)

    ex, rs = gfla_b200.BlockExtractor(k), gfla_b200.LocalAttnReshape()
    bs = ex(src, flow)
    bt = ex(tgt, torch.zeros_like(flow))
    attn = m.fully_connect_layer(torch.cat((bt, bs), 1))            # includes the Softmax
    ref = torch.nn.functional.avg_pool2d(rs(attn, k) * bs, k, k)
    rgrads = torch.autograd.grad(ref, (src, tgt, flow) + tuple(m.parameters()), g)
    np.testing.assert_allclose(host(out), host(ref), rtol=1e-5, atol=1e-5)
    for a, b in zip(grads, rgrads):
        np.testing.assert_allclose(host(a), host(b), rtol=2e-4, atol=2e-4 * max(1.0, float(b.abs().max())))
    p, res = m.hook_attn_param(src, tgt, flow)
    np.testing.assert_allclose(host(p), host(attn), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(host(res), host(ref), rtol=1e-5, atol=1e-5)


def test_legacy_pybind_surface(oracle_lib):
    """the reference's own wrapper logic (block_extractor.py:21-26: zero-filled output, then
    `block_extractor_cuda.forward`) runs on the shim modules"""
    import gfla_b200
    gfla_b200.compat.install()
    import block_extractor_cuda, local_attn_reshape_cuda, resample2d_cuda  # noqa: E401
    rng = np.random.default_rng(11)
    s = rng.standard_normal((1, 4, 10, 10)).astype(np.float32)
    f = rng.uniform(-4, 4, (1, 2, 10, 10)).astype(np.float32)
    ts, tf = cu(s), cu(f)
    out = tf.new(1, 4, 30, 30).zero_()
    assert block_extractor_cuda.forward(ts, tf, out, 3) == 1
    assert np.array_equal(host(out), oracle_lib.block_extract_fwd(s, f, 3))
    go = torch.randn_like(out)
    gs, gf = ts.new(ts.size()).zero_(), tf.new(tf.size()).zero_()
    assert block_extractor_cuda.backward(ts, tf, go, gs, gf, 3) == 1
    ogs, ogf = oracle_lib.block_extract_bwd(s, f, host(go), 3)
    np.testing.assert_allclose(host(gs), ogs, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(host(gf), ogf, rtol=1e-4, atol=1e-4)
    x = torch.randn(1, 9, 5, 5, device=DEV)
    o = x.new(1, 1, 15, 15).zero_()
    assert local_attn_reshape_cuda.forward(x, o, 3) == 1
    assert np.array_equal(host(o), oracle_lib.attn_reshape_fwd(host(x), 3))
    in2 = torch.cat([tf, torch.full((1, 1, 10, 10), 5.0, device=DEV)], 1)
    o2 = ts.new(1, 4, 10, 10).zero_()
    assert resample2d_cuda.forward(ts, in2, o2, 2, 1) == 1
    np.testing.assert_allclose(host(o2), oracle_lib.resample2d_fwd(s, host(in2), 2, 1), rtol=1e-6, atol=1e-6)


# ----------------------------------------------------------------------------- full-size properties (BASELINE cfg2 / cfg3)
def _smooth_flow_t(B, H, W, amp=8.0, cell=16):
    coarse = (torch.rand(B, 2, H // cell, W // cell, device=DEV) * 2 - 1) * amp
    return torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True).contiguous()


@pytest.mark.parametrize("algo", ["gather"])
def test_cfg2_fused_equals_unfused_composition(F_, algo):
    """B=2 slice of cfg2 (C=256, 256x256, k=5, bf16 data, fp32 flow): the fused kernel equals the
    literal extractor -> softmax -> reshape -> mul -> avg_pool chain built from the (oracle-checked)
    unfused kernels.  (The reference cannot run this shape at B=16 in one call: int overflow.)"""
    torch.manual_seed(0)
    B, C, H, W, k = 2, 256, 256, 256, 5
    s = torch.randn(B, C, H, W, device=DEV).bfloat16()
    f = _smooth_flow_t(B, H, W)
    l = torch.randn(B, k * k, H, W, device=DEV).bfloat16()
    out = F_.local_attn_fwd(s, f, l, k, algo=algo).float()
    ref = torch.empty_like(out)
    for b in range(B):      # block tensor of one sample: 256*1280*1280*4 B = 1.7 GB in fp32
        blk = F_.block_extract_fwd(s[b:b + 1].float().contiguous(), f[b:b + 1].contiguous(), k)
        attn = F_.attn_reshape_fwd(torch.softmax(l[b:b + 1].float(), 1).contiguous(), k)
        ref[b:b + 1] = torch.nn.functional.avg_pool2d(attn * blk, k, k)
        del blk, attn
    err = (out - ref).abs().max().item()
    assert err <= 1e-2, err
    # property: one-hot attention at the centre tap with zero flow reproduces source / k^2
    l1 = torch.full((1, k * k, H, W), -30000.0, device=DEV)
    l1[:, (k * k) // 2] = 0
    o1 = F_.local_attn_fwd(s[:1].contiguous(), torch.zeros(1, 2, H, W, device=DEV), l1.bfloat16(), k, algo=algo)
    np.testing.assert_allclose(host(o1), host(s[:1]) / (k * k), rtol=0, atol=4e-3)


def test_cfg2_linearity_in_source(F_):
    """out is linear in source for fixed (flow, logits): f(a*s1 + s2) == a*f(s1) + f(s2) (fp32, full 256x256)"""
    torch.manual_seed(1)
    B, C, H, W, k = 1, 64, 256, 256, 5
    s1, s2 = torch.randn(B, C, H, W, device=DEV), torch.randn(B, C, H, W, device=DEV)
    f = (torch.rand(B, 2, H, W, device=DEV) * 16 - 8)
    l = torch.randn(B, k * k, H, W, device=DEV)
    o12 = F_.local_attn_fwd(0.5 * s1 + s2, f, l, k)
    o = 0.5 * F_.local_attn_fwd(s1, f, l, k) + F_.local_attn_fwd(s2, f, l, k)
    assert (o12 - o).abs().max().item() < 1e-5


def test_cfg3_resample2d_properties(F_):
    """cfg3-sized planes (512x512), reduced batch: (a) a constant image resamples to the same constant
    for any flow (weights are normalised), (b) adjointness <resample(x), g> == <x, grad_in1(g)>."""
    torch.manual_seed(2)
    B, C, H, W = 2, 16, 512, 512
    flow = torch.rand(B, 2, H, W, device=DEV) * 16 - 8
    for ks, sigma in ((2, 5.0), (4, 2.0)):
        in2 = torch.cat([flow, torch.full((B, 1, H, W), sigma, device=DEV)], 1).contiguous()
        const = torch.full((B, C, H, W), 3.25, device=DEV)
        out = F_.resample2d_fwd(const, in2, ks, 1)
        assert (out - 3.25).abs().max().item() < 1e-5
        x = torch.randn(B, C, H, W, device=DEV)
        g = torch.randn(B, C, H, W, device=DEV)
        # forward weights use floor(), grad_input1 uses int() for the fraction (reference quirk): restrict the
        # adjoint identity to non-negative sample coordinates where the two agree
        pos_flow = flow.abs()
        in2p = torch.cat([pos_flow, torch.full((B, 1, H, W), sigma, device=DEV)], 1).contiguous()
        y = F_.resample2d_fwd(x, in2p, ks, 1)
        g1, _ = F_.resample2d_bwd(x, in2p, g, ks, 1)
        lhs, rhs = (y.double() * g.double()).sum().item(), (x.double() * g1.double()).sum().item()
        assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), 1.0) + 1.0, (lhs, rhs)


def test_large_index_no_int_overflow(F_):
    """output numel > 2^31 (the reference's `int n` overflows, block_extractor_kernel.cu:33,180):
    B=1, C=64 bf16, 1024x1024 flow, k=6 -> 2.4e9 elements; spot-check against the small-shape kernel."""
    torch.manual_seed(3)
    C, H, W, k = 64, 1024, 1024, 6
    s = torch.randn(1, C, H, W, device=DEV).bfloat16()
    f = torch.rand(1, 2, H, W, device=DEV) * 8 - 4
    out = F_.block_extract_fwd(s, f, k)
    assert out.numel() > 2**31
    # the last channel / bottom-right corner lives beyond the 2^31 boundary
    y0, x0 = H - 16, W - 16
    sub = F_.block_extract_fwd(s[:, -1:, :, :].contiguous(), f, k)
    assert torch.equal(out[0, -1, y0 * k:, x0 * k:], sub[0, 0, y0 * k:, x0 * k:])


# ----------------------------------------------------------------------------- tcgen05 tile kernel (bf16 forward)
def _tile_inputs(B, C, Hs, Ws, H, W, k, kind, seed):
    rng = np.random.default_rng(seed)
    s = torch.from_numpy(rng.standard_normal((B, C, Hs, Ws)).astype(np.float32)).to(DEV).bfloat16()
    f = torch.from_numpy(_flow(rng, kind, B, H, W).astype(np.float32)).to(DEV)
    l = torch.from_numpy((2 * rng.standard_normal((B, k * k, H, W))).astype(np.float32)).to(DEV).bfloat16()
    return s, f, l


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
@pytest.mark.parametrize("kind", ["smooth", "iid", "border", "zero", "int"])
@pytest.mark.parametrize("shape", [
    (2, 64, 32, 32, 32, 32, 5),      # aligned
    (1, 128, 40, 24, 40, 24, 3),     # k = 3, CN = 128
    (2, 64, 21, 40, 21, 40, 5),      # ragged: H, W not multiples of the 16x8 pixel group
    (1, 256, 16, 16, 16, 16, 5),     # CN = 256 (512 TMEM columns)
    (1, 64, 24, 32, 19, 27, 3),      # source larger than the flow field (external_function.py:61-66 usage)
    (1, 512, 16, 24, 16, 24, 5),     # two channel chunks of 256
])
def test_local_attn_tile_vs_oracle(F_, oracle_lib, shape, kind, layout):
    B, C, Hs, Ws, H, W, k = shape
    s, f, l = _tile_inputs(B, C, Hs, Ws, H, W, k, kind, seed=sum(shape) + len(kind))
    if layout == "nhwc":             # channels_last storage: same logical tensor, the tile kernel's fast layout
        s = s.contiguous(memory_format=torch.channels_last)
    out, probs = F_.local_attn_fwd(s, f, l, k, return_probs=True, algo="tile")
    assert out.is_contiguous(memory_format=torch.channels_last if layout == "nhwc" else torch.contiguous_format)
    ref, rprobs = oracle_lib.local_attn_fwd(host(s), f.cpu().numpy(), host(l), k, return_probs=True)
    np.testing.assert_allclose(host(probs), rprobs, rtol=0, atol=4e-3)
    np.testing.assert_allclose(host(out), ref, rtol=0, atol=1e-2)            # north_star tolerance
    # and much tighter than the contract against our own fp32-accumulating gather kernel:
    # the only extra error is the bf16 rounding of the collapsed weights (2^-9 relative)
    g = F_.local_attn_fwd(s, f, l, k, algo="gather")
    err = (out.float() - g.float()).abs().max().item()
    assert err <= 3e-3, err


def test_local_attn_tile_rejects_what_it_cannot_serve(F_):
    from gfla_b200 import _lib
    s = torch.randn(1, 64, 16, 16, device=DEV)            # fp32: no tile kernel
    f = torch.zeros(1, 2, 16, 16, device=DEV)
    l = torch.randn(1, 25, 16, 16, device=DEV)
    with pytest.raises(_lib.GflaError):
        F_.local_attn_fwd(s, f, l, 5, algo="tile")
    F_.local_attn_fwd(s, f, l, 5, algo="auto")             # auto falls back to the gather kernel


def test_cfg2_tile_equals_unfused_composition(F_):
    test_cfg2_fused_equals_unfused_composition(F_, "tile")


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
def test_local_attn_channels_last_gather_and_backward(F_, oracle_lib, dt):
    """channels_last tensors through the CUDA-core kernels (forward and backward), any dtype"""
    torch.manual_seed(5)
    B, C, H, W, k = 2, 16, 13, 11, 3
    s = torch.randn(B, C, H, W, device=DEV).to(dt).contiguous(memory_format=torch.channels_last)
    f = torch.rand(B, 2, H, W, device=DEV) * 8 - 4
    l = torch.randn(B, k * k, H, W, device=DEV).to(dt)
    g = torch.randn(B, C, H, W, device=DEV).to(dt).contiguous(memory_format=torch.channels_last)
    out = F_.local_attn_fwd(s, f if dt == torch.float32 else f, l, k, algo="gather")
    gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k)
    assert gs.is_contiguous(memory_format=torch.channels_last)
    tol_ = 1e-5 if dt == torch.float32 else 1e-2
    ref = oracle_lib.local_attn_fwd(host(s), host(f), host(l), k)
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), host(f), host(l), host(g), k)
    np.testing.assert_allclose(host(out), ref, rtol=tol_, atol=tol_)
    np.testing.assert_allclose(host(gs), ogs, rtol=10 * tol_, atol=10 * tol_)
    np.testing.assert_allclose(host(gl), ogl, rtol=10 * tol_, atol=10 * tol_)
    np.testing.assert_allclose(host(gf), ogf, rtol=20 * tol_, atol=20 * tol_ * max(1.0, np.abs(ogf).max()))


def _irregular_flow_values(xs, k, rng):
    """flows f (for pixel column x) for which the reference's fp32 tap arithmetic
    floor((f + (j - k//2)) + x) is NOT consecutive in j: the rounding of the two additions straddles an
    integer for some taps only (block_extractor_kernel.cu:62-69).  The kernels must follow it bit for bit."""
    out = {}
    for x in xs:
        for n in (-3, 0, 2, 5):
            for _ in range(4000):
                f = np.float32(np.float32(n) + np.float32(rng.uniform(-4e-6, 4e-6)))
                fl = [int(np.floor(np.float32(np.float32(f + np.float32(j - k // 2)) + np.float32(x)))) for j in range(k)]
                if any(fl[j] != fl[0] + j for j in range(k)):
                    out[x] = float(f)
                    break
            if x in out:
                break
    return out


@pytest.mark.parametrize("layout", ["nchw", "nhwc"])
def test_local_attn_tile_irregular_taps(F_, oracle_lib, layout):
    """pixels whose taps are not consecutive integers take the literal 4-tap path inside the tile kernel
    (warp-cooperative): results still match the oracle, i.e. the reference's tap selection is kept."""
    rng = np.random.default_rng(42)
    B, C, H, W, k = 1, 64, 24, 64, 5
    vals = _irregular_flow_values(range(3, W - 3, 2), k, rng)
    assert len(vals) >= 10
    flow = rng.uniform(-3, 3, (B, 2, H, W)).astype(np.float32)
    n_irr = 0
    for i, (x, f) in enumerate(vals.items()):
        y = (5 * i) % H
        flow[0, 0, y, x] = f                       # irregular along x
        flow[0, 1, (y + 3) % H, x] = np.float32(_irregular_flow_values([(y + 3) % H], k, rng).get((y + 3) % H, 0.25))
        n_irr += 1
    s = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16()
    if layout == "nhwc":
        s = s.contiguous(memory_format=torch.channels_last)
    f = torch.from_numpy(flow).to(DEV)
    l = torch.from_numpy(rng.standard_normal((B, k * k, H, W)).astype(np.float32)).to(DEV).bfloat16()
    out = F_.local_attn_fwd(s, f, l, k, algo="tile")
    ref = oracle_lib.local_attn_fwd(host(s), flow, host(l), k)
    np.testing.assert_allclose(host(out), ref, rtol=0, atol=1e-2)
    g = F_.local_attn_fwd(s, f, l, k, algo="gather")
    assert (out.float() - g.float()).abs().max().item() <= 3e-3


# ----------------------------------------------------------------------------- tile backward (grad_source GEMM + TMA reduce-add)
@pytest.mark.parametrize("kind", ["smooth", "iid", "border", "zero"])
@pytest.mark.parametrize("shape", [
    (1, 64, 32, 32, 32, 32, 5),
    (2, 256, 24, 40, 24, 40, 5),
    (1, 128, 21, 27, 21, 27, 3),      # ragged groups, odd width
    (1, 64, 24, 32, 19, 27, 3),       # source larger than the flow field
    (1, 512, 16, 24, 16, 24, 5),      # two channel chunks
])
def test_local_attn_bwd_tile_vs_oracle(F_, oracle_lib, shape, kind):
    B, C, Hs, Ws, H, W, k = shape
    s, f, l = _tile_inputs(B, C, Hs, Ws, H, W, k, kind, seed=3 * sum(shape) + len(kind))
    s = s.contiguous(memory_format=torch.channels_last)
    rng = np.random.default_rng(7)
    g = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16()
    g = g.contiguous(memory_format=torch.channels_last)
    gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k, algo="tile")
    assert gs.is_contiguous(memory_format=torch.channels_last)
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), f.cpu().numpy(), host(l), host(g), k)
    scale = max(1.0, float(np.abs(ogs).max()))
    # north_star's flat 1e-2 wherever bf16 can hold it: one bf16 ulp at magnitude M is M * 2^-8, so above |g| = 2.56
    # (border flows pile hundreds of pixels onto one edge position) the bound scales with the largest gradient
    np.testing.assert_allclose(host(gs), ogs, rtol=0, atol=1e-2 * scale)
    np.testing.assert_allclose(host(gl), ogl, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gf), ogf, rtol=2e-2, atol=2e-2 * max(1.0, float(np.abs(ogf).max())))


@pytest.mark.parametrize("shape", [(6, 64, 16, 16, 3), (8, 128, 32, 32, 5), (9, 64, 8, 40, 3)])
def test_local_attn_bwd_tile_many_samples_few_groups(F_, oracle_lib, shape):
    """More samples than a CTA ever visits (one or two groups per CTA, B > 3): every CTA still has to zero-fill its slice of ALL
    samples of grad_source, also those it never computes on (in-kernel zero fill of the fused backward; the generator's
    32x32 / 64x64 attention levels at batch 8 are this case)."""
    B, C, H, W, k = shape
    s, f, l = _tile_inputs(B, C, H, W, H, W, k, "smooth", seed=sum(shape))
    s = s.contiguous(memory_format=torch.channels_last)
    rng = np.random.default_rng(11)
    g = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16().contiguous(memory_format=torch.channels_last)
    for _ in range(2):     # second call: the workspace comes back dirty from the allocator
        gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k, algo="tile")
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), f.cpu().numpy(), host(l), host(g), k)
    np.testing.assert_allclose(host(gs), ogs, rtol=0, atol=1e-2 * max(1.0, float(np.abs(ogs).max())))
    np.testing.assert_allclose(host(gl), ogl, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gf), ogf, rtol=2e-2, atol=2e-2 * max(1.0, float(np.abs(ogf).max())))


def test_local_attn_bwd_cooperative_launch_refused_falls_back(F_, oracle_lib, monkeypatch):
    """GFLA_BWD_COOP=2 makes the library behave as if the driver had refused the cooperative launch of the fused backward (an MPS
    client with a reduced SM share): it must zero grad_source with a memset and run the kernel with independent CTAs -- same results."""
    monkeypatch.setenv("GFLA_BWD_COOP", "2")
    B, C, H, W, k = 5, 128, 24, 40, 5
    s, f, l = _tile_inputs(B, C, H, W, H, W, k, "smooth", seed=77)
    s = s.contiguous(memory_format=torch.channels_last)
    rng = np.random.default_rng(5)
    g = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16().contiguous(memory_format=torch.channels_last)
    gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k, algo="tile")
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), f.cpu().numpy(), host(l), host(g), k)
    np.testing.assert_allclose(host(gs), ogs, rtol=0, atol=1e-2 * max(1.0, float(np.abs(ogs).max())))
    np.testing.assert_allclose(host(gl), ogl, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gf), ogf, rtol=2e-2, atol=2e-2 * max(1.0, float(np.abs(ogf).max())))


def test_local_attn_bwd_tile_irregular_taps(F_, oracle_lib):
    rng = np.random.default_rng(43)
    B, C, H, W, k = 1, 64, 24, 64, 5
    vals = _irregular_flow_values(range(3, W - 3, 2), k, rng)
    flow = rng.uniform(-3, 3, (B, 2, H, W)).astype(np.float32)
    for i, (x, fv) in enumerate(vals.items()):
        flow[0, 0, (5 * i) % H, x] = fv
    s = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16().contiguous(memory_format=torch.channels_last)
    g = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16().contiguous(memory_format=torch.channels_last)
    l = torch.from_numpy(rng.standard_normal((B, k * k, H, W)).astype(np.float32)).to(DEV).bfloat16()
    gs, gf, gl = F_.local_attn_bwd(s, torch.from_numpy(flow).to(DEV), l, g, k, algo="tile")
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), flow, host(l), host(g), k)
    np.testing.assert_allclose(host(gs), ogs, rtol=0, atol=1e-2)
    # the irregular pixels' grad_flow / grad_logits come from the literal 4-tap path of the same kernel
    np.testing.assert_allclose(host(gl), ogl, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gf), ogf, rtol=2e-2, atol=2e-2 * max(1.0, float(np.abs(ogf).max())))


def test_local_attn_bwd_nchw_bf16_routes_through_tile_kernels(F_, oracle_lib):
    """planar (NCHW) bf16 callers: 'auto' re-lays the feature tensors and uses the tile kernels; results come
    back contiguous NCHW and match the oracle like the channels_last path"""
    B, C, H, W, k = 1, 64, 24, 32, 5
    s, f, l = _tile_inputs(B, C, H, W, H, W, k, "smooth", seed=99)
    g = torch.randn(B, C, H, W, device=DEV).bfloat16()
    gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k)
    assert gs.is_contiguous()
    ogs, ogf, ogl = oracle_lib.local_attn_bwd(host(s), f.cpu().numpy(), host(l), host(g), k)
    np.testing.assert_allclose(host(gs), ogs, rtol=0, atol=1e-2 * max(1.0, float(np.abs(ogs).max())))
    np.testing.assert_allclose(host(gl), ogl, rtol=0, atol=1e-2)
    np.testing.assert_allclose(host(gf), ogf, rtol=2e-2, atol=2e-2 * max(1.0, float(np.abs(ogf).max())))


def test_cfg2_backward_tile_equals_cuda_core_backward(F_):
    """one full-size cfg2 sample (C=256, 256x256, k=5, bf16 channels_last): the three tensor-core backward
    kernels agree with the (oracle-checked) CUDA-core backward; also exercises > 50 groups per CTA."""
    torch.manual_seed(4)
    B, C, H, W, k = 1, 256, 256, 256, 5
    cl = torch.channels_last
    s = torch.randn(B, C, H, W, device=DEV).bfloat16().contiguous(memory_format=cl)
    g = torch.randn(B, C, H, W, device=DEV).bfloat16().contiguous(memory_format=cl)
    f = _smooth_flow_t(B, H, W)
    l = torch.randn(B, k * k, H, W, device=DEV).bfloat16()
    gs, gf, gl = F_.local_attn_bwd(s, f, l, g, k, algo="tile")
    # reference: fp32 CUDA-core kernels on the same (bf16-rounded) values: fp32 atomics, fp32 accumulation
    rs, rf, rl = F_.local_attn_bwd(s.float().contiguous(), f, l.float(), g.float().contiguous(), k, algo="gather")
    assert (gs.float() - rs).abs().max().item() <= 1e-2 * max(1.0, rs.abs().max().item())
    assert (gl.float() - rl).abs().max().item() <= 1e-2
    assert (gf - rf).abs().max().item() <= 2e-2 * max(1.0, rf.abs().max().item())


def test_tile_kernels_many_groups_small_grid(F_, oracle_lib):
    """more pixel groups per CTA than the info ring has slots, ragged last group: B=3, 40x72 (C=64)"""
    B, C, H, W, k = 3, 64, 40, 72, 3
    s, f, l = _tile_inputs(B, C, H, W, H, W, k, "smooth", seed=5)
    s = s.contiguous(memory_format=torch.channels_last)
    out = F_.local_attn_fwd(s, f, l, k, algo="tile")
    ref = oracle_lib.local_attn_fwd(host(s), f.cpu().numpy(), host(l), k)
    np.testing.assert_allclose(host(out), ref, rtol=0, atol=1e-2)


@pytest.mark.parametrize("ts", [0, 1, 3, 16])
@pytest.mark.parametrize("kind", ["smooth", "iid", "border"])
def test_local_attn_strip_schedule_long_columns(F_, oracle_lib, monkeypatch, kind, ts):
    """channels-last strip kernel: tall image (33 tile rows), more strips than SMs, every strip length incl. 1 (no row
    sharing) and longer-than-the-image; the per-tile kernel (GFLA_TC_STRIP=-1) must give the same result to rounding"""
    B, C, H, W, k = 4, 64, 264, 160, 5
    s, f, l = _tile_inputs(B, C, H, W, H, W, k, kind, seed=11 + ts)
    s = s.contiguous(memory_format=torch.channels_last)
    monkeypatch.setenv("GFLA_TC_STRIP", str(ts))
    out, probs = F_.local_attn_fwd(s, f, l, k, return_probs=True, algo="tile")
    monkeypatch.setenv("GFLA_TC_STRIP", "-1")
    per_tile = F_.local_attn_fwd(s, f, l, k, algo="tile")
    assert (out.float() - per_tile.float()).abs().max().item() <= 2e-3      # same products, different summation order
    ref, rprobs = oracle_lib.local_attn_fwd(host(s), f.cpu().numpy(), host(l), k, return_probs=True)
    np.testing.assert_allclose(host(probs), rprobs, rtol=0, atol=4e-3)
    np.testing.assert_allclose(host(out), ref, rtol=0, atol=1e-2)


@pytest.mark.parametrize("dt", [torch.bfloat16, torch.float32, torch.float64])
def test_relayout_roundtrip(F_, dt):
    torch.manual_seed(0)
    x = torch.randn(3, 70, 13, 9, device=DEV).to(dt)
    y = F_.relayout(x, True)
    assert y.is_contiguous(memory_format=torch.channels_last) and torch.equal(y, x)
    z = F_.relayout(y, False)
    assert z.is_contiguous() and torch.equal(z, x)


# ----------------------------------------------------------------------------- fused mask blend (SURVEY 8(f2), generator.py:130)
@pytest.mark.parametrize("cfg", [("fp32", "nchw", "gather"), ("fp32", "nhwc", "gather"), ("bf16", "nchw", "tile"), ("bf16", "nhwc", "tile")])
def test_local_attn_blend_fwd(F_, oracle_lib, cfg):
    """out = prev*(1-mask) + local_attention*mask in one kernel == oracle attention blended on the host"""
    prec, layout, algo = cfg
    rng = np.random.default_rng(17)
    B, C, H, W, k = 2, 64, 21, 40, 5
    dt = torch.float32 if prec == "fp32" else torch.bfloat16
    s = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).to(dt)
    prev = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).to(dt)
    mask = torch.from_numpy(rng.uniform(0, 1, (B, 1, H, W)).astype(np.float32)).to(DEV).to(dt)
    f = torch.from_numpy(_flow(rng, "smooth", B, H, W).astype(np.float32)).to(DEV)
    l = torch.from_numpy(rng.standard_normal((B, k * k, H, W)).astype(np.float32)).to(DEV).to(dt)
    if layout == "nhwc":
        s, prev = s.contiguous(memory_format=torch.channels_last), prev.contiguous(memory_format=torch.channels_last)
    out = F_.local_attn_blend_fwd(s, f, l, prev, mask, k, algo=algo)
    attn = oracle_lib.local_attn_fwd(host(s), f.cpu().numpy(), host(l), k)
    ref = host(prev) * (1 - host(mask)) + attn * host(mask)
    np.testing.assert_allclose(host(out), ref, rtol=0, atol=1e-5 if prec == "fp32" else 2e-2)   # bf16: |prev| ~ 3, one rounding


def test_extractor_attn_mask_blend_module():
    """ExtractorAttn(..., mask=m): fused store under no_grad == torch composition with autograd"""
    import gfla_b200
    torch.manual_seed(6)
    C, k, B, H, W = 64, 3, 1, 16, 24
    m = gfla_b200.ExtractorAttn(C, k, softmax=True).to(DEV).bfloat16().to(memory_format=torch.channels_last)
    cl = torch.channels_last
    src = torch.randn(B, C, H, W, device=DEV).bfloat16().contiguous(memory_format=cl)
    tgt = torch.randn(B, C, H, W, device=DEV).bfloat16().contiguous(memory_format=cl)
    flow = (torch.rand(B, 2, H, W, device=DEV) * 6 - 3)
    mask = torch.rand(B, 1, H, W, device=DEV).bfloat16()
    with torch.no_grad():
        fused = m(src, tgt, flow, mask=mask)
        plain = m(src, tgt, flow)
    ref = tgt.float() * (1 - mask.float()) + plain.float() * mask.float()
    assert (fused.float() - ref).abs().max().item() <= 3e-2
    src.requires_grad_()
    out = m(src, tgt, flow, mask=mask)        # gradient needed -> unfused composition, still correct and differentiable
    out.float().sum().backward()
    assert src.grad is not None and torch.isfinite(src.grad.float()).all()


def test_block_extractor_bf16_backward_fp32_accumulation(F_, oracle_lib):
    """16-bit storage: grad_source is scattered into an fp32 buffer and narrowed once (functional.block_extract_bwd)"""
    rng = np.random.default_rng(23)
    B, C, H, W, k = 1, 6, 12, 14, 3
    s = torch.from_numpy(rng.standard_normal((B, C, H, W)).astype(np.float32)).to(DEV).bfloat16()
    f = torch.from_numpy(rng.uniform(-4, 4, (B, 2, H, W)).astype(np.float32)).to(DEV)
    g = torch.from_numpy(rng.standard_normal((B, C, k * H, k * W)).astype(np.float32)).to(DEV).bfloat16()
    gs, gf = F_.block_extract_bwd(s, f, g, k)
    assert gs.dtype == torch.bfloat16
    ogs, ogf = oracle_lib.block_extract_bwd(host(s), f.cpu().numpy(), host(g), k)
    np.testing.assert_allclose(host(gs), ogs, rtol=1e-2, atol=1e-2 * max(1.0, float(np.abs(ogs).max())))
    np.testing.assert_allclose(host(gf), ogf, rtol=1e-3, atol=1e-3 * max(1.0, float(np.abs(ogf).max())))


@pytest.mark.parametrize("cfg", [(4, 1, "smooth"), (2, 1, "smooth"), (4, 2, "smooth"), (4, 1, "torn"), (6, 1, "smooth"), (4, 1, "far")])
def test_resample2d_ragged_tiles_and_torn_flows(F_, oracle_lib, cfg):
    """resample2d on 32x4 pixel tiles (resample2d.cu): ragged tiles (H % 4, W % 32 != 0), an odd channel count, dilation 2, a flow
    that tears a tile apart (columns 40.. jump 45 pixels), and a flow that leaves the image (every tap clamped onto the border
    column, i.e. maximal atomic contention in grad_input1): forward and both gradients against the oracle."""
    ks, dil, kind = cfg
    rng = np.random.default_rng(ks * 7 + dil + len(kind))
    B, C, H, W = 2, 7, 21, 70
    a = rng.standard_normal((B, C, H, W)).astype(np.float32)
    yy, xx = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    if kind == "smooth":
        fl = np.stack([3.0 * np.sin(xx / 9.0) + 0.3 * yy, 2.5 * np.cos(yy / 5.0) - 0.2 * xx / 4], 0)[None].repeat(B, 0)
    elif kind == "torn":       # columns 40.. of the middle tile jump 45 pixels to the left: its footprint is > 64 wide
        fl = np.stack([np.where(xx >= 40, -45.0, 1.5) + 0.3 * rng.random((H, W)), 0.7 * rng.random((H, W))], 0)[None].repeat(B, 0)
    else:
        fl = np.stack([np.full((H, W), 500.0), -300.0 + rng.random((H, W))], 0)[None].repeat(B, 0)
    fl = fl + 0.05 * rng.standard_normal(fl.shape)
    in2 = np.ascontiguousarray(np.concatenate([fl, np.full((B, 1, H, W), 2.0)], 1).astype(np.float32))
    g = rng.standard_normal((B, C, H, W)).astype(np.float32)
    g1, g2 = F_.resample2d_bwd(cu(a), cu(in2), cu(g), ks, dil)
    o1, o2 = oracle_lib.resample2d_bwd(a, in2, g, ks, dil)
    np.testing.assert_allclose(host(g1), o1, rtol=1e-5, atol=1e-5 * max(1.0, float(np.abs(o1).max())))
    np.testing.assert_allclose(host(g2), o2, rtol=1e-4, atol=1e-4 * max(1.0, float(np.abs(o2).max())))
    out = F_.resample2d_fwd(cu(a), cu(in2), ks, dil)
    np.testing.assert_allclose(host(out), oracle_lib.resample2d_fwd(a, in2, ks, dil), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("cfg", [(2, 5.0, "uniform"), (4, 2.0, "uniform"), (4, 2.0, "mixed"), (2, 5.0, "border")])
def test_resample2d_backward_uniform_mixed_border_flows(F_, oracle_lib, dt, cfg):
    """grad_input1 on flows with one integer tap shift per row, a shift that changes mid-row, and taps clamped at the border"""
    ks, sigma, kind = cfg
    rng = np.random.default_rng(ks + len(kind))
    B, C, H, W = 2, 5, 9, 64
    a = rng.standard_normal((B, C, H, W)).astype(dt)
    if kind == "uniform":      # floor(x + dx) - x == 2, floor(y + dy) - y == -1 everywhere (interior rows only matter)
        fl = np.stack([2.2 + 0.6 * rng.random((B, H, W)), -0.9 + 0.8 * rng.random((B, H, W))], 1)
    elif kind == "mixed":      # shift changes in the middle of some rows
        fl = np.stack([np.where(np.arange(W)[None, None, :] < 40, 1.3, 2.6) + 0.2 * rng.random((B, H, W)),
                       0.4 * rng.random((B, H, W))], 1)
    else:                      # taps clamped at the image border
        fl = np.stack([np.full((B, H, W), 7.5) * np.sign(rng.standard_normal((B, H, 1))), rng.uniform(-6, 6, (B, H, W))], 1)
    in2 = np.ascontiguousarray(np.concatenate([fl, np.full((B, 1, H, W), sigma)], 1).astype(dt))
    g = rng.standard_normal((B, C, H, W)).astype(dt)
    g1, g2 = F_.resample2d_bwd(cu(a), cu(in2), cu(g), ks, 1)
    o1, o2 = oracle_lib.resample2d_bwd(a, in2, g, ks, 1)
    t = tol(dt, 1e-5, 1e-12)
    np.testing.assert_allclose(host(g1), o1, rtol=t, atol=t * max(1.0, float(np.abs(o1).max())))
