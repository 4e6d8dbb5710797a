"""GPU (-m gpu): parity against the REFERENCE'S OWN kernels at BASELINE.json's full sizes.

The `<5,256>` tile instantiations that bench.py times are checked at 256x256, C=256, k=5 -- forward and
backward -- against the reference itself, not only against our own kernels.  What the reference computed on
these seeded inputs (its kernel bodies compiled for the host, oracle/_ref, composed like its ExtractorAttn) is
stored in tests/golden/reference_fullsize.npz by tests/golden/make_golden.py: each output at the same fixed
sample of positions (conftest.sample_index) plus its largest magnitude.  Tolerances = north_star: 1e-4 fp32,
1e-2 bf16 (absolute, flat).

test_refcuda_equals_host_reference checks the two builds of the reference's kernel text against each other:
  * ``oracle/_ref/libgfla_ref.so``       -- the reference kernel bodies compiled for the host (OpenMP);
  * ``oracle/_ref/libgfla_ref_cuda.so``  -- the same extracted text compiled by nvcc for sm_100a
    (``oracle/ref_cuda*.cu``: plain launchers, no ATen) = "the reference's CUDA kernels, recompiled".
Both are built by ``__graft_entry__.build()`` only where a checkout of the reference exists; it skips elsewhere.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, sample_index

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CL = torch.channels_last


@pytest.fixture(scope="module")
def RC():
    import oracle.ref_cuda as rc
    if not rc.available():
        pytest.skip("oracle/_ref/libgfla_ref_cuda.so not built (needs /root/reference at build time)")
    return rc


@pytest.fixture(scope="module")
def F_():
    import gfla_b200
    from gfla_b200 import _lib
    _lib.check(_lib.lib().gfla_device_check(), "device check")
    return gfla_b200.functional


def _smooth_flow(B, H, W, amp=8.0, seed=0, device=DEV):
    g = torch.Generator(device="cpu").manual_seed(seed)
    coarse = torch.rand(B, 2, max(H // 16, 2), max(W // 16, 2), generator=g) * 2 * amp - amp
    return torch.nn.functional.interpolate(coarse, size=(H, W), mode="bilinear", align_corners=True).to(device).contiguous()


def _inputs(B, C, H, W, k, kind, seed, device=DEV):
    g = torch.Generator(device="cpu").manual_seed(seed)
    src = torch.randn(B, C, H, W, generator=g).to(device)
    logits = torch.randn(B, k * k, H, W, generator=g).to(device)
    gout = torch.randn(B, C, H, W, generator=g).to(device)
    flow = _smooth_flow(B, H, W, seed=seed, device=device) if kind == "smooth" else ((torch.rand(B, 2, H, W, generator=g) * 16 - 8).to(device))
    return src, flow, logits, gout


# inputs of the full-size cases, on `device` (tests/golden/make_golden.py builds them on the host)
def cfg2_case(name, device=DEV):
    """-> (inputs in the dtype the reference ran on, k); the bf16 cases hand the reference the bf16-rounded values"""
    B, kind, seed, bf16 = {"tile_smooth": (2, "smooth", 21, True), "tile_iid": (2, "iid", 21, True), "planar": (1, "smooth", 22, True),
                           "fp32": (1, "smooth", 23, False), "host": (1, "smooth", 24, True)}[name]
    src, flow, logits, gout = _inputs(B, 256, 256, 256, 5, kind, seed, device)
    if bf16:
        src, logits, gout = (t.bfloat16().float() for t in (src, logits, gout))
    return (src, flow, logits, gout), 5


def block_extractor_case(device=DEV):
    B, C, H, W, k = 1, 256, 256, 256, 5
    src, flow, _, _ = _inputs(B, C, H, W, k, "smooth", seed=25, device=device)
    go = torch.randn(B, C, k * H, k * W, generator=torch.Generator(device="cpu").manual_seed(26)).to(device)
    return (src, flow, go), k


def resample2d_case(ks, sigma, device=DEV):
    B, C, H, W = 2, 128, 512, 512
    g = torch.Generator(device="cpu").manual_seed(31)
    x = torch.randn(B, C, H, W, generator=g).to(device)
    go = torch.randn(B, C, H, W, generator=g).to(device)
    in2 = torch.cat([_smooth_flow(B, H, W, seed=3, device=device), torch.full((B, 1, H, W), sigma, device=device)], 1).contiguous()
    return (x, in2, go), ks


@pytest.fixture(scope="module")
def REF():
    return load_golden("reference_fullsize")


class _Ref:
    """one case of the stored reference outputs: ref[name] = sampled values on the GPU, ref.absmax(name) = max |value|"""

    def __init__(self, case):
        self.case = case

    def __getitem__(self, name):
        return torch.from_numpy(self.case[name]).to(DEV)

    def absmax(self, name):
        return float(self.case[name + "_absmax"])


def _at(t):
    """t (any storage order) at the stored positions of its logical C-order flattening, as float32"""
    flat = t.detach().float().reshape(-1)
    return flat[torch.from_numpy(sample_index(flat.numel())).to(flat.device)]


# ----------------------------------------------------------------------------- the checker itself: nvcc build == host build
@pytest.mark.parametrize("k", [3, 4, 5])
def test_refcuda_equals_host_reference(RC, ref_lib, k):
    """same reference text through g++ (no FMA contraction) and through nvcc (FMA contraction on, like the
    reference's own build): equal up to that contraction"""
    rng = np.random.default_rng(k)
    B, C, H, W = 2, 6, 14, 10
    s = rng.standard_normal((B, C, H, W)).astype(np.float32)
    f = rng.uniform(-6, 6, (B, 2, H, W)).astype(np.float32)
    go = rng.standard_normal((B, C, k * H, k * W)).astype(np.float32)
    ts, tf, tg = (torch.from_numpy(a).to(DEV) for a in (s, f, go))
    np.testing.assert_allclose(RC.block_extract_fwd(ts, tf, k).cpu().numpy(), ref_lib.block_extract_fwd(s, f, k), rtol=1e-6, atol=1e-6)
    gs, gf = RC.block_extract_bwd(ts, tf, tg, k)
    rgs, rgf = ref_lib.block_extract_bwd(s, f, go, k)
    np.testing.assert_allclose(gs.cpu().numpy(), rgs, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(gf.cpu().numpy(), rgf, rtol=1e-4, atol=1e-4)
    x = rng.standard_normal((B, k * k, H, W)).astype(np.float32)
    assert np.array_equal(RC.attn_reshape_fwd(torch.from_numpy(x).to(DEV), k).cpu().numpy(), ref_lib.attn_reshape_fwd(x, k))
    if k == 4:
        in2 = np.concatenate([f, np.full((B, 1, H, W), 2.0, np.float32)], 1)
        t2 = torch.from_numpy(in2).to(DEV)
        np.testing.assert_allclose(RC.resample2d_fwd(ts, t2, 4, 1).cpu().numpy(), ref_lib.resample2d_fwd(s, in2, 4, 1), rtol=1e-5, atol=1e-6)


# ----------------------------------------------------------------------------- full-size cfg2 samples vs the reference's kernels
@pytest.mark.parametrize("kind", ["smooth", "iid"])
def test_cfg2_fullsize_tile_path_vs_reference_cuda(REF, F_, kind):
    """B=2, C=256, 256x256, k=5, bf16 channels_last -- exactly the <5,256> kernels of the bench step (strip forward,
    tile backward) -- vs the reference's unfused pipeline in fp32 on the bf16-rounded inputs"""
    (src, flow, logits, gout), k = cfg2_case(f"tile_{kind}")
    ref = _Ref(REF[f"tile_{kind}"])
    sb, lb, gb = src.bfloat16(), logits.bfloat16(), gout.bfloat16()
    s_cl, g_cl = sb.contiguous(memory_format=CL), gb.contiguous(memory_format=CL)
    out = F_.local_attn_fwd(s_cl, flow, lb, k, algo="tile")
    gs, gf, gl = F_.local_attn_bwd(s_cl, flow, lb, g_cl, k, algo="tile")
    assert (_at(out) - ref["out"]).abs().max().item() <= 1e-2
    assert (_at(gs) - ref["grad_source"]).abs().max().item() <= 1e-2                      # flat, like north_star
    assert (_at(gs) - ref["grad_source"]).abs().max().item() <= 1e-2 * max(1.0, ref.absmax("grad_source"))
    assert (_at(gl) - ref["grad_logits"]).abs().max().item() <= 1e-2
    # grad_flow sums C*k*k products of O(1) terms: bf16 inputs are exact here, the difference is summation order / Q in fp32
    assert (_at(gf) - ref["grad_flow"]).abs().max().item() <= 1e-2 * max(1.0, ref.absmax("grad_flow"))
    # error histogram of grad_source (the bf16 reduce-add path): how far from the bound the bulk sits
    err = (_at(gs) - ref["grad_source"]).abs()
    assert err.mean().item() <= 1e-3


def test_cfg2_fullsize_planar_nchw_vs_reference_cuda(REF, F_):
    """the reference's own contiguous-NCHW contract at full size (forward NCHW tile kernel, backward through the tile kernels)"""
    (src, flow, logits, gout), k = cfg2_case("planar")
    ref = _Ref(REF["planar"])
    sb, lb, gb = src.bfloat16(), logits.bfloat16(), gout.bfloat16()
    out = F_.local_attn_fwd(sb, flow, lb, k)
    gs, gf, gl = F_.local_attn_bwd(sb, flow, lb, gb, k)
    assert out.is_contiguous() and gs.is_contiguous()
    assert (_at(out) - ref["out"]).abs().max().item() <= 1e-2
    assert (_at(gs) - ref["grad_source"]).abs().max().item() <= 1e-2
    assert (_at(gl) - ref["grad_logits"]).abs().max().item() <= 1e-2
    assert (_at(gf) - ref["grad_flow"]).abs().max().item() <= 1e-2 * max(1.0, ref.absmax("grad_flow"))


def test_cfg2_fullsize_fp32_vs_reference_cuda(REF, F_):
    """fp32 (the reference's dtype), one full-size sample: 1e-4"""
    (src, flow, logits, gout), k = cfg2_case("fp32")
    ref = _Ref(REF["fp32"])
    out = F_.local_attn_fwd(src, flow, logits, k)
    gs, gf, gl = F_.local_attn_bwd(src, flow, logits, gout, k)
    assert (_at(out) - ref["out"]).abs().max().item() <= 1e-4
    assert (_at(gs) - ref["grad_source"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_source"))
    assert (_at(gl) - ref["grad_logits"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_logits"))
    assert (_at(gf) - ref["grad_flow"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_flow"))


def test_cfg2_one_fullsize_sample_vs_host_reference(REF, F_):
    """...and one more full-size sample, forward + backward, tile path"""
    (src, flow, logits, gout), k = cfg2_case("host")
    ref = _Ref(REF["host"])
    sb, lb, gb = src.bfloat16(), logits.bfloat16(), gout.bfloat16()
    s_cl, g_cl = sb.contiguous(memory_format=CL), gb.contiguous(memory_format=CL)
    out = F_.local_attn_fwd(s_cl, flow, lb, k, algo="tile")
    gs, gf, gl = F_.local_attn_bwd(s_cl, flow, lb, g_cl, k, algo="tile")
    assert (_at(out) - ref["out"]).abs().max().item() <= 1e-2
    assert (_at(gs) - ref["grad_source"]).abs().max().item() <= 1e-2
    assert (_at(gl) - ref["grad_logits"]).abs().max().item() <= 1e-2
    assert (_at(gf) - ref["grad_flow"]).abs().max().item() <= 1e-2 * max(1.0, ref.absmax("grad_flow"))


# ----------------------------------------------------------------------------- unfused ops at (chunks of) their BASELINE sizes
def test_block_extractor_cfg2_chunk_vs_reference_cuda(REF, F_):
    (src, flow, go), k = block_extractor_case()
    ref = _Ref(REF["block_extractor"])
    ours = F_.block_extract_fwd(src, flow, k)
    assert (_at(ours) - ref["out"]).abs().max().item() <= 1e-5
    del ours
    gs, gf = F_.block_extract_bwd(src, flow, go, k)
    assert (_at(gs) - ref["grad_source"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_source"))
    assert (_at(gf) - ref["grad_flow"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_flow"))


@pytest.mark.parametrize("ks,sigma", [(2, 5.0), (4, 2.0)])
def test_resample2d_cfg3_chunk_vs_reference_cuda(REF, F_, ks, sigma):
    """cfg3 shape (C=128, 512x512 fp32), two samples: forward and both gradients vs the reference's kernels"""
    (x, in2, go), ks = resample2d_case(ks, sigma)
    ref = _Ref(REF[f"resample2d_ks{ks}"])
    out = F_.resample2d_fwd(x, in2, ks, 1)
    assert (_at(out) - ref["out"]).abs().max().item() <= 1e-4
    g1, g2 = F_.resample2d_bwd(x, in2, go, ks, 1)
    assert (_at(g1) - ref["grad_in1"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_in1"))
    assert (_at(g2) - ref["grad_in2"]).abs().max().item() <= 1e-4 * max(1.0, ref.absmax("grad_in2"))
