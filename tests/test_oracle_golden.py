"""CPU: the oracle (our C restatement) against the committed golden vectors,
which were produced by the reference's own kernel bodies (tests/golden/make_golden.py).

Bit-exact for the three ops (same arithmetic, same order, no FMA contraction);
the fused tail is compared with a tolerance because the goldens use torch's
vectorised softmax / avg_pool2d."""
import numpy as np
import pytest

from conftest import load_golden, sha256


@pytest.mark.parametrize("case", sorted(load_golden("block_extractor")))
def test_block_extractor(oracle_lib, case):
    g = load_golden("block_extractor")[case]
    k = int(g["k"])
    out = oracle_lib.block_extract_fwd(g["source"], g["flow"], k)
    assert sha256(out) == str(g["out_sha256"])
    gs, gf = oracle_lib.block_extract_bwd(g["source"], g["flow"], g["grad_out"], k)
    assert np.array_equal(gs, g["grad_source"])
    assert np.array_equal(gf, g["grad_flow"])


def test_block_extractor_zero_flow_identity(oracle_lib):
    """test_block_extractor.py:55: with zero flow the k x k tile of pixel (1,1)
    is the 3x3 neighbourhood of the source around (1,1)."""
    g = load_golden("block_extractor")["zero_flow"]
    out = oracle_lib.block_extract_fwd(g["source"], g["flow"], 3)
    assert np.array_equal(out[0, 0, 3:6, 3:6], g["source"][0, 0, 0:3, 0:3])


@pytest.mark.parametrize("case", sorted(load_golden("local_attn_reshape")))
def test_local_attn_reshape(oracle_lib, case):
    g = load_golden("local_attn_reshape")[case]
    k = int(g["k"])
    out = oracle_lib.attn_reshape_fwd(g["in"], k)
    assert np.array_equal(out, g["out"])
    if case == "layout":  # test_local_attn_reshape.py:29-43
        assert np.array_equal(out[0, 0, :3, :3], np.arange(9, dtype=np.float32).reshape(3, 3))
    else:
        assert np.array_equal(oracle_lib.attn_reshape_bwd(g["in"], g["grad_out"], k), g["grad_in"])


@pytest.mark.parametrize("case", sorted(load_golden("resample2d")))
def test_resample2d(oracle_lib, case):
    g = load_golden("resample2d")[case]
    ks, dil = int(g["ks"]), int(g["dil"])
    out = oracle_lib.resample2d_fwd(g["in1"], g["in2"], ks, dil)
    assert np.array_equal(out, g["out"], equal_nan=True)
    g1, g2 = oracle_lib.resample2d_bwd(g["in1"], g["in2"], g["grad_out"], ks, dil)
    assert np.array_equal(g1, g["grad_in1"], equal_nan=True)
    assert np.array_equal(g2, g["grad_in2"], equal_nan=True)


@pytest.mark.parametrize("case", sorted(load_golden("local_attn")))
def test_local_attn(oracle_lib, case):
    g = load_golden("local_attn")[case]
    k = int(g["k"])
    tol = 2e-6 if g["source"].dtype == np.float32 else 1e-13
    out, probs = oracle_lib.local_attn_fwd(g["source"], g["flow"], g["logits"], k, return_probs=True)
    np.testing.assert_allclose(probs, g["probs"], rtol=tol, atol=tol)
    np.testing.assert_allclose(out, g["out"], rtol=tol, atol=tol)
    gs, gf, gl = oracle_lib.local_attn_bwd(g["source"], g["flow"], g["logits"], g["grad_out"], k)
    np.testing.assert_allclose(gs, g["grad_source"], rtol=10 * tol, atol=10 * tol)
    np.testing.assert_allclose(gf, g["grad_flow"], rtol=10 * tol, atol=10 * tol)
    np.testing.assert_allclose(gl, g["grad_logits"], rtol=10 * tol, atol=10 * tol)
