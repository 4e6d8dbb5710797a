"""CPU: the oracle against the reference's own kernel bodies compiled for the host (oracle/_ref), on seeded
random inputs -- bit for bit, one host thread so the atomics' accumulation order is the thread-index order.
The reference's outputs on these inputs are stored as digests (conftest.sha256) in
tests/golden/oracle_vs_ref.npz by tests/golden/make_golden.py."""
import numpy as np
import pytest

from conftest import load_golden, sha256

BLOCK_SHAPES = [(1, 8, 32, 32, 32, 32, 3), (2, 3, 7, 9, 7, 9, 4), (2, 4, 9, 11, 6, 5, 5), (1, 2, 5, 5, 5, 5, 2)]
RESAMPLE_CFGS = [(2, 3, 8, 9, 8, 9, 2, 1, 5.0, 4.0), (1, 4, 10, 12, 7, 6, 4, 1, 2.0, 12.0), (1, 2, 9, 9, 9, 9, 4, 2, 2.0, 3.0),
                 (1, 2, 6, 6, 6, 6, 2, 1, 0.0, 2.0)]
RESHAPE_KS = (2, 3, 4, 5)


def block_inputs(dt, shape):
    B, C, Hs, Ws, H, W, k = shape
    rng = np.random.default_rng(list(shape))
    s = rng.standard_normal((B, C, Hs, Ws)).astype(dt)
    f = rng.uniform(-1.5 * W, 1.5 * W, (B, 2, H, W)).astype(dt)
    g = rng.standard_normal((B, C, k * H, k * W)).astype(dt)
    return s, f, g, k


def resample_inputs(dt, cfg):
    B, C, Hi, Wi, H, W, ks, dil, sig, amp = cfg
    rng = np.random.default_rng(7)
    a1 = rng.standard_normal((B, C, Hi, Wi)).astype(dt)
    in2 = np.concatenate([rng.uniform(-amp, amp, (B, 2, H, W)), np.full((B, 1, H, W), sig)], 1).astype(dt)
    g = rng.standard_normal((B, C, H, W)).astype(dt)
    return a1, in2, g, ks, dil


def reshape_inputs(k):
    rng = np.random.default_rng(3 + k)
    x = rng.standard_normal((2, k * k, 5, 7)).astype(np.float32)
    g = rng.standard_normal((2, 1, 5 * k, 7 * k)).astype(np.float32)
    return x, g


def case_name(op, *params):
    return op + "-" + "-".join(str(p) for p in params)


def block_outputs(lib, dt, shape):
    s, f, g, k = block_inputs(dt, shape)
    return {"out": lib.block_extract_fwd(s, f, k), **dict(zip(("grad_source", "grad_flow"), lib.block_extract_bwd(s, f, g, k)))}


def resample_outputs(lib, dt, cfg):
    a1, in2, g, ks, dil = resample_inputs(dt, cfg)
    return {"out": lib.resample2d_fwd(a1, in2, ks, dil), **dict(zip(("grad_in1", "grad_in2"), lib.resample2d_bwd(a1, in2, g, ks, dil)))}


def reshape_outputs(lib, k):
    x, g = reshape_inputs(k)
    return {"out": lib.attn_reshape_fwd(x, k), "grad_in": lib.attn_reshape_bwd(x, g, k)}


@pytest.fixture(scope="module")
def REF():
    return load_golden("oracle_vs_ref")


def _check(REF, name, outputs):
    want = REF[name]
    assert sorted(want) == sorted(outputs)
    for key, a in outputs.items():
        assert sha256(a) == str(want[key]), key


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("shape", BLOCK_SHAPES)
def test_block_extractor(oracle_lib, REF, dt, shape):
    _check(REF, case_name("block_extractor", np.dtype(dt).name, *shape), block_outputs(oracle_lib, dt, shape))


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("cfg", RESAMPLE_CFGS)
def test_resample2d(oracle_lib, REF, dt, cfg):
    _check(REF, case_name("resample2d", np.dtype(dt).name, *cfg), resample_outputs(oracle_lib, dt, cfg))


def test_reshape(oracle_lib, REF):
    for k in RESHAPE_KS:
        _check(REF, case_name("reshape", k), reshape_outputs(oracle_lib, k))
