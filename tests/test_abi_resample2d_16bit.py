"""CPU: the channels-last 16-bit resample2d entry points reject bad arguments with the documented GFLA_E_* code before
anything is launched (no device is touched here)."""
import ctypes

import pytest

BF16, F16, F32, F64 = 2, 3, 0, 1


@pytest.fixture(scope="module")
def so():
    import __graft_entry__ as ge
    ge.build_cuda()
    import gfla_b200
    return gfla_b200._lib.lib()


@pytest.fixture(scope="module")
def p():
    buf = (ctypes.c_double * 64)()          # 8-byte aligned; kept alive with the address
    return ctypes.addressof(buf), buf


def _calls(so, p, *, null=None, size=1, ks=2, dtype=BF16, gdtype=BF16, mis=None):
    """one call of each entry; `null`/`mis` name the argument to replace with NULL / an odd address"""
    def a(name):
        if name == null:
            return None
        if name == mis:
            return p + 1
        return p
    d = 1.0e-8
    return {
        "fwd": so.gfla_resample2d_fwd_nhwc(a("in1"), a("in2"), a("out"), 1, size, 2, 2, 2, 2, ks, 1, dtype, None),
        "bwd": so.gfla_resample2d_bwd_nhwc(a("in1"), a("in2"), a("out"), a("grad_in1"), a("grad_in2"), 1, size, 2, 2, 2, 2, ks, 1, dtype,
                                           gdtype, 0, None),
        "cos_fwd": so.gfla_resample2d_cosine_fwd_nhwc(a("in1"), a("in2"), a("target"), a("out"), a("stats"), 1, size, 2, 2, 2, 2, ks, 1, d,
                                                      dtype, None),
        "cos_bwd": so.gfla_resample2d_cosine_bwd_nhwc(a("in1"), a("in2"), a("target"), a("stats"), a("out"), a("grad_in1"), a("grad_in2"),
                                                      a("grad_val"), None, 1, size, 2, 2, 2, 2, ks, 1, d, dtype, gdtype, 0, None),
    }


def test_null_pointer(so, p):
    p, _ = p
    for name in ("in1", "in2"):
        assert set(_calls(so, p, null=name).values()) == {-1}, name
    assert _calls(so, p, null="grad_in2")["bwd"] == -1
    assert _calls(so, p, null="grad_val")["cos_bwd"] == -1      # grad_in1 wanted without its grad_val scratch


def test_bad_size_or_kernel_size(so, p):
    p, _ = p
    for kw in ({"size": 0}, {"size": -3}, {"ks": 1}, {"ks": 10}):
        assert set(_calls(so, p, **kw).values()) == {-2}, kw


@pytest.mark.parametrize("dtype", [F32, F64, 7, -1])
def test_dtype_not_16bit(so, p, dtype):
    p, _ = p
    assert set(_calls(so, p, dtype=dtype, gdtype=F32).values()) == {-3}


@pytest.mark.parametrize("gdtype", [F64, F16, 9])
def test_bad_grad_in1_dtype(so, p, gdtype):
    p, _ = p
    r = _calls(so, p, dtype=BF16, gdtype=gdtype)
    assert r["bwd"] == -3 and r["cos_bwd"] == -3


def test_misaligned(so, p):
    p, _ = p
    assert set(_calls(so, p, mis="in1").values()) == {-4}
    assert set(_calls(so, p, mis="in2").values()) == {-4}       # in2 is fp32
    assert _calls(so, p, mis="grad_in1", gdtype=F32)["bwd"] == -4


def test_planar_entries_still_reject_16bit(so, p):
    p, _ = p
    assert so.gfla_resample2d_fwd(p, p, p, 1, 1, 2, 2, 2, 2, 2, 1, BF16, None) == -3
    assert so.gfla_abi_version() == 1
