"""The C-ABI library loads on a machine without a GPU and exports every symbol that
include/pyro_b200.h declares; entry points validate their arguments without launching."""
import ctypes
import os
import re

import pytest

from pyro_b200 import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    with open(os.path.join(ROOT, "include", "pyro_b200.h")) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b2_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported():
    lib = ctypes.CDLL(N.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "missing export: " + n
    assert set(names) == set(N.SIGNATURES), set(names) ^ set(N.SIGNATURES)


def test_argument_validation_without_gpu():
    L = N.lib()
    assert L.b2_version() >= 100
    assert L.b2_last_error(-3).decode().startswith("unknown distribution family")
    assert L.b2_site_score_workspace() > 0
    t = N.b2_tensor()
    # bad family / null pointers are rejected before any CUDA call
    assert L.b2_site_score(999, ctypes.byref(t), ctypes.byref(t), 1, None, 1.0, None, 1.0, 1.0, 0,
                           None, None, None, None, None, 0, None) == -3
    assert L.b2_site_score(0, None, None, 2, None, 1.0, None, 1.0, 1.0, 0, None, None, None, None,
                           None, 0, None) == -4
    assert L.b2_glm_bernoulli_logits(None, None, None, None, 10, 32, 8, 1.0, 1.0, 1.0, 0, None, None,
                                     None, None, None, 0, None) == -4
    # retired GLM flag bits (8, 16, 64) and unknown bits are refused; the supported ones get as far as the
    # workspace check (no workspace given).  The pointers are 16-byte aligned and never dereferenced.
    x = ctypes.c_void_p(4096)
    for bit in (8, 16, 64, 128):
        assert L.b2_glm_bernoulli_logits(x, x, x, None, 10, 32, 8, 1.0, 1.0, 1.0, bit, None, None,
                                         None, None, None, 0, None) == -2, bit
    ok = N.B2_FLAG_ACCUMULATE_SUM | N.B2_FLAG_GLM_FP32 | N.B2_FLAG_GLM_3XTF32
    assert L.b2_glm_bernoulli_logits(x, x, x, None, 10, 32, 8, 1.0, 1.0, 1.0, ok, None, None,
                                     None, None, None, 0, None) == -5
    assert L.b2_nuts_small(None, None, None, None, None, None, 1, 1, 10, 1000.0, 0, None, None, None,
                           None, None, None, None) == -4


def test_cpu_tensors_are_refused_loudly():
    import torch
    import pyro_b200.distributions as dist
    with pytest.raises(RuntimeError, match="no CPU"):
        dist.Normal(torch.zeros(3), torch.ones(3)).log_prob(torch.zeros(3))


def test_latent_and_gamma_entry_points_validate_before_launching():
    """Round-2 entry points (csrc/latent.cu, gamma_rsample.cu): null pointers, job counts, shapes, dtypes and
    32-bit offset limits are rejected before any CUDA call -- which also pins the ctypes layout of
    ``b2_latent_job`` against the header (each check reads a different field group of the struct)."""
    L = N.lib()
    one = (N.b2_latent_job * 1)()
    j = one[0]
    j.dtype, j.ndim = N._DTYPES[__import__("torch").float32], 2
    j.shape[0], j.shape[1] = 4, 8
    dummy = ctypes.c_void_p(4096)                      # never dereferenced: validation fails first
    assert L.b2_latent_normal_draw(one, 1, None, None) == -4                  # no RNG state
    assert L.b2_latent_normal_draw(None, 1, dummy, None) == -4                # no jobs
    assert L.b2_latent_normal_draw(one, 0, dummy, None) == -2                 # job count
    assert L.b2_latent_normal_draw(one, N.LATENT_MAX_JOBS + 1, dummy, None) == -2
    assert L.b2_latent_normal_draw(one, 1, dummy, None) == -4                 # operands missing
    j.ndim = 9
    assert L.b2_latent_normal_prior(one, 1, None) == -2                       # too many dims
    j.ndim = 2
    j.shape[0] = 0
    assert L.b2_latent_normal_backward(one, 1, None) == -2                    # empty dim
    j.shape[0], j.shape[1] = 1024, 1024
    assert L.b2_latent_normal_backward(one, 1, None) == -8                    # > B2_RSAMPLE_MAX_N elements
    j.shape[0], j.shape[1] = 4, 8
    j.scale_stride[1] = 1 << 20
    assert L.b2_latent_normal_prior(one, 1, None) == -8                       # offset would leave 32 bits
    j.scale_stride[1] = 1
    j.prior_scale_stride[0] = -(1 << 20)
    assert L.b2_latent_normal_prior(one, 1, None) == -8
    j.prior_scale_stride[0] = 0
    j.dtype = 77
    assert L.b2_latent_normal_prior(one, 1, None) == -1                       # dtype
    two = (N.b2_latent_job * 2)()
    for k, dt in enumerate((__import__("torch").float32, __import__("torch").float64)):
        two[k].dtype, two[k].ndim = N._DTYPES[dt], 1
        two[k].shape[0] = 3
    assert L.b2_latent_normal_prior(two, 2, None) == -1                       # mixed dtypes in one launch
    coeffs = (ctypes.c_double * 1)(1.0)
    assert L.b2_latent_normal_prior_combine(one, 1, coeffs, None, None, 0, None, None) == -4   # no output
    assert L.b2_latent_normal_prior_combine(one, 1, coeffs, None, None, N.LATENT_MAX_TERMS + 1, dummy, None) == -4
    t = N.b2_tensor()
    assert L.b2_gamma_rsample(None, None, 1, None, None, None, None, None) == -4
    shp = (ctypes.c_int64 * 1)(5)
    t.dtype = N._DTYPES[__import__("torch").float32]
    t2 = N.b2_tensor()
    t2.dtype = N._DTYPES[__import__("torch").float64]
    assert L.b2_gamma_rsample(ctypes.byref(t), ctypes.byref(t2), 1, shp, dummy, None, dummy, None) == -1
    assert L.b2_gamma_rsample(ctypes.byref(t), ctypes.byref(t), 7, shp, dummy, None, dummy, None) == -2
