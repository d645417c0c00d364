"""ctypes binding of ``libpyro_b200.so`` (the C ABI declared in include/pyro_b200.h).

This is the ONLY place the product path touches native code.  There is no CPU fallback: if the
shared object is missing, or an op is asked to run on a non-CUDA tensor, a ``RuntimeError`` is
raised (reference precedent for loading a native extension lazily with a backend switch:
pyro/distributions/spanning_tree.py:222-258).
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpyro_b200.so")

B2_MAX_DIMS = 8
B2_MAX_PARAMS = 4
B2_F32, B2_F64, B2_I64, B2_U8 = 0, 1, 2, 3
B2_FLAG_ACCUMULATE_SUM = 1
B2_FLAG_GLM_FP32 = 2
B2_FLAG_SITE_LARGE = 4
B2_FLAG_GLM_3XTF32 = 32
FORCE_LARGE_SITE_KERNELS = False   # tests: score small fixtures with the multi-CTA kernels too
B2_ERR_UNSUPPORTED_REDUCTION = -6

# family ids (include/pyro_b200.h)
NORMAL, BERNOULLI_LOGITS, GAMMA, BETA, POISSON, CAUCHY, HALFCAUCHY, EXPONENTIAL, LOGNORMAL, \
    HALFNORMAL, BERNOULLI_PROBS, UNIFORM, KL_NORMAL_NORMAL, KL_GAMMA_GAMMA, NORMAL_RSAMPLE, \
    NORMAL_RSAMPLE_BWD = range(16)
FUSED_DRAW = True         # Normal.rsample draws and scores in one kernel (b2 family 14)
PHILOX_DRAW = True        # ... and generates its noise in that kernel (b2_normal_rsample) instead of torch.randn
RSAMPLE_MAX_N = 65536
EMULATE_RSAMPLE = False   # tests/cpu_emulation.py flips this to exercise the fused-draw host logic on CPU
SITE_SMALL_N = 8192   # B2_SITE_SMALL_N: one-CTA kernel with fused stored-shape gradient reductions
DIRICHLET, CATEGORICAL, MVN_TRIL = 32, 33, 34
MODEL_HIER_NORMAL, MODEL_LOGISTIC = 0, 1
NUTS_SMALL_MAX_D = 64


LATENT_MAX_JOBS = 8
LATENT_MAX_TERMS = 24
LATENT_COMBINE_MAX_N = 32768   # one CTA scores every prior of the step and assembles the loss up to this size
LATENT_LOG_SCALE = 1
LATENT_ACC_OUT0, LATENT_ACC_OUT1 = 2, 4
LATENT_BLOCK = True       # Normal guide sites + Normal priors go through the latent-sites kernels (latent.cu)
LATENT_ACCUMULATE = True  # the draw's backward kernel adds into existing leaf .grad buffers itself
GAMMA_RSAMPLE = True      # Gamma.rsample draws with the own kernel (b2_gamma_rsample) instead of ATen
LAZY_PARAM = True         # positive-constrained parameters are handed out as deferred exp(u) (_lazyparam.py)


class b2_latent_job(ctypes.Structure):
    _fields_ = [("dtype", ctypes.c_int32), ("ndim", ctypes.c_int32), ("flags", ctypes.c_int32),
                ("pad_", ctypes.c_int32),
                ("shape", ctypes.c_int64 * 8),
                ("loc_stride", ctypes.c_int64 * 8), ("scale_stride", ctypes.c_int64 * 8),
                ("prior_loc_stride", ctypes.c_int64 * 8), ("prior_scale_stride", ctypes.c_int64 * 8),
                ("loc", ctypes.c_void_p), ("scale", ctypes.c_void_p), ("prior_loc", ctypes.c_void_p),
                ("prior_scale", ctypes.c_void_p), ("z", ctypes.c_void_p), ("eps", ctypes.c_void_p),
                ("gz", ctypes.c_void_p), ("out0", ctypes.c_void_p), ("out1", ctypes.c_void_p),
                ("c", ctypes.c_double), ("prior_weight", ctypes.c_double)]


class b2_tensor(ctypes.Structure):
    _fields_ = [("ptr", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("ndim", ctypes.c_int32),
                ("shape", ctypes.c_int64 * B2_MAX_DIMS), ("stride", ctypes.c_int64 * B2_MAX_DIMS)]


class b2_model(ctypes.Structure):
    _fields_ = [("model", ctypes.c_int32), ("dtype", ctypes.c_int32), ("J", ctypes.c_int64),
                ("D", ctypes.c_int64), ("data0", ctypes.c_void_p), ("data1", ctypes.c_void_p),
                ("hyper", ctypes.c_double * 4)]


class b2_nuts_lockstep(ctypes.Structure):
    """Mirror of ``b2_nuts_lockstep`` (include/pyro_b200.h): device pointers of the lockstep tree state."""
    _fields_ = [("zL", ctypes.c_void_p), ("rL", ctypes.c_void_p), ("zR", ctypes.c_void_p),
                ("rR", ctypes.c_void_p), ("dir", ctypes.c_void_p), ("gscL", ctypes.c_void_p),
                ("gscR", ctypes.c_void_p), ("minv", ctypes.c_void_p),
                ("minv_chain_stride", ctypes.c_int64), ("rsub", ctypes.c_void_p), ("zs", ctypes.c_void_p),
                ("rck", ctypes.c_void_p), ("sck", ctypes.c_void_p), ("eps", ctypes.c_void_p),
                ("gsc_s", ctypes.c_void_p), ("U", ctypes.c_void_p),
                ("Us", ctypes.c_void_p), ("energy0", ctypes.c_void_p), ("logw_sub", ctypes.c_void_p),
                ("sum_accept", ctypes.c_void_p), ("num_prop", ctypes.c_void_p), ("done", ctypes.c_void_p),
                ("diverged", ctypes.c_void_p), ("take", ctypes.c_void_p), ("num_leapfrogs", ctypes.c_void_p),
                ("rng_counter", ctypes.c_void_p), ("seed", ctypes.c_uint64),
                ("max_delta_energy", ctypes.c_double), ("C", ctypes.c_int64)]


_lib = None
_lib_lock = threading.Lock()

_vp, _i32, _i64, _f64, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t
_tp = ctypes.POINTER(b2_tensor)
_mp = ctypes.POINTER(b2_model)

# name -> (restype, argtypes); also used by the symbol-export test
SIGNATURES = {
    "b2_site_score": (_i32, [_i32, _tp, _tp, _i32, _tp, _f64, _tp, _f64, _f64, _i32, _tp, _vp, _tp,
                             _tp, _vp, _sz, _vp]),
    "b2_site_score_workspace": (_sz, []),
    "b2_event_score": (_i32, [_i32, _tp, _tp, _i32, _i32, _tp, _f64, _tp, _f64, _f64, _i32, _tp,
                              _vp, _tp, _tp, _vp, _sz, _vp]),
    "b2_reduce_to": (_i32, [_tp, _tp, _vp, _sz, _vp]),
    "b2_normal_rsample": (_i32, [_tp, _tp, _i32, ctypes.POINTER(ctypes.c_int64), _vp, _vp, _vp, _vp, _vp]),
    "b2_gamma_rsample": (_i32, [_tp, _tp, _i32, ctypes.POINTER(ctypes.c_int64), _vp, _vp, _vp, _vp]),
    "b2_latent_normal_draw": (_i32, [_vp, _i32, _vp, _vp]),
    "b2_latent_normal_prior": (_i32, [_vp, _i32, _vp]),
    "b2_latent_normal_backward": (_i32, [_vp, _i32, _vp]),
    "b2_latent_normal_prior_combine": (_i32, [_vp, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "b2_elbo_combine": (_i32, [_vp, _vp, _i32, _i32, _vp, _vp]),
    "b2_glm_bernoulli_logits": (_i32, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _f64, _f64, _f64, _i32,
                                       _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "b2_glm_workspace": (_sz, [_i64, _i32, _i32]),
    "b2_clipped_adam": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp]),
    "b2_adagrad_rmsprop": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp]),
    "b2_leapfrog_half_kick_drift": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i32, _vp]),
    "b2_leapfrog_half_kick": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _i32, _vp,
                                     _sz, _vp]),
    "b2_mcmc_workspace": (_sz, [_i64]),
    "b2_potential_grad": (_i32, [_mp, _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "b2_potential_workspace": (_sz, [_mp, _i64]),
    "b2_nuts_small": (_i32, [_mp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _f64, ctypes.c_uint64,
                             _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2_nuts_leaf_vector": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32,
                                   _i32, _vp, _i64, _i64, _i32, _vp, _sz, _vp]),
    "b2_nuts_leaf_hier": (_i32, [_mp, ctypes.POINTER(b2_nuts_lockstep), _i32, _i32, _i32, _i32, _vp, _sz, _vp]),
    "b2_nuts_leaf_hier_workspace": (_sz, [_i64, _i64]),
    "b2_rows_copy_masked": (_i32, [_vp, _vp, _vp, _i64, _i64, _i32, _vp]),
    "b2_nuts_tree_merge": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _sz, _vp]),
    "b2_last_error": (ctypes.c_char_p, [_i32]),
    "b2_version": (_i32, []),
    "b2_launch_count": (_i64, []),
}


def lib():
    """Load (once) and return the native library; raise loudly if it is not built."""
    global _lib
    if _lib is None:
        with _lib_lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "pyro_b200: native library %s is missing. Build it with "
                        "`python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
                L = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(L, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = L
    return _lib


def launch_count():
    return int(lib().b2_launch_count())


class NativeError(RuntimeError):
    pass


def check(code, what):
    if code != 0:
        msg = lib().b2_last_error(code).decode()
        raise NativeError("pyro_b200 native call %s failed: %s (code %d)" % (what, msg, code))


_DTYPES = {torch.float32: B2_F32, torch.float64: B2_F64, torch.int64: B2_I64, torch.bool: B2_U8,
           torch.uint8: B2_U8}


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(
            "pyro_b200: %s needs CUDA tensors (got device %s). The B200 backend has no CPU "
            "path; move the inputs to the GPU." % (what, t.device))


def desc(t, shape=None):
    """b2_tensor view of ``t`` broadcast (without copying) to ``shape``."""
    d = b2_tensor()
    if t is None:
        d.ptr = None
        d.dtype = 0
        d.ndim = len(shape) if shape is not None else 0
        return d
    if type(t) is not torch.Tensor and hasattr(t, "dense"):
        # a storage-less lazy tensor: the caller must materialise it BEFORE the autograd boundary
        raise RuntimeError("pyro_b200: a lazy tensor (%s) reached the native boundary" % type(t).__name__)
    if shape is not None and tuple(t.shape) != tuple(shape):
        t = t.expand(shape)
    nd = t.dim()
    if nd > B2_MAX_DIMS:
        raise ValueError("pyro_b200: tensors with more than %d dims are not supported" % B2_MAX_DIMS)
    d.ptr = t.data_ptr()
    d.dtype = _DTYPES[t.dtype]
    d.ndim = nd
    sh, st = t.shape, t.stride()
    for i in range(nd):
        d.shape[i] = sh[i]
        d.stride[i] = st[i] if sh[i] != 1 else 0
    return d


def capturing():
    """True while the current stream is being captured into a CUDA graph."""
    return torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


# ---- per-(device, stream) zero-initialised reduction workspace --------------------------------
_workspaces = {}
_retired = []


def workspace(device, nbytes=None, tag="reduce"):
    """Reduction scratch of ``device``.  One buffer per device: the fused kernels are stream
    ordered, and eager steps, graph capture and graph replay all issue on one stream at a time;
    running reducing kernels concurrently on two streams of one device is not supported.  The
    library leaves the ticket area zeroed.  ``tag`` separates the ticketed reduction scratch
    ("reduce") from plain scratch areas ("glm", "mcmc") so they never overlap."""
    need = int(lib().b2_site_score_workspace()) if nbytes is None else int(nbytes)
    key = (device.index if device.index is not None else torch.cuda.current_device(), tag)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < need:
        if capturing():
            raise RuntimeError("pyro_b200: workspace must be allocated before CUDA graph capture; "
                               "run one eager step first")
        if ws is not None:
            _retired.append(ws)   # captured CUDA graphs may still hold the old buffer's address
        ws = torch.zeros(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws
