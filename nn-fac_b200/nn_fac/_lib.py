"""ctypes binding of ``libnnfac_b200.so`` (C ABI declared in ``include/nnfac_b200.h``).

There is no CPU fallback: importing this module without the built library, or calling any
operator without a CUDA device, raises.  PyTorch is used for device memory and streams only.
"""
import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NNFAC_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libnnfac_b200.so")

F32, F64 = 0, 1
ERR_UNSUPPORTED = -3
HALS_NORMALIZE, HALS_NONZERO, HALS_NO_TC = 1, 2, 4

_c = ctypes
_P, _I64, _INT, _DBL, _U32 = _c.c_void_p, _c.c_int64, _c.c_int, _c.c_double, _c.c_uint

# name -> argument ctypes (every function returns int unless listed in _RESTYPES)
SIGNATURES = {
    "nnfac_abi_version": [],
    "nnfac_last_error": [],
    "nnfac_ctx_create": [_INT, _c.POINTER(_P)],
    "nnfac_ctx_destroy": [_P],
    "nnfac_ctx_sm_count": [_P],
    "nnfac_ctx_launch_count": [_P],
    "nnfac_ctx_board_export": [_P, _P],
    "nnfac_ctx_board_attach": [_P, _INT, _INT, _P],
    "nnfac_ctx_collective": [_P, _INT, _P],
    "nnfac_ctx_sweep_variant": [_P, _INT],
    "nnfac_xchg_create": [_P, _I64, _I64, _c.POINTER(_P)],
    "nnfac_xchg_export": [_P, _P],
    "nnfac_xchg_attach": [_P, _INT, _INT, _P],
    "nnfac_xchg_destroy": [_P],
    "nnfac_xchg_ptr": [_P, _INT],
    "nnfac_xchg_post": [_P, _INT, _P],
    "nnfac_xchg_post_tail": [_P, _P, _INT, _I64, _I64, _P],
    "nnfac_xchg_pull_tail": [_P, _INT, _P, _I64, _INT, _I64, _I64, _INT, _P],
    "nnfac_nmf_plan_set_factor_pulled": [_P, _INT, _P, _I64, _I64, _P, _I64, _P],
    "nnfac_hals_nnls": [_P, _INT, _P, _I64, _P, _I64, _P, _I64, _INT, _I64, _INT, _DBL, _DBL, _U32, _P, _P],
    "nnfac_hals_solve_f32": [_P, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _INT, _I64, _INT, _DBL, _DBL, _P, _P],
    "nnfac_hals_solve_slabs_f32": [_P, _P, _I64, _INT, _I64, _INT, _P, _P, _I64, _P, _I64, _P, _I64, _INT, _I64, _INT, _DBL, _DBL, _P, _P],
    "nnfac_xchg_inbox_mu_apply": [_P, _I64, _INT, _I64, _I64, _I64, _P, _I64, _INT, _I64, _I64, _DBL, _I64, _P],
    "nnfac_nmf_plan_set_push": [_P, _P, _I64, _I64, _c.POINTER(_INT), _c.POINTER(_I64)],
    "nnfac_reduce_slabs_f32": [_P, _P, _I64, _INT, _INT, _INT, _I64, _P, _I64, _P],
    "nnfac_gemm_strided": [_P, _INT, _P, _I64, _I64, _P, _I64, _I64, _I64, _I64, _P, _I64, _I64, _I64, _I64,
                           _I64, _I64, _I64, _I64, _I64, _P],
    "nnfac_gram": [_P, _INT, _P, _I64, _P, _I64, _INT, _I64, _P],
    "nnfac_mu_terms": [_P, _INT, _DBL, _P, _P, _P, _P, _I64, _P],
    "nnfac_mu_apply": [_P, _INT, _P, _P, _P, _P, _P, _INT, _I64, _I64, _DBL, _DBL, _P],
    "nnfac_beta_divergence": [_P, _INT, _DBL, _P, _P, _I64, _P, _P],
    "nnfac_sq_diff": [_P, _INT, _P, _P, _I64, _P, _P],
    "nnfac_dot": [_P, _INT, _P, _P, _I64, _P, _P],
    "nnfac_row_sums": [_P, _INT, _P, _I64, _I64, _I64, _P, _P],
    "nnfac_norm1": [_P, _INT, _P, _I64, _I64, _I64, _P, _P],
    "nnfac_transpose": [_P, _INT, _P, _I64, _P, _I64, _I64, _I64, _P],
    "nnfac_khatri_rao": [_P, _INT, _P, _P, _I64, _P, _I64, _I64, _P],
    "nnfac_hadamard": [_P, _INT, _P, _P, _P, _I64, _P],
    "nnfac_axpby": [_P, _INT, _P, _DBL, _P, _DBL, _P, _I64, _P],
    "nnfac_normalize_rows": [_P, _INT, _P, _I64, _I64, _I64, _P],
    "nnfac_core_pg_step": [_P, _INT, _P, _P, _P, _I64, _DBL, _DBL, _DBL, _P, _P],
    "nnfac_core_pg_step_dev": [_P, _INT, _P, _P, _P, _I64, _DBL, _P, _P],
    "nnfac_core_pg_step3": [_P, _INT, _P, _P, _P, _P, _P, _INT, _INT, _INT, _P, _DBL, _DBL, _INT, _DBL, _P, _P],
    "nnfac_philox_uniform": [_P, _P, _I64, _I64, _I64, _I64, _I64, _c.c_uint64, _U32, _DBL, _INT, _P],
    "nnfac_nmf_plan_create": [_P, _I64, _I64, _INT, _c.POINTER(_P)],
    "nnfac_nmf_plan_bytes": [_P, _I64, _I64, _INT, _c.POINTER(_c.c_size_t)],
    "nnfac_nmf_plan_create_in": [_P, _I64, _I64, _INT, _P, _c.c_size_t, _P, _c.POINTER(_P)],
    "nnfac_nmf_plan_bytes_sided": [_P, _I64, _I64, _INT, _INT, _c.POINTER(_c.c_size_t)],
    "nnfac_nmf_plan_create_sided": [_P, _I64, _I64, _INT, _INT, _P, _c.c_size_t, _P, _c.POINTER(_P)],
    "nnfac_nmf_plan_bytes_planes": [_P, _I64, _I64, _INT, _INT, _INT, _c.POINTER(_c.c_size_t)],
    "nnfac_nmf_plan_create_planes": [_P, _I64, _I64, _INT, _INT, _INT, _P, _c.c_size_t, _P, _c.POINTER(_P)],
    "nnfac_nmf_plan_view_bytes": [_P, _P, _I64, _I64, _I64, _INT, _c.POINTER(_c.c_size_t)],
    "nnfac_nmf_plan_create_view": [_P, _P, _I64, _I64, _I64, _INT, _P, _c.c_size_t, _P, _c.POINTER(_P)],
    "nnfac_nmf_plan_destroy": [_P],
    "nnfac_nmf_plan_load_x": [_P, _P, _I64, _P],
    "nnfac_nmf_plan_load_x_rows": [_P, _P, _I64, _I64, _I64, _P],
    "nnfac_nmf_plan_load_x_done": [_P, _P],
    "nnfac_nmf_plan_f32_bytes": [_P, _c.POINTER(_c.c_size_t)],
    "nnfac_nmf_plan_enable_f32": [_P, _P, _c.c_size_t, _P],
    "nnfac_nmf_plan_cross": [_P, _INT, _P, _I64, _P, _I64, _P],
    "nnfac_nmf_plan_set_factor": [_P, _INT, _P, _I64, _P],
    "nnfac_nmf_plan_set_factor_gathered": [_P, _INT, _P, _I64, _P, _I64, _P],
    "nnfac_nmf_plan_reduce": [_P, _INT, _P, _I64, _P],
    "nnfac_nmf_plan_reduce_chunked": [_P, _INT, _P, _I64, _INT, _P, _I64, _INT, _P],
    "nnfac_nmf_plan_set_krao": [_P, _P, _I64, _I64, _P, _I64, _I64, _P],
    "nnfac_nmf_plan_set_krao_rows": [_P, _P, _I64, _I64, _P, _I64, _I64, _P],
    "nnfac_nmf_plan_hals_solve": [_P, _INT, _P, _I64, _P, _I64, _P, _I64, _P, _I64, _INT, _DBL, _DBL, _P, _P],
    "nnfac_nmf_plan_fused": [_P, _INT, _INT, _INT, _P, _I64, _P, _P],
    "nnfac_nmf_plan_mu_finish": [_P, _INT, _P, _I64, _P, _DBL, _P, _I64, _P],
    "nnfac_nmf_plan_fused_beta_bytes": [_P, _c.POINTER(_c.c_size_t)],
    "nnfac_nmf_plan_fused_beta": [_P, _INT, _DBL, _INT, _P, _P, _P],
    "nnfac_nmf_plan_mu_finish_beta": [_P, _INT, _P, _I64, _P, _DBL, _DBL, _P, _I64, _P],
    "nnfac_nmf_plan_info": [_P, _INT, _c.POINTER(_INT), _c.POINTER(_INT), _c.POINTER(_INT), _c.POINTER(_INT),
                            _c.POINTER(_INT)],
}
_RESTYPES = {"nnfac_last_error": _c.c_char_p, "nnfac_ctx_launch_count": _I64, "nnfac_xchg_ptr": _P}

_lib = None
_ctxs = {}


class NnfacError(RuntimeError):
    """A call into libnnfac_b200 failed (status < 0); the message comes from nnfac_last_error()."""


def load_library():
    """dlopen the in-tree library and declare every prototype.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `bash nn-fac_b200/build.sh` "
                          "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _RESTYPES.get(name, _INT)
    if lib.nnfac_abi_version() != 1:
        raise ImportError("libnnfac_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(status):
    if status != 0:
        raise NnfacError(f"nnfac status {status}: {load_library().nnfac_last_error().decode()}")


_cuda_ok = None


def device_index(device=None):
    global _cuda_ok
    if _cuda_ok is None:                              # (torch.cuda.is_available() costs microseconds on every call)
        if not torch.cuda.is_available():
            raise NnfacError("nn_fac (B200 build) needs a CUDA device; there is no CPU fallback")
        _cuda_ok = True
    if device is None:
        return torch.cuda.current_device()
    if isinstance(device, torch.device):
        return device.index or 0
    return torch.device(device).index or 0


def ctx(device=None):
    """Per-device nnfac context (workspace + launch limits), created on first use."""
    idx = device_index(device)
    if idx not in _ctxs:
        handle = _P()
        check(load_library().nnfac_ctx_create(idx, ctypes.byref(handle)))
        _ctxs[idx] = handle
    return _ctxs[idx]


def launch_count(device=None):
    return int(load_library().nnfac_ctx_launch_count(ctx(device)))


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr():
    """The current CUDA stream of the current device as a pointer (the raw getter is ~30x cheaper than building a
    torch.cuda.Stream object: the outer loops make a dozen calls per iteration and must stay ahead of the GPU)."""
    if _raw_stream is not None:
        return _P(_raw_stream(torch.cuda.current_device()))
    return _P(torch.cuda.current_stream().cuda_stream)


def code_of(dtype):
    if dtype == torch.float32:
        return F32
    if dtype == torch.float64:
        return F64
    raise NnfacError(f"unsupported dtype {dtype}")


def ptr(t):
    return _P(t.data_ptr()) if t is not None else _P(None)


def to_device(x, dtype, device=None):
    """numpy / torch / sequence -> contiguous CUDA tensor of `dtype` (a copy is always made for numpy)."""
    dev = torch.device("cuda", device_index(device))
    if isinstance(x, torch.Tensor):
        return x.to(device=dev, dtype=dtype).contiguous()
    arr = np.ascontiguousarray(np.asarray(x))
    return torch.from_numpy(arr).to(device=dev, dtype=dtype)


def resolve_dtype(*arrays):
    """Working precision: config.precision, or float64 unless every input is float32 (the reference
    is dtype-preserving)."""
    from . import config
    if config.precision == "fp32":
        return torch.float32
    if config.precision in ("fp64", "fp32x3"):
        return torch.float64
    for a in arrays:
        if a is None:
            continue
        dt = a.dtype
        if dt in (torch.float32, np.float32) or str(dt) == "float32":
            continue
        return torch.float64
    return torch.float32


def as_output(x):
    """A result handed back to the caller (torch tensor or numpy array): float32 under precision "fp32x3", which computes every
    path outside its 3-plane tensor-core NMF in float64; unchanged under the other precisions."""
    from . import config
    if config.precision != "fp32x3":
        return x
    if isinstance(x, torch.Tensor):
        return x if x.dtype == torch.float32 else x.to(torch.float32)
    x = np.asarray(x)
    return x if x.dtype == np.float32 else x.astype(np.float32)


def working_dtype(numel, *arrays):
    """(arithmetic dtype, dtype of the returned arrays): resolve_dtype, except that in "auto" mode a float32 problem of at most
    config.small_problem_elements data elements computes in float64, and that "fp32x3" computes in float64 and returns float32
    wherever its 3-plane tensor-core path does not apply (see nn_fac/config.py)."""
    from . import config
    if config.precision == "fp32x3":
        return torch.float64, torch.float32
    dt = resolve_dtype(*arrays)
    if dt == torch.float32 and config.precision == "auto" and int(numel) <= config.small_problem_elements:
        return torch.float64, torch.float32
    return dt, dt
