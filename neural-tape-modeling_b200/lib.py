"""ctypes binding of libntm_b200.so -- every symbol include/ntm_b200.h declares, nothing else.

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

PKG = os.path.dirname(os.path.abspath(__file__))
# NTM_B200_LIB: developer override to A/B another BUILD of the same library (never a different implementation)
LIB_PATH = os.environ.get("NTM_B200_LIB") or os.path.join(PKG, "libntm_b200.so")

MODE_FP32, MODE_TF32, MODE_BF16, MODE_TF32X3, MODE_F16 = 0, 1, 2, 3, 4
MODE_F16X3 = MODE_TF32X3
# "f16x3" (aliases "strict", "tf32x3"): fp32-grade result on tensor cores, see include/ntm_b200.h NTM_MODE_F16X3
MODES = {"fp32": MODE_FP32, "tf32": MODE_TF32, "bf16": MODE_BF16, "f16x3": MODE_F16X3, "strict": MODE_F16X3,
         "tf32x3": MODE_F16X3, "f16": MODE_F16}
Q_VERSION, Q_DEVICE_COUNT, Q_SM_COUNT, Q_MODE_MASK, Q_KERNEL_LAUNCHES, Q_LAST_KERNEL = 0, 1, 2, 3, 4, 5
KERNEL_NAMES = {0: "gru_fp32_kernel (CUDA-core FFMA)", 1: "gru_mma_kernel (warp-level mma.sync)",
                3: "gru_tcs_kernel (tcgen05 + TMEM, stream-major)",
                4: "gru_mma4_kernel (warp-level mma.sync, lean 4-stream form)"}
E_DELAY = -5
E_CLOSED = -7

_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_int = ctypes.c_int

# name -> (restype, argtypes): must list exactly the functions of include/ntm_b200.h
SIGNATURES = {
    "ntm_query": (_int, [_int]),
    "ntm_strerror": (ctypes.c_char_p, [_int]),
    "ntm_last_cuda_error": (_int, []),
    "ntm_gru_prepare": (_int, [_vp] * 6 + [_int, _int, ctypes.POINTER(_vp)]),
    "ntm_destroy": (None, [_vp]),
    "ntm_retain": (_int, [_vp]),
    "ntm_release": (None, [_vp]),
    "ntm_handle_set_tuning": (_int, [_vp, _int, _int]),
    "ntm_handle_last_kernel": (_int, [_vp]),
    "ntm_esr_sums_rows": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _int, _vp, _int, _vp]),
    "ntm_gru_forward": (_int, [_vp, _int, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _int, _vp]),
    "ntm_diffdel_forward": (_int, [_vp, _int, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp,
                                   _i64, _i64, _i64, _int, _int, _vp]),
    "ntm_delay_forward": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _i64, _int, _int, _vp]),
    "ntm_delay_check": (_int, [_vp, _i64, _i64, _i64, _i64, _int, _vp]),
    "ntm_gru_predict_host": (_int, [_vp, _int, _vp, _vp, _vp, _i64, _i64, _int, _i64]),
    "ntm_gru_predict_host_f16": (_int, [_vp, _int, _vp, _vp, _vp, _i64, _i64, _int, _i64]),
    "ntm_diffdel_predict_host": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _i64]),
    "ntm_set_tuning": (_int, [_int, _int]),
    "ntm_rt_open": (_int, [_vp, _int, _vp, _i64, _i64, _int, _int, ctypes.POINTER(_vp)]),
    "ntm_rt_process": (_int, [_vp, _vp, _vp]),
    "ntm_rt_close": (_int, [_vp, _vp]),
    "ntm_rt_diffdel_open": (_int, [_vp, _int, _vp, _vp, _i64, _i64, _i64, _int, _int, _int, ctypes.POINTER(_vp)]),
    "ntm_rt_diffdel_process": (_int, [_vp, _vp, _vp, _vp, _vp]),
    "ntm_rt_diffdel_close": (_int, [_vp, _vp, _vp]),
    "ntm_esr_sums": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _int, _vp, _int, _vp]),
    "ntm_mrstft_sums_rows": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _int, _vp, _vp, _vp, _vp, _int, _vp]),
}

_lib = None


def load():
    """dlopen the in-tree library (build it with `python neural-tape-modeling_b200/build.py`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it first (python neural-tape-modeling_b200/build.py); "
                               "ntm_b200 has no fallback path")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


TORCH_LIB_PATH = os.environ.get("NTM_B200_TORCH_LIB") or os.path.join(PKG, "ntm_b200_torch.so")
_ops = None


def ops():
    """torch.ops.ntm -- the PyTorch C++ extension (csrc/torch_binding.cpp) over the same C ABI.  No fallback either."""
    global _ops
    if _ops is None:
        import torch
        if not os.path.exists(TORCH_LIB_PATH):
            raise RuntimeError(f"{TORCH_LIB_PATH} is missing: build it first (python neural-tape-modeling_b200/build.py); "
                               "ntm_b200 has no fallback path")
        load()                                   # the extension resolves libntm_b200.so next to itself ($ORIGIN rpath)
        torch.ops.load_library(TORCH_LIB_PATH)
        _ops = torch.ops.ntm
    return _ops


def check(rc):
    """0 -> None; NTM_EDELAY -> AssertionError (the reference asserts, code/model.py:283); else RuntimeError."""
    if rc == 0:
        return
    msg = load().ntm_strerror(rc).decode()
    if rc == E_DELAY:
        raise AssertionError(msg)
    raise RuntimeError(f"ntm_b200: {msg} (code {rc})")


def query(what):
    return load().ntm_query(what)
