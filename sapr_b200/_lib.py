"""ctypes binding of libsaprb200.so (the C ABI declared in include/sapr_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is
present when a context is created, this module raises.  PyTorch is used only to
own device memory and streams (tensor hand-off via ``data_ptr()``).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libsaprb200.so")

FP32, FP64, FP32_SIMT = 0, 1, 2
EMIT_DIAG, EMIT_SAPR = 0, 1
TOPO_ENTRY_EXIT, TOPO_DENSE = 0, 1
E_SHORT = -5

_vp, _i32, _i64, _dbl = C.c_void_p, C.c_int, C.c_int64, C.c_double


class MfccParams(C.Structure):
    _fields_ = [("sample_rate", C.c_int), ("n_fft", C.c_int), ("win_length", C.c_int), ("hop_length", C.c_int),
                ("n_mels", C.c_int), ("n_mfcc", C.c_int), ("center", C.c_int), ("mel_slaney", C.c_int),
                ("log_db", C.c_int), ("top_db", C.c_float), ("preemph", C.c_float), ("fmin", C.c_float),
                ("fmax", C.c_float)]


# name -> (restype, argtypes); mirrors include/sapr_b200.h one to one
SIGNATURES = {
    "sapr_version": (_i32, []),
    "sapr_ctx_create": (_i32, [_i32, _vp, C.POINTER(_vp)]),
    "sapr_ctx_destroy": (_i32, [_vp]),
    "sapr_last_error": (C.c_char_p, [_vp]),
    "sapr_launch_count": (_i64, [_vp]),
    "sapr_sync": (_i32, [_vp]),
    "sapr_profile": (_i32, [_vp, _i32]),
    "sapr_profile_read": (_i32, [_vp, _i32, C.POINTER(_dbl), C.POINTER(_i64)]),
    "sapr_models_create": (_i32, [_vp, _i32, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "sapr_models_destroy": (_i32, [_vp]),
    "sapr_models_set": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "sapr_models_get": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "sapr_init_stats": (_i32, [_vp, _vp, _i32, _vp, _i32, _i32, _vp, _vp]),
    "sapr_viterbi": (_i32, [_vp, _vp, _vp, _i32, _vp, _i32, _i64, _i32, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "sapr_debug_tc_emission": (_i32, [_vp, _vp, _vp, _i32, _vp, _i32, _i64, _i32, _vp, C.POINTER(_i32)]),
    "sapr_viterbi_host": (_i32, [_vp, _vp, _vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "sapr_stats_stride": (_i64, [_i32, _i32]),
    "sapr_estep": (_i32, [_vp, _vp, _vp, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "sapr_mstep": (_i32, [_vp, _vp, _vp, _vp]),
    "sapr_emission": (_i32, [_vp, _vp, _i32, _vp, _i32, _i32, _vp]),
    "sapr_forward": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "sapr_backward": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "sapr_gamma": (_i32, [_vp, _i32, _vp, _vp, _i32, _vp]),
    "sapr_xi": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp]),
    "sapr_decode_mat": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _vp]),
    "sapr_update_A": (_i32, [_vp, _vp, _i32, _vp, _vp]),
    "sapr_update_B": (_i32, [_vp, _vp, _i32, _vp, _i32, _i64, _vp, _dbl]),
    "sapr_estep_compat": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _i64, _vp, _vp, _vp, _vp]),
    "sapr_decode_compat": (_i32, [_vp, _vp, _i32, _vp, _i32, _i32, _i32, _vp, _vp]),
    "sapr_hl_score": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _i64, _vp]),
    "sapr_ergodic_score": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _i32, _vp]),
    "sapr_score_words": (_i32, [_vp, _vp, _vp, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp]),
    "sapr_hl_decode": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _i64, _vp, _vp]),
    "sapr_hl_stats_len": (_i64, [_i32, _i32]),
    "sapr_hl_estep": (_i32, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _i64, _vp, _vp]),
    "sapr_hl_mstep": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "sapr_viterbi_flagged": (_i32, [_vp, _vp]),
    "sapr_confusion": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "sapr_comm_unique_id": (_i32, [_vp]),
    "sapr_comm_init_rank": (_i32, [_vp, _vp, _i32, _i32, _vp]),
    "sapr_stats_allreduce": (_i32, [_vp, _vp, _vp, _i64]),
    "sapr_comm_destroy": (_i32, [_vp]),
    "sapr_mfcc_num_frames": (_i64, [C.POINTER(MfccParams), _i64]),
    "sapr_mfcc": (_i32, [_vp, C.POINTER(MfccParams), _vp, _vp, _i32, _vp, _i32, _vp]),
}

_lib = None
_lock = threading.Lock()


class SaprError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libsaprb200 error {code}: {msg}")
        self.code = code


def load():
    """Load libsaprb200.so; raises if it has not been built (no fallback path exists)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(SO_PATH):
                raise ImportError(
                    f"{SO_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "or `make -C sapr_b200/csrc`. sapr_b200 has no CPU fallback.")
            lib = C.CDLL(SO_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
            _lib = lib
    return _lib


class Context:
    """One per (device, stream).  Not thread-safe; multi-GPU = one Context per process/device."""

    def __init__(self, device=None):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("sapr_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = load()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        torch.cuda.set_device(self.device)
        self.stream = torch.cuda.current_stream(self.device)
        h = _vp()
        rc = self.lib.sapr_ctx_create(self.device.index, _vp(self.stream.cuda_stream), C.byref(h))
        if rc != 0:
            raise SaprError(rc, "sapr_ctx_create failed")
        self.h = h

    def check(self, rc):
        if rc != 0:
            raise SaprError(rc, self.lib.sapr_last_error(self.h).decode())

    def launches(self) -> int:
        return int(self.lib.sapr_launch_count(self.h))

    def sync(self):
        self.check(self.lib.sapr_sync(self.h))

    def viterbi_flagged(self) -> int:
        """Utterances the last fp32 Viterbi or word-scoring call flagged as word near-ties and re-decoded in float64."""
        n = _i64(0)
        self.check(self.lib.sapr_viterbi_flagged(self.h, C.byref(n)))
        return int(n.value)

    def profile(self, enable: bool):
        self.check(self.lib.sapr_profile(self.h, int(enable)))

    def profile_read(self, which: int):
        """(summed device ms, launches) of kernel class `which` since profile(True)."""
        ms, n = _dbl(0.0), _i64(0)
        self.check(self.lib.sapr_profile_read(self.h, which, C.byref(ms), C.byref(n)))
        return ms.value, int(n.value)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.sapr_ctx_destroy(self.h)
                self.h = None
        except Exception:
            pass


_default_ctx = {}


def default_context(device=None) -> Context:
    import torch

    idx = torch.cuda.current_device() if (device is None and torch.cuda.is_available()) else device
    key = (os.getpid(), idx)
    if key not in _default_ctx:
        _default_ctx[key] = Context(idx)
    return _default_ctx[key]


def ptr(t):
    """data_ptr of a torch tensor / numpy array as c_void_p (None -> NULL)."""
    if t is None:
        return _vp(0)
    if hasattr(t, "data_ptr"):
        return _vp(t.data_ptr())
    return _vp(t.ctypes.data)
