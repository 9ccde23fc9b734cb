"""ctypes binding of libavctc_b200.so (the C ABI declared in include/avctc_b200.h).

There is NO CPU fallback: if the shared library is missing or a call fails, a RuntimeError is raised
(the reference trainer's `except Exception: continue`, /root/reference/model/trainer.py:162-164, then
behaves as it does for a failing PyTorch op).
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libavctc_b200.so")
_lib = None

F32, BF16 = 0, 1
REDUCTION = {"none": 0, "mean": 1, "sum": 2}

_vp, _i, _i64, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_size_t
_d, _u64 = ctypes.c_double, ctypes.c_uint64

# name -> (restype, argtypes); must list every symbol include/avctc_b200.h declares
SIGNATURES = {
    "avctc_version": (ctypes.c_char_p, []),
    "avctc_status_string": (ctypes.c_char_p, [_i]),
    "avctc_set_tuning": (_i, [ctypes.c_char_p, _i]),
    "avctc_ctc_workspace_bytes": (_sz, [_i, _i, _i]),
    "avctc_ctc_forward": (_i, [_vp, _i, _i64, _i64, _i, _i, _i, _vp, _i64, _vp, _vp, _vp, _i, _i, _i,
                               _vp, _vp, _sz, _vp]),
    "avctc_ctc_reduce": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "avctc_ctc_backward": (_i, [_vp, _i, _i64, _i64, _i, _i, _i, _vp, _i64, _vp, _vp, _vp, _i, _i, _i, _i,
                                _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "avctc_ctc_forward_backward": (_i, [_vp, _i, _i64, _i64, _i, _i, _i, _vp, _i64, _vp, _vp, _vp, _i, _i, _i, _i,
                                        _vp, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "avctc_ctc_scale_grad": (_i, [_vp, _i, _i, _i, _i, _vp, _i64, _vp]),
    "avctc_ctc_align_supported": (_i, [_i, _i]),
    "avctc_ctc_align": (_i, [_vp, _i, _i64, _i64, _i, _i, _i, _vp, _i64, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "avctc_beam_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "avctc_beam_route": (_i, [_i, _i, _i, _i]),
    "avctc_beam_search": (_i, [_vp, _i64, _i64, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "avctc_ctc_prefix_beam_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "avctc_ctc_prefix_beam": (_i, [_vp, _i64, _i64, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "avctc_ctc_prefix_beam_lm": (_i, [_vp, _i64, _i64, _i, _i, _i, _vp, _i, _i, _i, _vp, _d, _d, _vp, _vp, _vp, _vp,
                                      _vp, _vp, _vp, _sz, _vp]),
    "avctc_ctc_prefix_beam_biased": (_i, [_vp, _i64, _i64, _i, _i, _i, _vp, _i, _i, _i, _vp, _d, _d, _vp, _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "avctc_gemm_bf16": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, ctypes.c_longlong, ctypes.c_longlong,
                             ctypes.c_longlong, _vp, _i, ctypes.c_float, _i, _vp]),
    "avctc_resample_workspace_bytes": (_sz, [_i, _i]),
    "avctc_resample_forward": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "avctc_resample_backward": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "avctc_softmax_forward": (_i, [_vp, _vp, ctypes.c_longlong, _i, _i, _vp]),
    "avctc_softmax_backward": (_i, [_vp, _vp, _vp, ctypes.c_longlong, _i, _i, _vp]),
    "avctc_colsum": (_i, [_vp, _i, ctypes.c_longlong, _i, ctypes.c_longlong, _vp, _i, _vp]),
    "avctc_log_softmax_forward": (_i, [_vp, _i, _vp, _i, ctypes.c_longlong, _i, _vp]),
    "avctc_log_softmax_backward": (_i, [_vp, _vp, _i, _vp, ctypes.c_longlong, _i, ctypes.c_longlong, _vp]),
    "avctc_ctc_head_forward": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp]),
    "avctc_ctc_head_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "avctc_attention_forward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "avctc_attention_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "avctc_fusion_workspace_bytes": (_sz, [_i] * 8),
    "avctc_fusion_forward": (_i, [_vp, _vp, _i, _vp] + [_vp] * 10 + [_i] * 7 + [_vp, _i, _vp, _vp, _vp, _sz, _i, _vp, _sz,
                                  _vp, _sz, _vp]),
    "avctc_fusion_backward": (_i, [_vp, _i, _vp] + [_i] * 7 + [_vp] * 10 + [_vp, _vp, _i, _vp, _sz, _vp, _sz, _vp, _sz, _i,
                                   _vp]),
    "avctc_bilstm_workspace_bytes": (_sz, [_i] * 5),
    "avctc_bilstm_forward": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _i, _vp]),
    "avctc_bilstm_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    "avctc_infonce_workspace_bytes": (_sz, [_i, _i]),
    "avctc_infonce_forward": (_i, [_vp, _i, ctypes.c_longlong, _vp, _i, _i, ctypes.c_float, ctypes.c_float,
                                   ctypes.c_float, _vp, _vp, _sz, _vp]),
    "avctc_infonce_backward": (_i, [_vp, _i, _i, ctypes.c_float, ctypes.c_float, ctypes.c_float, _vp, _vp, _i,
                                    ctypes.c_longlong, _vp, _sz, _vp]),
    "avctc_visual_frontend_ctas": (_i, [_i, _i, _i, _i]),
    "avctc_visual_frontend": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "avctc_bn_stats_ctas": (_i, [ctypes.c_longlong, _i]),
    "avctc_bn_stats": (_i, [_vp, ctypes.c_longlong, _i, _vp, _i, _vp]),
    "avctc_bn_finalize": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, ctypes.c_float, ctypes.c_float, _i, _vp, _vp]),
    "avctc_visual_frontend_pool": (_i, [_vp, ctypes.c_longlong, _i, _i, _vp, _vp, _vp, _vp]),
    "avctc_bn_act": (_i, [_vp, ctypes.c_longlong, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp]),
    "avctc_w2v_workspace_bytes": (_sz, [ctypes.c_longlong, _i, _i, _i]),
    "avctc_w2v_dropout_increment": (ctypes.c_longlong, [ctypes.c_longlong, _i, _i, _d, _d, _d, _i]),
    "avctc_w2v_dropout": (_i, [_vp, ctypes.c_longlong, _d, _u64, _u64, _vp, _vp]),
    "avctc_w2v_attn_in_forward": (_i, [_vp, ctypes.c_longlong, _i, _vp, _vp, ctypes.c_float, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _sz, _vp]),
    "avctc_w2v_attn_in_backward": (_i, [_vp, _vp, _vp, _vp, ctypes.c_longlong, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _sz, _vp, _sz, _vp]),
    "avctc_w2v_attn_out_ffn_forward": (_i, [_vp, _vp, ctypes.c_longlong, _i, _i, _vp, _vp, _vp, _vp, ctypes.c_float,
                                            _vp, _vp, _vp, _vp, _d, _d, _d, _i, _u64, _u64, _vp, _vp, _sz, _vp]),
    "avctc_w2v_attn_out_ffn_backward": (_i, [_vp, _vp, ctypes.c_longlong, _i, _i, _vp, _vp, _vp, _vp, _d, _d, _d, _i,
                                             _u64, _u64, _vp, _vp] + [_vp] * 8 + [_vp, _sz, _vp, _sz, _vp]),
}


class GemmOperand(ctypes.Structure):
    """Mirror of avctc_gemm_operand (include/avctc_b200.h)."""
    _fields_ = [("ptr", ctypes.c_void_p), ("rows", ctypes.c_longlong), ("kdim", ctypes.c_longlong),
                ("zdim", ctypes.c_longlong), ("ld", ctypes.c_longlong), ("zstride", ctypes.c_longlong),
                ("k_outer", _i), ("k_inner", _i), ("r_outer", _i), ("r_inner", _i), ("z_outer", _i),
                ("z_inner", _i), ("mn_major", _i)]


class NgramLMDesc(ctypes.Structure):
    """Mirror of avctc_ngram_lm (include/avctc_b200.h)."""
    _fields_ = [("order", _i), ("num_words", _i), ("bos", _i), ("eos", _i), ("map_len", _i),
                ("token_word", ctypes.c_void_p), ("unigram", ctypes.c_void_p), ("table", ctypes.c_void_p * 4),
                ("capacity", ctypes.c_uint64 * 4)]


class ContextGraphDesc(ctypes.Structure):
    """Mirror of avctc_context_graph (include/avctc_b200.h)."""
    _fields_ = [("num_nodes", _i), ("alphabet", _i), ("token_sym", ctypes.c_void_p), ("map_len", _i),
                ("delta", ctypes.c_void_p), ("node", ctypes.c_void_p)]


# kernels launched by each entry point (bench.py reports "gpu_launches" from this table); CTC forward / backward with a
# workspace = the probability-domain kernel + its guarded log-domain twin (which exits at once unless the range guard tripped)
KERNELS = {"avctc_ctc_forward": 2, "avctc_ctc_reduce": 1, "avctc_ctc_backward": 2, "avctc_ctc_forward_backward": 5, "avctc_ctc_scale_grad": 1, "avctc_ctc_align": 1, "avctc_beam_search": 2,
           "avctc_ctc_prefix_beam": 2, "avctc_ctc_prefix_beam_lm": 2, "avctc_ctc_prefix_beam_biased": 2,
           "avctc_gemm_bf16": 1, "avctc_resample_forward": 2, "avctc_resample_backward": 1, "avctc_softmax_forward": 1,
           "avctc_softmax_backward": 1, "avctc_colsum": 1, "avctc_log_softmax_forward": 1,
           "avctc_log_softmax_backward": 1, "avctc_infonce_forward": 4, "avctc_infonce_backward": 2,
           "avctc_ctc_head_forward": 1, "avctc_ctc_head_backward": 3, "avctc_attention_forward": 1, "avctc_attention_backward": 1, "avctc_fusion_forward": 7, "avctc_fusion_backward": 8,
           "avctc_bilstm_forward": 7, "avctc_bilstm_backward": 20, "avctc_visual_frontend": 1, "avctc_bn_stats": 1,
           "avctc_bn_finalize": 1, "avctc_visual_frontend_pool": 1, "avctc_bn_act": 1, "avctc_w2v_dropout": 1,
           "avctc_w2v_attn_in_forward": 2, "avctc_w2v_attn_out_ffn_forward": 6, "avctc_w2v_attn_in_backward": 3,
           "avctc_w2v_attn_out_ffn_backward": 6}
# wav2vec2 layer backward: 2 more kernels (bias / LayerNorm gradient reductions) when the weight-gradient pointer at this
# argument index is set
_WGRAD_ARG = {"avctc_w2v_attn_in_backward": 9, "avctc_w2v_attn_out_ffn_backward": 17}
launch_count = 0


class _Counted:
    """Thin proxy over the CDLL that counts kernel launches per entry point."""

    def __init__(self, cdll):
        object.__setattr__(self, "_cdll", cdll)

    def __getattr__(self, name):
        fn = getattr(self._cdll, name)
        n = KERNELS.get(name, 0)
        if n == 0:
            return fn

        if name == "avctc_beam_search":         # 1 kernel on the fused / single-kernel routes, 2 on the two-phase route
            route = self._cdll.avctc_beam_route

            def call(*a):
                global launch_count
                launch_count += 2 if route(a[3], a[4], a[5], a[7]) == 2 else 1
                return fn(*a)
        elif name in _WGRAD_ARG:
            arg = _WGRAD_ARG[name]

            def call(*a):
                global launch_count
                launch_count += n + (2 if a[arg] else 0)
                return fn(*a)
        else:
            def call(*a):
                global launch_count
                launch_count += n
                return fn(*a)
        object.__setattr__(self, name, call)
        return call


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback for the AV-CTC hot path.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = _Counted(L)
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().avctc_status_string(int(status)).decode()
        raise RuntimeError(f"{what} failed: {msg} (status {status})")


def dtype_enum(t) -> int:
    import torch
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise RuntimeError(f"unsupported dtype {t.dtype}: the sm_100a kernels take float32 or bfloat16")


def stream_ptr(device) -> int:
    """cudaStream_t of torch's CURRENT stream on `device` (what every kernel of the library is enqueued on).  The raw
    C accessor: torch.cuda.current_stream() builds a Python Stream object per call (~8 us x ~26 calls per hot-path step)."""
    import torch
    idx = device.index
    if idx is None:
        idx = torch.cuda.current_device()
    return torch._C._cuda_getCurrentRawStream(idx)


class _NoSwitch:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NO_SWITCH = _NoSwitch()


def device_guard(device):
    """`with device_guard(dev):` = torch.cuda.device(dev), without the two device switches (and ~8 us of Python) when
    `dev` already is the current device — the case for every call of a one-process-per-GPU job."""
    import torch
    idx = device.index
    if idx is None or idx == torch.cuda.current_device():
        return _NO_SWITCH
    return torch.cuda.device(device)


def require_cuda(t, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the AV-CTC hot path has no CPU implementation "
                           "(the CPU restatement under oracle/ is test infrastructure only)")


_PY_TUNING = {"lstm_custom": 1}


def tuning_enabled(key: str) -> bool:
    """Host-side switches of the Python layer (e.g. lstm_custom=0 routes temporal_model to nn.LSTM / cuDNN)."""
    return bool(_PY_TUNING.get(key, 1))


def set_py_tuning(key: str, value: int) -> None:
    _PY_TUNING[key] = int(value)


def set_tuning(key: str, value: int) -> None:
    check(lib().avctc_set_tuning(key.encode(), int(value)), f"avctc_set_tuning({key})")
