"""ctypes binding of libllamarec_b200.so (the C ABI declared in include/llamarec_b200.h).

The library is built in-tree (llamarec_b200/lib/) by `make -C llamarec_b200/csrc` or
`__graft_entry__.build()`.  There is no CPU fallback: a missing library raises at first use.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libllamarec_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "llamarec_b200.h")

# name -> (restype, argtypes); must list every symbol the header declares
# (tests/test_cabi_symbols.py parses the header and checks this table and the .so against it).
SIGNATURES = {
    "lrb_last_error": (c_char_p, []),
    "lrb_version": (c_int, []),
    "lrb_device_info": (c_int, [POINTER(c_int), POINTER(c_int)]),
    "lrb_bias_blk_bytes": (c_size_t, [c_int64]),
    "lrb_prepare_table": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "lrb_excl_stride": (c_int, [c_int]),
    "lrb_prepare_sequences": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p]),
    "lrb_encoder_weight_floats": (c_size_t, [c_int]),
    "lrb_encode_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "lrb_encode_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "lrb_score_topk_slots": (c_int, [c_int, c_int64, c_int, POINTER(c_int)]),
    "lrb_score_scratch_bytes": (c_size_t, [c_int]),
    "lrb_score_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p,
                               c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "lrb_score_dense": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_int64,
                                c_void_p]),
    "lrb_merge_metrics": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_int64, c_int,
                                  c_int, c_int, c_void_p, POINTER(ctypes.c_int32), c_int, c_void_p, c_void_p,
                                  c_int64, c_void_p, c_void_p, c_void_p]),
    "lrb_ce_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "lrb_ce_loss_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p,
                                c_void_p, c_size_t, c_void_p]),
    "lrb_train_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "lrb_train_step": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                               c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "lrb_train_step_dropout": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p,
                                       c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_size_t, c_void_p, c_float, c_float, c_float, c_uint64]),
    "lrb_dropout_mask": (c_int, [c_uint64, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "lrb_peer_push": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "lrb_merge_metrics_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_int64,
                                          c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p]),
    "lrb_verbalizer_from_logits": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                           c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "lrb_verbalizer_score": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p, c_int, c_int,
                                     c_int, c_int, c_void_p, c_void_p, c_void_p]),
}

_lib = None


class LrbError(RuntimeError):
    """A non-zero return code from the C ABI (code > 0: cudaError_t, code < 0: LRB_ERR_*)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"llamarec_b200 error {code}: {message}")
        self.code = code


def load() -> ctypes.CDLL:
    """Loads the shared library once; raises ImportError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C llamarec_b200/csrc` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
                "llamarec_b200 has no CPU or PyTorch fallback for its kernels.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().lrb_last_error()
        raise LrbError(rc, msg.decode("utf-8", "replace") if msg else "")


def ptr(t) -> int | None:
    """Device (or host) address of a torch tensor, None for a missing optional argument."""
    if t is None:
        return None
    assert t.is_contiguous(), "llamarec_b200 kernels take contiguous tensors"
    return t.data_ptr()


def stream_handle(device=None) -> int | None:
    """Handle of torch's current stream on `device` (default: the current device)."""
    import torch
    return torch.cuda.current_stream(device).cuda_stream or None


class on_device:
    """Context manager: makes the device that owns `tensor` current for the enclosed C-ABI calls (the kernels
    launch on the current device's stream; pointers of another device would fault or go through peer access)."""

    def __init__(self, tensor_or_device):
        import torch
        dev = tensor_or_device.device if hasattr(tensor_or_device, "device") else torch.device(tensor_or_device)
        if dev.type != "cuda":
            raise RuntimeError("llamarec_b200 has no CPU path: tensors must live on a CUDA device")
        self._guard = torch.cuda.device(dev)

    def __enter__(self):
        self._guard.__enter__()
        return self

    def __exit__(self, *exc):
        return self._guard.__exit__(*exc)
