"""ctypes binding of libb200convlstm.so.

The prototypes are read from include/b200_convlstm.h, the single source of truth for the C ABI.
There is deliberately NO fallback: if the library is missing or a call fails, a RuntimeError is
raised (the product path never routes through PyTorch ops or the CPU oracle).
"""
from __future__ import annotations

import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "b200_convlstm.h")
# B200_LIB: developer override to A/B two builds of the library in one GPU session (tools/bench_ops.py)
LIB_PATH = os.environ.get("B200_LIB") or os.path.join(HERE, "libb200convlstm.so")

_CTYPES = {
    "int": ctypes.c_int,
    "long long": ctypes.c_longlong,
    "float": ctypes.c_float,
    "double": ctypes.c_double,
}


def parse_header(path: str = HEADER):
    """Returns {name: (restype, [argtypes])} for every prototype of the header."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"^\s*#.*$", "", src, flags=re.M)
    protos = {}
    for m in re.finditer(r"([\w\s\*]+?)\b(b200_\w+)\s*\(([^)]*)\)\s*;", src):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        restype = ctypes.c_char_p if "char" in ret else ctypes.c_int
        argtypes = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(ctypes.c_void_p)
                else:
                    base = re.sub(r"\bconst\b", "", a).strip()
                    base = " ".join(base.split()[:-1])  # drop the parameter name
                    argtypes.append(_CTYPES[base])
        protos[name] = (restype, argtypes)
    return protos


_lib = None
_protos = None

# C-ABI calls made so far, by entry point (bench.py turns these into its `gpu_launches` claim)
CALLS: dict = {}
# device kernels launched per call of each entry point (memsets are not counted)
KERNELS_PER_CALL = {
    "b200_convlstm_cell_fwd_splitk_tc": 2, "b200_conv_affine_relu_splitk_tc": 2,
    "b200_conv_tc_fwd": 1, "b200_conv_bnstats_tc_fwd": 1, "b200_convT2x2_tc_fwd": 1, "b200_conv_affine_relu_tc_fwd": 1, "b200_convlstm_cell_fwd_tc": 1, "b200_convlstm_seq_fwd_tc": 1, "b200_convlstm_seq_bwd_tc": 1, "b200_wgrad_tc": 1, "b200_conv_simt_fwd": 1,
    "b200_wgrad_simt": 1, "b200_bn_stats": 1, "b200_bn_finalize": 1, "b200_bn_relu_apply": 1,
    "b200_bn_relu_bwd_reduce": 1, "b200_bn_bwd_finalize": 1, "b200_bn_relu_bwd_apply": 1,
    "b200_maxpool2_fwd": 1, "b200_maxpool2_bwd": 1, "b200_bn_relu_apply_pool": 1, "b200_bn_relu_pool_bwd_reduce": 1,
    "b200_bn_relu_pool_bwd_apply": 1, "b200_bn_relu_outconv_fwd": 1, "b200_bn_relu_outconv_bwd_reduce": 2,
    "b200_bn_relu_outconv_bwd_apply": 1, "b200_lstm_gates_fwd": 1, "b200_lstm_gates_bwd": 1,
    "b200_colsum": 2, "b200_wl1_grad_loss_fwd": 2, "b200_wl1_grad_loss_bwd": 1, "b200_denorm_metrics_accum": 1, "b200_sequence_batch": 1, "b200_pack_weight": 1, "b200_unpack_wgrad": 1, "b200_grad_sqnorm_multi": 1, "b200_grad_clip_multi": 1, "b200_adamw_multi": 1, "b200_adamw_pack": 1, "b200_adamw_pack_multi": 1, "b200_outconv_fwd": 1, "b200_outconv_bwd": 5, "b200_shuffle2x2": 1, "b200_strided_copy": 1,
}


def kernel_launches() -> int:
    return sum(KERNELS_PER_CALL.get(k, 1) * v for k, v in CALLS.items())


def lib():
    global _lib, _protos
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -m unet_convlstm_b200.build` "
                "(there is no fallback path)")
        l = ctypes.CDLL(LIB_PATH)
        _protos = parse_header()
        for name, (restype, argtypes) in _protos.items():
            fn = getattr(l, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = l
    return _lib


def last_error() -> str:
    return lib().b200_last_error().decode()


# When set to a list (bench.py --breakdown), every call is bracketed by CUDA events on the current
# stream: entries are (label, start_event, end_event, work) with work = (flops, bytes) or None.
TIMER = None


# ------------------------------------------------------------------------------------------------
# Binding.  "torch" (default): the TORCH_LIBRARY(b200convlstm, ...) custom ops of libb200convlstm_torch.so
# (csrc/torch_ops.cpp, generated from the header): tensors in, launch on torch's current stream, TORCH_CHECK -> RuntimeError.
# "ctypes": the C ABI called directly.  A call whose pointer arguments are raw addresses or host arrays (tests, the
# strided-copy and multi-tensor entry points) always takes the ctypes route.
# ------------------------------------------------------------------------------------------------
BINDING = os.environ.get("B200_BINDING", "torch")
TORCH_LIB_PATH = os.path.join(HERE, "libb200convlstm_torch.so")
_torch_ops = None     # {entry point: (op, number of pointer-typed parameters mask)}
TORCH_OP_CALLS = [0]  # calls that went through torch.ops.b200convlstm (tests)


def torch_ops():
    """{name: (torch op, [is_pointer per C parameter, without the trailing stream])}; loads the op library once."""
    global _torch_ops
    if _torch_ops is None:
        import torch
        lib()
        if not os.path.exists(TORCH_LIB_PATH):
            raise RuntimeError(f"{TORCH_LIB_PATH} not found: build it with `python -m unet_convlstm_b200.build` "
                               "(or set B200_BINDING=ctypes to call the C ABI directly)")
        torch.ops.load_library(TORCH_LIB_PATH)
        ops = {}
        for name, (_, argtypes) in _protos.items():
            short = name[len("b200_"):]
            if argtypes and argtypes[-1] is ctypes.c_void_p and hasattr(torch.ops.b200convlstm, short):
                ops[name] = (getattr(torch.ops.b200convlstm, short), [a is ctypes.c_void_p for a in argtypes[:-1]])
        _torch_ops = ops
    return _torch_ops


def _is_tensor(a) -> bool:
    return hasattr(a, "data_ptr")


def call(name: str, *args, tag: str = "", work=None):
    """Calls an int-returning entry point and raises on a non-zero status.  Pointer arguments may be tensors (or None)."""
    timer = TIMER
    if timer is not None:
        import torch
        e0 = torch.cuda.Event(enable_timing=True)
        e0.record()
    op = None
    if BINDING == "torch":
        ent = torch_ops().get(name)
        if ent is not None and len(ent[1]) == len(args) - 1 and any(_is_tensor(a) for a in args) and all(
                (a is None or _is_tensor(a)) if isptr else not _is_tensor(a) for a, isptr in zip(args, ent[1])):
            op = ent[0]
    if op is not None:
        op(*args[:-1])      # the op takes torch's current stream itself and raises on a non-zero status
        TORCH_OP_CALLS[0] += 1
        rc = 0
    else:
        rc = getattr(lib(), name)(*[a.data_ptr() if _is_tensor(a) else a for a in args])
    if timer is not None:
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        timer.append((name + (" " + tag if tag else ""), e0, e1, work, torch.cuda.current_stream().cuda_stream))
    CALLS[name] = CALLS.get(name, 0) + 1
    if rc != 0:
        raise RuntimeError(f"{name} failed: rc={rc}: {last_error()}")


def supported(name: str, *args) -> bool:
    return bool(getattr(lib(), name)(*args))
