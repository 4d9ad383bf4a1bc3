"""auto_cast / decorate. Parity: python/paddle/amp/auto_cast.py, amp_lists.py.

O1: white-list ops (matmul/conv/linear/attention...) run in low precision, black-list ops in fp32 — implemented with
torch.autocast (same op-level policy).  O2: ``decorate`` casts parameters to the low dtype (norm layers excluded like
the reference) and switches the optimizer to multi_precision master weights.
"""
from __future__ import annotations

import contextlib

import torch

from ..framework import dtype as _dt
from ..framework.place import _default_device

WHITE_LIST = {"conv2d", "einsum", "matmul", "matmul_v2", "max_pool2d_with_index", "mul", "fused_gemm_epilogue", "linear", "flash_attn"}
BLACK_LIST = {"exp", "square", "log", "mean", "sum", "cos_sim", "softmax", "softmax_with_cross_entropy", "sigmoid_cross_entropy_with_logits",
              "c_softmax_with_cross_entropy", "cross_entropy", "cross_entropy2", "reduce_sum", "layer_norm", "batch_norm", "rms_norm"}

_state = {"enabled": False, "level": "O0", "dtype": torch.float32, "black": frozenset(), "white": frozenset()}


def fp32_guard(op, *tensors):
    """For white-list ops that the user moved to `custom_black_list`: returns (context, tensors cast to fp32) so the op runs
    outside autocast; a no-op context and the tensors unchanged otherwise."""
    if _state["enabled"] and op in _state["black"]:
        return torch.autocast(device_type=_default_device().type, enabled=False), tuple(t.float() if isinstance(t, torch.Tensor) and t.is_floating_point() else t for t in tensors)
    if _state["enabled"] and _state["level"] == "O2" and len(tensors) >= 2:
        # O2: parameters are low precision; an fp32 activation (typically the model input) meeting them is cast down, like the
        # reference's O2 autocast of white-list op inputs.  Only reached on paths where the dtypes would otherwise clash.
        x, w = tensors[0], tensors[1]
        if isinstance(x, torch.Tensor) and isinstance(w, torch.Tensor) and x.is_floating_point() and w.dtype in (torch.float16, torch.bfloat16) and x.dtype != w.dtype:
            rest = tuple(t.to(w.dtype) if isinstance(t, torch.Tensor) and t.is_floating_point() and t.dtype != w.dtype else t for t in tensors[2:])
            tensors = (x.to(w.dtype), w) + rest
    return contextlib.nullcontext(), tensors


def black_dtype(op, x, dtype=None):
    """Compute dtype for a black-list op under O1: fp32 for low-precision inputs unless the user white-listed the op."""
    if dtype is None and _state["enabled"] and _state["level"] == "O1" and op in BLACK_LIST and op not in _state["white"] \
            and x.dtype in (torch.float16, torch.bfloat16):
        return torch.float32
    return dtype


def low_precision_forced(op):
    """True for black-list ops the user moved to `custom_white_list` (they then run in the autocast dtype)."""
    return _state["enabled"] and op in _state["white"]


def white_list():
    return {"float16": {"O1": set(WHITE_LIST), "O2": set(WHITE_LIST)}, "bfloat16": {"O1": set(WHITE_LIST), "O2": set(WHITE_LIST)}}


def black_list():
    return {"float16": {"O1": set(BLACK_LIST), "O2": set()}, "bfloat16": {"O1": set(BLACK_LIST), "O2": set()}}


def is_float16_supported(device=None):
    return True


def is_bfloat16_supported(device=None):
    return True


def amp_state():
    return dict(_state)


@contextlib.contextmanager
def auto_cast(enable=True, custom_white_list=None, custom_black_list=None, level="O1", dtype="float16", use_promote=True):
    if level not in ("O0", "OD", "O1", "O2"):
        raise ValueError("level should be O0, OD, O1 or O2")
    d = _dt.convert_dtype(dtype)
    prev = dict(_state)
    active = enable and level != "O0"
    _state.update(enabled=active, level=level if active else "O0", dtype=d if active else torch.float32,
                  black=frozenset(custom_black_list or ()) if active else frozenset(), white=frozenset(custom_white_list or ()) if active else frozenset())
    dev = _default_device().type   # the current device (paddle.set_device), like the reference's expected place
    try:
        if active and level in ("O1", "OD"):
            if dev == "cpu" and d == torch.float16:
                d = torch.bfloat16
            with torch.autocast(device_type=dev, dtype=d, enabled=True):
                yield
        else:
            yield  # O2: parameters are already low precision; ops follow their inputs
    finally:
        _state.clear()
        _state.update(prev)


amp_guard = auto_cast


def decorate(models, optimizers=None, level="O1", dtype="float16", master_weight=None, save_dtype=None, master_grad=False, excluded_layers=None):
    """Parity: amp/auto_cast.py:amp_decorate."""
    from ..nn.conv_norm_pool import LayerNorm, _BatchNormBase, _InstanceNormBase

    if level not in ("O1", "O2"):
        raise ValueError("level should be O1 or O2")
    single_m = not isinstance(models, (list, tuple))
    ms = [models] if single_m else list(models)
    single_o = optimizers is not None and not isinstance(optimizers, (list, tuple))
    os_ = [] if optimizers is None else ([optimizers] if single_o else list(optimizers))
    if level == "O2":
        d = _dt.convert_dtype(dtype)
        excluded = [_BatchNormBase, LayerNorm, _InstanceNormBase]
        if excluded_layers:
            for e in (excluded_layers if isinstance(excluded_layers, (list, tuple)) else [excluded_layers]):
                excluded.append(e if isinstance(e, type) else type(e))
        for m in ms:
            m._cast_floating(d, excluded_layers=tuple(excluded))
        for o in os_:
            if master_weight is not False:
                o._multi_precision = True
    if optimizers is None:
        return ms[0] if single_m else ms
    return (ms[0] if single_m else ms), (os_[0] if single_o else os_)
