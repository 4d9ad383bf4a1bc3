"""paddle.tensorrt: ahead-of-time inference lowering. Parity (API): python/paddle/tensorrt/export.py (Input, TensorRTConfig,
PrecisionMode, convert, convert_loaded_model).

There is no TensorRT on this target and none is wanted: the role TensorRT plays in the reference (fuse + pick kernels + freeze
shapes + remove launch overhead) is played here by the hand-written sm_100a kernels plus CUDA-graph capture. `convert` therefore
loads the saved model, casts it to the requested precision, captures one CUDA graph per shape profile (min / opt / max are
warmed, the optimum is captured) and saves the result where `paddle.inference.create_predictor` / `paddle.jit.load` find it."""
from __future__ import annotations

import os

import numpy as np


class PrecisionMode:
    FP32 = "float32"
    FP16 = "float16"
    BF16 = "bfloat16"
    INT8 = "int8"


class Input:
    """Shape profile of one input: min / optimal / max shapes (or concrete warm-up data)."""

    def __init__(self, min_input_shape=None, max_input_shape=None, optim_input_shape=None, input_data_type="float32", input_range=None, name=None,
                 warmup_data=None):
        self.min_input_shape = tuple(min_input_shape) if min_input_shape is not None else None
        self.max_input_shape = tuple(max_input_shape) if max_input_shape is not None else self.min_input_shape
        self.optim_input_shape = tuple(optim_input_shape) if optim_input_shape is not None else self.max_input_shape
        self.input_data_type, self.input_range, self.name, self.warmup_data = input_data_type, input_range, name, warmup_data

    def generate_input_data(self):
        if self.warmup_data is not None:
            return tuple(self.warmup_data)
        lo, hi = self.input_range if self.input_range is not None else ((0.0, 1.0) if "float" in self.input_data_type else (1, 10))

        def gen(shape):
            if "int" in self.input_data_type:
                return np.random.randint(int(lo), int(hi), size=shape).astype(self.input_data_type)
            return np.random.uniform(lo, hi, size=shape).astype(self.input_data_type)
        return gen(self.min_input_shape), gen(self.optim_input_shape), gen(self.max_input_shape)


class TensorRTConfig:
    def __init__(self, inputs, min_subgraph_size=3, save_model_dir=None, disable_ops=None, precision_mode=PrecisionMode.FP32, ops_run_float=None,
                 optimization_level=3, disable_passes=None, workspace_size=1 << 30, use_cuda_graph=True):
        self.inputs, self.save_model_dir, self.precision_mode = list(inputs), save_model_dir, precision_mode
        self.min_subgraph_size, self.disable_ops, self.ops_run_float = min_subgraph_size, disable_ops or [], ops_run_float or []
        self.optimization_level, self.disable_passes, self.workspace_size, self.use_cuda_graph = optimization_level, disable_passes or [], workspace_size, use_cuda_graph


def _lower(layer, config):
    import torch

    from . import jit
    from .framework.place import _default_device
    from .tensor import Tensor

    if config.precision_mode in (PrecisionMode.FP16, PrecisionMode.BF16) and hasattr(layer, "to"):
        layer.to(dtype=config.precision_mode)
    layer.eval() if hasattr(layer, "eval") else None
    profiles = [inp.generate_input_data() for inp in config.inputs]
    on_gpu = _default_device().type == "cuda"     # the current device (paddle.set_device), not merely a visible GPU
    fn = jit.to_static(layer) if (config.use_cuda_graph and on_gpu) else layer
    with torch.no_grad():
        for which in (0, 2, 1, 1, 1):   # min, max, then the optimum often enough for the capture to happen
            args = []
            for inp, prof in zip(config.inputs, profiles):
                t = torch.as_tensor(prof[which])
                if t.is_floating_point() and config.precision_mode in (PrecisionMode.FP16, PrecisionMode.BF16):
                    t = t.to(getattr(torch, config.precision_mode))
                args.append((t.cuda() if on_gpu else t).as_subclass(Tensor))
            fn(*args)
    return fn


def convert(model_path, config):
    """Load `model_path` (jit.save prefix), lower it, save under `config.save_model_dir`; returns the lowered callable."""
    from . import jit

    layer = jit.load(model_path)
    fn = _lower(layer, config)
    if config.save_model_dir:
        os.makedirs(os.path.dirname(config.save_model_dir) or ".", exist_ok=True)
        from .static import InputSpec

        specs = [InputSpec(list(i.optim_input_shape), i.input_data_type, i.name) for i in config.inputs]
        jit.save(layer, config.save_model_dir, input_spec=specs)
    return fn


def convert_loaded_model(model, config):
    return _lower(model, config)
