"""``torch.ops.metrics_b200.*``: the hot-path entry points as registered PyTorch operators (csrc/torch_ops/ops.cpp).

The operators are thin C++ shims over the plain-C ABI of ``include/metrics_b200.h``: they give the kernels a dispatcher
identity — schema-checked arguments, ``TORCH_CHECK`` errors, the current CUDA stream taken in C++, shape-only "fake"
implementations so that code calling them traces under ``torch.compile`` / fake tensors, TorchScript-callable — which a
ctypes call cannot have.  The metric classes keep calling the C-ABI through ctypes by default (``_native.py``: measured the
shorter host path); ``MB200_BINDING=torch`` routes the operators that exist here through the dispatcher instead, and
``tests/test_torch_ops_gpu.py`` holds the two bindings to identical results.

`build()` compiles the shim in-tree (``_lib/torch_ops/metrics_b200_torch_ops.so``, g++ only: no device code in it);
`load()` registers it with ``torch.ops``.  There is no CPU dispatch: calling an operator with CPU tensors raises.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD_DIR = os.path.join(_HERE, "_lib", "torch_ops")
_SO = os.path.join(_BUILD_DIR, "metrics_b200_torch_ops.so")
_loaded = False


def library_path() -> str:
    return _SO


def build(verbose: bool = False) -> str:
    """Compile csrc/torch_ops/ops.cpp against this interpreter's torch and link it to ``_lib/libmetrics_b200.so``."""
    from torch.utils import cpp_extension

    os.makedirs(_BUILD_DIR, exist_ok=True)
    lib_dir = os.path.join(_HERE, "_lib")
    cpp_extension.load(
        name="metrics_b200_torch_ops",
        sources=[os.path.join(_HERE, "csrc", "torch_ops", "ops.cpp")],
        extra_cflags=["-O2", "-std=c++17"],
        # no .cu source here, but with_cuda makes cpp_extension derive nvcc arch flags, which fails on a machine without a
        # GPU unless TORCH_CUDA_ARCH_LIST is set; an explicit arch skips that probe
        extra_cuda_cflags=["-gencode=arch=compute_100a,code=sm_100a"],
        extra_include_paths=[os.path.join(cpp_extension.CUDA_HOME or "/usr/local/cuda", "include")],
        extra_ldflags=[f"-L{lib_dir}", "-lmetrics_b200", "-Wl,-rpath,'$$ORIGIN/..'", "-lc10_cuda", "-ltorch_cuda"],
        build_directory=_BUILD_DIR,
        is_python_module=False,
        with_cuda=True,
        verbose=verbose,
    )
    return _SO


def load() -> None:
    """Register the operators with ``torch.ops`` (idempotent); fails loudly when the shim has not been built."""
    global _loaded
    if _loaded:
        return
    if not os.path.exists(_SO):
        raise RuntimeError(f"metrics_b200: {_SO} is missing — run `python -c 'import __graft_entry__ as g; g.build()'`")
    torch.ops.load_library(_SO)
    _register_fakes()
    _loaded = True


def available() -> bool:
    return os.path.exists(_SO)


def _register_fakes() -> None:
    """Shape / dtype propagation only (fake tensors, torch.compile tracing); never touches data."""
    fake = torch.library.register_fake

    @fake("metrics_b200::confmat_update_")
    def _(confmat, preds, target, num_classes, ignore_index=None, err_flag=None):
        return None

    @fake("metrics_b200::stat_scores_update_")
    def _(tp, fp, tn, fn, workspace, preds, target, num_classes, ignore_index=None, micro=False, err_flag=None):
        return None

    @fake("metrics_b200::stats_softmax_update_")
    def _(tp, fp, tn, fn, workspace, preds, target, num_classes, micro=False, err_flag=None):
        return torch.empty_like(preds, memory_format=torch.contiguous_format)

    @fake("metrics_b200::normalize_logits_if_needed")
    def _(preds, normalization):
        return torch.empty_like(preds, memory_format=torch.contiguous_format)

    @fake("metrics_b200::curve_evaluate")
    def _(preds, target, num_classes=1, pos_label=1, want_curve=False):
        n = target.numel() if want_curve else 0
        f32 = dict(dtype=torch.float32, device=preds.device)
        thr_dtype = torch.float64 if preds.dtype == torch.float64 else torch.float32
        return (torch.empty(num_classes, **f32), torch.empty(num_classes, **f32),
                torch.empty((num_classes, 3), dtype=torch.int64, device=preds.device), torch.empty((num_classes, n), **f32),
                torch.empty((num_classes, n), **f32), torch.empty((num_classes, n), dtype=thr_dtype, device=preds.device))

    @fake("metrics_b200::binned_curve_update_")
    def _(confmat, scratch, preds, target, thresholds, num_classes=1, multilabel=False):
        return None

    @fake("metrics_b200::regression_sums")
    def _(preds, target, op, num_outputs=1, param=0.0, eps=0.0):
        from metrics_b200 import _native

        k = int(_native.lib().mb200_regression_num_sums(int(op)))
        return torch.empty((k, num_outputs), dtype=torch.float64, device=preds.device)


def ops() -> Optional[object]:
    load()
    return torch.ops.metrics_b200
