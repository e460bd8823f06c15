"""Ops: fused sm_100a kernels (``_C`` extension) + PyTorch oracles."""
from __future__ import annotations

import importlib
import os

_EXT = None
_EXT_ERR = None


def load_ext(required: bool = False):
    """Import the in-tree extension ``nn_distributed_training_b200/ops/_C*.so``
    (built by ``__graft_entry__.build()`` / ``python -m nn_distributed_training_b200.ops.build``)."""
    global _EXT, _EXT_ERR
    if _EXT is None and _EXT_ERR is None:
        try:
            import torch  # noqa: F401  (libtorch symbols must be loaded first)
            _EXT = importlib.import_module("nn_distributed_training_b200.ops._C")
        except Exception as e:  # noqa: BLE001
            _EXT_ERR = e
    if _EXT is None and required:
        raise RuntimeError(
            "the sm_100a extension nn_distributed_training_b200.ops._C is not built/loadable "
            f"({_EXT_ERR!r}); run `python -c 'import __graft_entry__ as g; g.build()'`")
    return _EXT


def fused_available() -> bool:
    """True iff a CUDA device is present AND the extension loads.  On a GPU box
    a missing extension is an error, not a silent fallback."""
    import torch

    if not torch.cuda.is_available():
        return False
    if os.environ.get("NNDT_FORCE_TORCH", "0") == "1":
        return False
    load_ext(required=True)
    return True


def mnist_kernel_is_paper_shape(spec) -> bool:
    """The specialised kernels (mnist.cu / mnist_tc.cu) are written for the paper's MNISTConvNet(3, 5, 64)."""
    return (spec.in_hw == 28 and spec.num_classes == 10 and spec.kernel_size == 5
            and spec.num_filters == 3 and spec.linear_width == 64)


def mnist_kernel_supports(spec, batch_size: int, dtype=None) -> bool:
    """Conv-net shapes / dtypes with a hand-written forward+backward kernel: the paper shape in fp32 (specialised
    kernels) and, through csrc/mnist_generic.cu, num_filters <= 8, kernel_size in {3, 5}, linear_width <= 128 in fp32 or
    fp64."""
    import torch

    if not (spec.in_hw == 28 and spec.num_classes == 10 and 1 <= batch_size <= 4096):
        return False
    if dtype not in (None, torch.float32, torch.float64):
        return False
    if dtype in (None, torch.float32) and mnist_kernel_is_paper_shape(spec):
        return True
    return 1 <= spec.num_filters <= 8 and spec.kernel_size in (3, 5) and 1 <= spec.linear_width <= 128


def mlp_kernel_supports(spec, base_loss, dtype=None) -> bool:
    """Shapes/losses/dtypes the implicit-density MLP kernels are instantiated for: csrc/mlp_tc.cu (tcgen05) in fp32,
    csrc/mlp_f64.cu in fp64, the same network family in both."""
    import torch

    try:
        from .mlp_fused import supports
    except Exception:  # noqa: BLE001
        return False
    return supports(spec, base_loss, torch.float32 if dtype is None else dtype)
