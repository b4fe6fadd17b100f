"""The TF32 twin of the PPO oracles: ``oracle.ppo_ref`` / ``oracle.ppo_categorical_ref`` / ``tests/ppo_options_oracle.py``
run unchanged, with every operand of the four hidden Linear layers truncated to TF32 in the forward and in the backward.

Math mode 1 runs the hidden-layer GEMMs as single-pass TF32 tensor-core products: tcgen05 ``kind::tf32`` keeps the top
10 mantissa bits of each fp32 operand (``trunc``, as ``tools/tf32_probe.py`` measures it) and accumulates in fp32.  The
twin reproduces those products in fp64: inside ``tf32()`` every ``a @ b`` whose result has ``H`` columns -- the
``shared.0``, ``shared.2``, ``actor_mean.0`` and ``critic.0`` layers; the heads have A, n or 1 columns -- becomes
``trunc(a) @ trunc(b)``, and its backward forms ``trunc(g) @ trunc(b)^T`` and ``trunc(a)^T @ trunc(g)`` (the input- and
weight-gradient GEMMs the kernels run).  ``|twin - oracle|`` is then the size of the error that operand truncation
alone causes, which sets the mode-1 tolerances of tests/test_ppo_paths_gpu.py.

With ``truncate=False`` the twin goes through the same interception and the same backward code and must equal the
oracle bit for bit (tests/test_ppo_paths_cpu.py): that is what makes it the oracle's twin and not a restatement.
"""
import threading

import torch
from torch.overrides import TorchFunctionMode


def trunc(x):
    """fp32 -> TF32 by truncation: the low 13 mantissa bits cleared (tools/tf32_probe.py)."""
    return (x.view(torch.int32) & -8192).view(torch.float32)


def trunc64(x):
    """An fp64 operand as the kernel would hold it: rounded to fp32 (what the fp32 buffers store), then truncated."""
    return trunc(x.to(torch.float32).contiguous()).to(x.dtype)


_inside = threading.local()
# what `a @ b` reaches a TorchFunctionMode as
_MATMUL = (torch.Tensor.__matmul__, torch.Tensor.matmul, torch._C.TensorBase.matmul, torch.matmul)


class _Tf32Matmul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, truncate):
        ctx.save_for_backward(a, b)
        ctx.truncate = truncate
        q = trunc64 if truncate else (lambda t: t)
        return q(a) @ q(b)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        q = trunc64 if ctx.truncate else (lambda t: t)
        # torch's own matmul backward on the (truncated) operands: with truncate=False exactly the oracle's arithmetic
        need = [t for t, n in zip((a, b), ctx.needs_input_grad[:2]) if n]
        if not need:
            return None, None, None
        with torch.enable_grad():
            a_ = q(a).detach().requires_grad_(ctx.needs_input_grad[0])
            b_ = q(b).detach().requires_grad_(ctx.needs_input_grad[1])
            _inside.on = True
            try:
                grads = torch.autograd.grad(a_ @ b_, [t for t in (a_, b_) if t.requires_grad], q(g))
            finally:
                _inside.on = False
        grads = list(grads)
        ga = grads.pop(0) if ctx.needs_input_grad[0] else None
        gb = grads.pop(0) if ctx.needs_input_grad[1] else None
        return ga, gb, None


class _Mode(TorchFunctionMode):
    def __init__(self, H, truncate):
        super().__init__()
        self.H, self.truncate = H, truncate

    def __torch_function__(self, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        if (func in _MATMUL and not getattr(_inside, "on", False) and not kwargs
                and len(args) == 2 and args[0].dim() == 2 and args[1].dim() == 2 and args[1].shape[1] == self.H):
            return _Tf32Matmul.apply(args[0], args[1], self.truncate)
        return func(*args, **kwargs)


def tf32(H, truncate=True):
    """A context inside which the oracle functions compute the TF32 twin of a policy of hidden width H."""
    return _Mode(H, truncate)
