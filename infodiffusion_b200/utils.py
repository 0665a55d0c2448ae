"""Loss helper of the hot path -- mirror of the reference's ``utils.compute_mmd`` (utils.py:74-90)."""
from __future__ import annotations

import torch

from . import _lib


class _MMD(torch.autograd.Function):
    """MMD(x, y) with the gradient wrt y produced by the same fused kernel (idf_mmd_fwd_bwd)."""

    @staticmethod
    def forward(ctx, x, y):
        if not (x.is_cuda and y.is_cuda):
            raise RuntimeError("compute_mmd runs on the sm_100a kernel only (no CPU path)")
        lib = _lib.load()
        x = x.detach().contiguous().float()
        yc = y.detach().contiguous().float()
        B, D = yc.shape
        if x.shape != yc.shape:
            raise ValueError("compute_mmd expects x and y of the same [B, D] shape")
        loss = torch.empty((), dtype=torch.float32, device=y.device)
        grad = torch.empty_like(yc)
        stream = torch.cuda.current_stream(y.device).cuda_stream
        if torch.are_deterministic_algorithms_enabled():          # partials summed in a fixed order, no atomics
            ws = torch.empty(int(lib.idf_mmd_ws_floats(B)), dtype=torch.float32, device=y.device)
            tickets = torch.zeros(1, dtype=torch.int32, device=y.device)
            _lib.check(lib.idf_mmd_fwd_bwd_ordered(x.data_ptr(), yc.data_ptr(), loss.data_ptr(), grad.data_ptr(), B, D,
                                                   ws.data_ptr(), tickets.data_ptr(), stream))
        else:
            _lib.check(lib.idf_mmd_fwd_bwd(x.data_ptr(), yc.data_ptr(), loss.data_ptr(), grad.data_ptr(), B, D, stream))
        _lib.count_launch()
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, g):
        (grad,) = ctx.saved_tensors
        return None, grad * g


def compute_mmd(x, y):
    """mean k(x,x) + mean k(y,y) - 2 mean k(x,y), k(u,v) = exp(-mean_d((u-v)^2)/D); differentiable in y."""
    return _MMD.apply(x, y)
