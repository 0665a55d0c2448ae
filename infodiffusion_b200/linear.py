"""fp32 Linear with autograd on the library's own kernels (idf_linear_f32 forward, idf_gemm_f32 backward).

The small fully-connected layers of the path -- TimeEmbedding and the per-block temb_proj / aemb_proj (modules.py:24-27,
211, 271-275), the encoder heads fc_a / fc_mu / fc_var (models.py:470-472) and every layer of the LatentUNet
(models.py:147-163, 223-234) -- stay in fp32 like the reference.  In training they sit inside torch's autograd graph;
this Function keeps them off cuBLAS: y = x W^T + b, dX = dY W, dW = dY^T X, db = 1^T dY are all launches of
libidf_b200.so.  Elementwise glue around them (SiLU, LayerNorm, dropout) remains ordinary torch ops.

While torch.are_deterministic_algorithms_enabled(), the split-K GEMMs combine their partial tiles in split order
(idf_gemm_f32_ordered) instead of with atomics, so forward and backward are bitwise reproducible.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _gemm(lib, A, lda, tA, B, ldb, tB, Cm, ldc, M, N, K, acc, st) -> None:
    """Cm[M,N] (+)= op(A) . op(B) on idf_gemm_f32, or on its ordered variant in torch's deterministic mode."""
    if not torch.are_deterministic_algorithms_enabled():
        _lib.check(lib.idf_gemm_f32(A, lda, tA, B, ldb, tB, Cm, ldc, M, N, K, acc, st))
        return
    n = int(lib.idf_gemm_f32_ws_floats(M, N, K))
    ws = torch.empty(max(n, 4), dtype=torch.float32, device="cuda")
    tickets = torch.zeros(64, dtype=torch.int32, device="cuda")
    _lib.check(lib.idf_gemm_f32_ordered(A, lda, tA, B, ldb, tB, Cm, ldc, M, N, K, acc, ws.data_ptr(), tickets.data_ptr(), st))


class _LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b):
        if not x.is_cuda:
            raise RuntimeError("infodiffusion_b200.linear needs CUDA tensors: there is no CPU path")
        lib = _lib.load()
        K, N = w.shape[1], w.shape[0]
        x2 = x.reshape(-1, K).contiguous().float()
        w = w.contiguous().float()
        M = x2.shape[0]
        bb = None if b is None else b.contiguous().float()
        if K >= 1024 and ((N + 63) // 64) * ((M + 63) // 64) < 32:
            # few output tiles and a long reduction (the encoder's fc_a: [B, 4096] -> a_dim): split-K GEMM accumulated on
            # top of the bias (atomic partial sums -- training only; the inference plans keep the deterministic kernel)
            y = (bb if bb is not None else torch.zeros(N, device=x.device)).expand(M, N).contiguous()
            _gemm(lib, x2.data_ptr(), K, 0, w.data_ptr(), K, 1, y.data_ptr(), N, M, N, K, 1, _stream(x))
        else:
            y = torch.empty(M, N, dtype=torch.float32, device=x.device)
            _lib.check(lib.idf_linear_f32(x2.data_ptr(), K, w.data_ptr(), None if bb is None else bb.data_ptr(), y.data_ptr(), N,
                                          M, N, K, 0, _stream(x)))
        _lib.count_launch()
        ctx.save_for_backward(x2, w)
        ctx.has_bias = b is not None
        ctx.xshape = x.shape
        return y.view(*x.shape[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        x2, w = ctx.saved_tensors
        lib = _lib.load()
        N, K = w.shape
        M = x2.shape[0]
        dy2 = dy.reshape(M, N).contiguous().float()
        st = _stream(dy2)
        dx = dw = db = None
        n = 0
        if ctx.needs_input_grad[0]:                  # dX[M,K] = dY[M,N] . W[N,K]
            dx = torch.empty(M, K, dtype=torch.float32, device=dy2.device)
            _gemm(lib, dy2.data_ptr(), N, 0, w.data_ptr(), K, 0, dx.data_ptr(), K, M, K, N, 0, st)
            dx = dx.view(ctx.xshape)
            n += 1
        if ctx.needs_input_grad[1]:                  # dW[N,K] = dY^T[N,M] . X[M,K]
            dw = torch.empty(N, K, dtype=torch.float32, device=dy2.device)
            _gemm(lib, dy2.data_ptr(), N, 1, x2.data_ptr(), K, 0, dw.data_ptr(), K, N, K, M, 0, st)
            n += 1
        if ctx.has_bias and ctx.needs_input_grad[2]:  # db[N] = 1^T[1,M] . dY[M,N]
            ones = torch.ones(1, M, dtype=torch.float32, device=dy2.device)
            db = torch.empty(N, dtype=torch.float32, device=dy2.device)
            _gemm(lib, ones.data_ptr(), M, 0, dy2.data_ptr(), N, 0, db.data_ptr(), N, 1, N, M, 0, st)
            n += 1
        _lib.count_launch(n)
        return dx, dw, db


def linear(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Drop-in for torch.nn.functional.linear (fp32, CUDA) with forward and backward on libidf_b200.so."""
    return _LinearFn.apply(x, weight, bias)


def apply(module: torch.nn.Linear, x: torch.Tensor) -> torch.Tensor:
    """module(x) for an nn.Linear parameter container."""
    return _LinearFn.apply(x, module.weight, module.bias)
