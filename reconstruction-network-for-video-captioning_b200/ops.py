"""Operator-level autograd wrappers (one kernel family each) over the C ABI.

These back the per-step ``nn.Module.forward`` mirrors (the reference's single-timestep API,
models/decoder.py:45) and the per-kernel parity tests.  The training hot path uses the sequence-level
Functions in ``functional.py`` instead (one host call for the whole loop).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from .functional import _stream, _ptr


def _op_dtype(precision: int):
    return torch.bfloat16 if precision == L.PREC_BF16 else torch.float32


def gemm(precision: int, A: torch.Tensor, transA: bool, B: torch.Tensor, transB: bool, bias=None, out=None,
         accumulate: bool = False, splits: int = 1, bn_hint: int = 0) -> torch.Tensor:
    """C[m,n] = sum_k A(m,k) B(n,k) (+bias).  A: [M,K] (or [K,M] if transA); B: [N,K] (or [K,N] if transB).
    Operands must already be in the precision's storage type and row-contiguous (stride(1) == 1)."""
    dt = _op_dtype(precision)
    if not (A.is_cuda and B.is_cuda):
        raise RuntimeError(f"recnet_b200.ops.gemm: operands must be CUDA tensors, got {A.device} / {B.device} (recnet_b200 has no CPU path)")
    assert A.dtype == dt and B.dtype == dt and A.stride(1) == 1 and B.stride(1) == 1
    M, K = (A.shape[1], A.shape[0]) if transA else (A.shape[0], A.shape[1])
    N = B.shape[1] if transB else B.shape[0]
    assert (B.shape[0] if transB else B.shape[1]) == K
    if splits > 1:
        Cm = torch.empty(splits, M, N, dtype=torch.float32, device=A.device) if out is None else out
        ldc, sstride = N, M * N
    else:
        Cm = torch.empty(M, N, dtype=torch.float32, device=A.device) if out is None else out
        ldc, sstride = Cm.stride(-2), 0
    L.check(L.lib().recnet_gemm(precision, A.data_ptr(), A.stride(0), int(transA), B.data_ptr(), B.stride(0), int(transB),
                                Cm.data_ptr(), ldc, None, 0, _ptr(bias), M, N, K, splits, sstride, int(accumulate), bn_hint,
                                _stream()), "recnet_gemm")
    return Cm


class LinearFn(torch.autograd.Function):
    """y = x @ W^T (+ b)  -- nn.Linear on our GEMM provider."""

    @staticmethod
    def forward(ctx, x, W, bias, precision):
        dt = _op_dtype(precision)
        xo, Wo = x.contiguous().to(dt), W.contiguous().to(dt)
        ctx.k = x.shape[1]
        if precision == L.PREC_BF16 and ctx.k % 8:      # TMA needs 16-byte row pitch: zero-pad K (e.g. 2004 = 468 + 1536)
            pad = 8 - ctx.k % 8
            xo, Wo = torch.nn.functional.pad(xo, (0, pad)), torch.nn.functional.pad(Wo, (0, pad))
        ctx.precision = precision
        ctx.has_bias = bias is not None
        ctx.n = W.shape[0]
        ctx.save_for_backward(xo, Wo)
        return gemm(precision, xo, False, Wo, False, bias=bias.contiguous() if bias is not None else None)

    @staticmethod
    def backward(ctx, gy):
        xo, Wo = ctx.saved_tensors
        p = ctx.precision
        go = gy.contiguous().to(_op_dtype(p))
        if p == L.PREC_BF16 and go.shape[1] % 8:        # same pitch rule for the N-contiguous operands of the backward GEMMs
            pad = 8 - go.shape[1] % 8
            go, Wo = torch.nn.functional.pad(go, (0, pad)), torch.nn.functional.pad(Wo, (0, 0, 0, pad))
        gx = gemm(p, go, False, Wo, True)[:, :ctx.k] if ctx.needs_input_grad[0] else None              # [M,N] @ [N,K]
        gW = gemm(p, go, True, xo, True)[:W_rows(ctx, go), :ctx.k] if ctx.needs_input_grad[1] else None  # [N,M] @ [M,K]
        gb = gy.sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return gx, gW, gb, None


def W_rows(ctx, go):
    return ctx.n


def linear(x, W, bias, precision):
    return LinearFn.apply(x, W, bias, precision)


class AdditiveAttentionFn(torch.autograd.Function):
    """ctx[b] = mean_tau( (w . tanh(Wh[b] + Uv[b,tau] + bias)) * V[b,tau] )   (models/decoder.py:55-61).
    softmax=True: the paper's attention, ctx[b] = sum_tau alpha[b,tau] V[b,tau] with alpha = softmax_tau(e).
    Wh (B,A) f32; Uv (B,Tn,A) f32; V (B,Tn,D) f32 (cast to the operand type internally)."""

    @staticmethod
    def forward(ctx, Wh, Uv, attn_b, attn_w, V, precision, softmax=False):
        lib = L.lib()
        B, Tn, A = Uv.shape
        D = V.shape[2]
        dt = _op_dtype(precision)
        Wh, Uv, Vo = Wh.contiguous(), Uv.contiguous(), V.contiguous().to(dt)
        attn_b, attn_w = attn_b.contiguous(), attn_w.contiguous().view(-1)
        e = torch.empty(B, Tn, dtype=torch.float32, device=Uv.device)
        out = torch.empty(B, D, dtype=dt, device=Uv.device)
        L.check(lib.recnet_attn_fwd(precision, Wh.data_ptr(), 1, 0, Uv.data_ptr(), Tn * A, A, attn_b.data_ptr(), attn_w.data_ptr(),
                                    Vo.data_ptr(), Tn * D, D, B, Tn, A, D, int(softmax), None, e.data_ptr(), out.data_ptr(), D, 0.0, None, 0, 0,
                                    _stream()), "recnet_attn_fwd")
        ctx.precision, ctx.softmax = precision, bool(softmax)
        ctx.save_for_backward(Wh, Uv, attn_b, attn_w, Vo, e)         # e holds alpha when softmax
        return out.float()

    @staticmethod
    def backward(ctx, g):
        lib = L.lib()
        Wh, Uv, attn_b, attn_w, Vo, e = ctx.saved_tensors
        B, Tn, A = Uv.shape
        D = Vo.shape[2]
        g = g.contiguous().float()
        dWh = torch.empty(B, A, dtype=torch.float32, device=g.device)
        dUv = torch.empty_like(Uv)
        dw = torch.empty(B, A, dtype=torch.float32, device=g.device)
        if ctx.softmax:
            L.check(lib.recnet_attn_bwd_softmax(ctx.precision, g.data_ptr(), 1, 0, D, Vo.data_ptr(), Tn * D, D, e.data_ptr(), Wh.data_ptr(),
                                                Uv.data_ptr(), Tn * A, A, attn_b.data_ptr(), attn_w.data_ptr(), B, Tn, A, D, dWh.data_ptr(),
                                                None, dUv.data_ptr(), dw.data_ptr(), 1, None, 0.0, None, 0, 0, _stream()),
                    "recnet_attn_bwd_softmax")
        else:
            L.check(lib.recnet_attn_bwd(ctx.precision, g.data_ptr(), 1, 0, D, Vo.data_ptr(), Tn * D, D, Wh.data_ptr(), Uv.data_ptr(),
                                        Tn * A, A, attn_b.data_ptr(), attn_w.data_ptr(), B, Tn, A, D, dWh.data_ptr(), None, dUv.data_ptr(),
                                        dw.data_ptr(), 1, None, 0.0, None, 0, 0, _stream()), "recnet_attn_bwd")
        gV = None
        if ctx.needs_input_grad[4]:
            # value gradient: tiny outer product, only the local reconstructor needs it (alpha * g, or e * g / Tn for the mean)
            gV = e.unsqueeze(2) * g.unsqueeze(1)
            if not ctx.softmax:
                gV = gV / Tn
        return dWh, dUv, dWh.sum(0), dw.sum(0).view(1, -1), gV, None, None


def additive_attention(Wh, Uv, attn_b, attn_w, V, precision, softmax=False):
    return AdditiveAttentionFn.apply(Wh, Uv, attn_b, attn_w, V, precision, softmax)


class LSTMCellFn(torch.autograd.Function):
    """(pre-activations (B,4H) incl. biases, c_prev (B,H)) -> (h', c')   gate order i,f,g,o."""

    @staticmethod
    def forward(ctx, pre, c_prev, precision):
        lib = L.lib()
        B, H4 = pre.shape
        H = H4 // 4
        pre, c_prev = pre.contiguous(), c_prev.contiguous()
        gates = torch.empty(B, H4, dtype=_op_dtype(precision), device=pre.device)
        c = torch.empty(B, H, dtype=torch.float32, device=pre.device)
        h = torch.empty(B, H, dtype=torch.float32, device=pre.device)
        L.check(lib.recnet_lstm_cell_fwd(precision, pre.data_ptr(), 1, 0, H4, None, 0, None, None, c_prev.data_ptr(), B, H,
                                         gates.data_ptr(), c.data_ptr(), h.data_ptr(), H, None, 0, None, 0, _stream()),
                "recnet_lstm_cell_fwd")
        ctx.precision = precision
        ctx.save_for_backward(gates, c_prev, c)
        return h, c

    @staticmethod
    def backward(ctx, gh, gc):
        lib = L.lib()
        gates, c_prev, c = ctx.saved_tensors
        B, H = c.shape
        gh = gh.contiguous().float() if gh is not None else torch.zeros_like(c)
        dc = gc.contiguous().float().clone() if gc is not None else torch.zeros_like(c)
        dG = torch.empty(B, 4 * H, dtype=_op_dtype(ctx.precision), device=c.device)
        L.check(lib.recnet_lstm_cell_bwd(ctx.precision, gh.data_ptr(), H, None, None, 0, None, 0, 0, 0, 0, None, 0, 0, 0,
                                         dc.data_ptr(), 0, gates.data_ptr(), c_prev.data_ptr(), c.data_ptr(), B, H, dG.data_ptr(),
                                         4 * H, _stream()), "recnet_lstm_cell_bwd")
        return dG.float(), dc, None


def lstm_cell(pre, c_prev, precision):
    return LSTMCellFn.apply(pre, c_prev, precision)


class GRUCellFn(torch.autograd.Function):
    """(gi (B,3H) = x W_ih^T + b_ih, gh (B,3H) = h W_hh^T + b_hh, h (B,H)) -> h'   gate order r,z,n (nn.GRU)."""

    @staticmethod
    def forward(ctx, gi, gh, h_prev, precision):
        lib = L.lib()
        B, H3 = gi.shape
        H = H3 // 3
        gi, gh, h_prev = gi.contiguous(), gh.contiguous(), h_prev.contiguous()
        stash = torch.empty(B, 4 * H, dtype=_op_dtype(precision), device=gi.device)
        h = torch.empty(B, H, dtype=torch.float32, device=gi.device)
        L.check(lib.recnet_gru_cell_fwd(precision, gi.data_ptr(), 1, 0, H3, gh.data_ptr(), 1, 0, H3, None, 0, None, None,
                                        h_prev.data_ptr(), H, B, H, stash.data_ptr(), h.data_ptr(), H, None, 0, _stream()),
                "recnet_gru_cell_fwd")
        ctx.precision = precision
        ctx.save_for_backward(stash, h_prev)
        return h

    @staticmethod
    def backward(ctx, gh_out):
        lib = L.lib()
        stash, h_prev = ctx.saved_tensors
        B, H = h_prev.shape
        g = gh_out.contiguous().float()
        carry = torch.empty(B, H, dtype=torch.float32, device=g.device)
        dt = _op_dtype(ctx.precision)
        dgi = torch.empty(B, 3 * H, dtype=dt, device=g.device)
        dgh = torch.empty(B, 3 * H, dtype=dt, device=g.device)
        L.check(lib.recnet_gru_cell_bwd(ctx.precision, g.data_ptr(), H, None, 0, None, 0, 0, 0, None, 0, 0, 0, carry.data_ptr(), 1,
                                        stash.data_ptr(), h_prev.data_ptr(), H, B, H, dgi.data_ptr(), dgh.data_ptr(), 3 * H,
                                        _stream()), "recnet_gru_cell_bwd")
        return dgi.float(), dgh.float(), carry, None


def gru_cell(gi, gh, h_prev, precision):
    return GRUCellFn.apply(gi, gh, h_prev, precision)
