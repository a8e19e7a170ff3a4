"""Host-side mirror of DLRM.jl's dot-interaction entry points (src/model/interact.jl).

``DotInteraction`` is the callable stored in ``DLRMModel.interaction`` (src/model/model.jl:119,163);
its ``torch.autograd.Function`` plays the role of ``ChainRulesCore.rrule(::DotInteraction, X, Y)``
(src/model/interact.jl:438-447).  Forward and backward are single launches of the sm_100a
kernels in csrc/interact.cu.
"""
from __future__ import annotations

from typing import List, Sequence

import torch

from . import _lib, _prof

POST_INTERACTION_PAD_TO_MUL = 1  # src/model/model.jl:32


def cdiv(x: int, y: int) -> int:
    return 1 + (x - 1) // y


def up_to_mul_of(x: int, y: int) -> int:
    return y * cdiv(x, y)


def interaction_width(F: int, d: int, pad_to_mul: int = POST_INTERACTION_PAD_TO_MUL) -> int:
    """src/model/interact.jl:453-455."""
    return up_to_mul_of(d + F * (F - 1) // 2, pad_to_mul)


def _stream(t: torch.Tensor) -> int:
    return int(torch.cuda.current_stream(t.device).cuda_stream)


def _require_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.DLRMB200Error(_lib.EINVAL, "dot interaction runs on the GPU only (no CPU fallback)")


class _DotInteractionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: torch.Tensor, T: torch.Tensor, pad_to_mul: int):
        _require_cuda(x, T)
        B, F, d = T.shape
        assert T.is_contiguous() and T.dtype == torch.float32
        xc = x.contiguous() if x is not None else None
        assert xc is None or xc.shape == (B, d)
        out = torch.empty((B, interaction_width(F, d, pad_to_mul)), dtype=torch.float32, device=T.device)
        lib = _lib.load()
        # fast_vcat (interact.jl:271-281) is fused: x lands in slot 0 of T inside the kernel
        with _prof.range("interaction_fwd"):
            _lib.check(lib.dlrmb_interaction_fwd(
                T.device.index or 0, T.data_ptr(), xc.data_ptr() if xc is not None else None,
                B, F, d, pad_to_mul, out.data_ptr(), _stream(T)))
        ctx.save_for_backward(T)
        ctx.pad_to_mul = pad_to_mul
        ctx.has_x = x is not None
        return out

    @staticmethod
    def backward(ctx, dOut: torch.Tensor):
        (T,) = ctx.saved_tensors
        B, F, d = T.shape
        dOut = dOut.contiguous()
        dT = torch.empty_like(T)
        dx = torch.empty((B, d), dtype=torch.float32, device=T.device)
        lib = _lib.load()
        with _prof.range("interaction_bwd"):
            _lib.check(lib.dlrmb_interaction_bwd(
                T.device.index or 0, dOut.data_ptr(), T.data_ptr(), B, F, d, ctx.pad_to_mul,
                dT.data_ptr(), dx.data_ptr(), _stream(T)))
        # (dx, dy): dy is the whole (d*F) x B matrix, slot 0 included (interact.jl:428-435)
        if not ctx.has_x:
            # dot_interaction entry point: x IS slot 0 of the stacked input, so its gradient is the sum of
            # both roles -- the pass-through copy out[:, :d] and the Gram row -- which is what the kernel
            # returns as dx = dOut[:, :d] + dT[:, 0] (Zygote differentiates concat([X, Zflat]) the same way)
            dT[:, 0, :] = dx
            return None, dT, None
        return dx, dT, None


class ScatterPlan:
    """Where the interaction backward stores the gradient row of every feature slot when the
    embedding tables are sharded: `dests` is a device int64 tensor [F][3] laid out as the C struct
    dlrmb_slot_dest {base pointer, floats per destination sample, float offset of the table}.  With ``Q`` > 1
    it is [F * Q][3]: entry f * Q + q receives columns [q d / Q, (q + 1) d / Q) of slot f (column-wise sharded
    tables, dlrmb_interaction_bwd_scatter_cols)."""

    def __init__(self, dests: torch.Tensor, sample_offset: int, stream: "torch.cuda.Stream" = None, Q: int = 1):
        """``stream``: when given, the backward is split -- dx alone (dlrmb_interaction_bwd_dx) on the
        current stream, the full pullback with the peer stores on ``stream`` -- so whatever consumes dx
        (the bottom MLP's backward) overlaps the gradient exchange; wait for ``done`` before using the
        exchanged rows (ShardedEmbedding.finish_backward does)."""
        assert dests.dtype == torch.int64 and dests.dim() == 2 and dests.shape[1] == 3 and dests.is_contiguous()
        self.dests = dests
        self.Q = int(Q)
        self.sample_offset = int(sample_offset)
        self.stream = stream
        self.done = torch.cuda.Event() if stream is not None else None
        self._keep = None
        self.on_launched = None      # callable run right after the scattering backward has been launched


def _scatter(lib, T, dOut, B, F, d, pad_to_mul, plan: ScatterPlan, dx, stream) -> None:
    if plan.Q == 1:
        _lib.check(lib.dlrmb_interaction_bwd_scatter(
            T.device.index or 0, dOut.data_ptr(), T.data_ptr(), B, F, d, pad_to_mul,
            plan.dests.data_ptr(), plan.sample_offset, dx.data_ptr(), stream))
    else:
        _lib.check(lib.dlrmb_interaction_bwd_scatter_cols(
            T.device.index or 0, dOut.data_ptr(), T.data_ptr(), B, F, d, pad_to_mul,
            plan.dests.data_ptr(), plan.Q, plan.sample_offset, dx.data_ptr(), stream))


class _DotInteractionScatterFn(torch.autograd.Function):
    """Forward as _DotInteractionFn; backward = interaction pullback fused with the gradient
    exchange (dlrmb_interaction_bwd_scatter): dT rows go straight to the table owners' buffers, only
    dx comes back through autograd.  T must not require grad."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, T: torch.Tensor, pad_to_mul: int, plan: ScatterPlan):
        _require_cuda(x, T)
        B, F, d = T.shape
        assert T.is_contiguous() and T.dtype == torch.float32 and plan.dests.shape[0] == F * plan.Q
        xc = x.contiguous()
        out = torch.empty((B, interaction_width(F, d, pad_to_mul)), dtype=torch.float32, device=T.device)
        lib = _lib.load()
        with _prof.range("interaction_fwd"):
            _lib.check(lib.dlrmb_interaction_fwd(
                T.device.index or 0, T.data_ptr(), xc.data_ptr(), B, F, d, pad_to_mul, out.data_ptr(), _stream(T)))
        ctx.T = T
        ctx.pad_to_mul = pad_to_mul
        ctx.plan = plan
        return out

    @staticmethod
    def backward(ctx, dOut: torch.Tensor):
        T, plan = ctx.T, ctx.plan
        B, F, d = T.shape
        dOut = dOut.contiguous()
        dx = torch.empty((B, d), dtype=torch.float32, device=T.device)
        lib = _lib.load()
        if plan.stream is not None and d % 4 == 0:
            # dx first, on this stream: autograd's consumers of dx do not wait for the peer stores
            _lib.check(lib.dlrmb_interaction_bwd_dx(
                T.device.index or 0, dOut.data_ptr(), T.data_ptr(), B, F, d, ctx.pad_to_mul, dx.data_ptr(), _stream(T)))
            cur = torch.cuda.current_stream(T.device)
            plan.stream.wait_stream(cur)
            dx_full = torch.empty_like(dx)
            with torch.cuda.stream(plan.stream):
                with _prof.range("interaction_bwd"):
                    _scatter(lib, T, dOut, B, F, d, ctx.pad_to_mul, plan, dx_full, plan.stream.cuda_stream)
                plan.done.record(plan.stream)
            plan._keep = (dOut, dx_full)      # alive until the exchange has been joined (finish_backward)
            if plan.on_launched is not None:
                plan.on_launched()
            return dx, None, None, None
        with _prof.range("interaction_bwd"):
            _scatter(lib, T, dOut, B, F, d, ctx.pad_to_mul, plan, dx, _stream(T))
        if plan.on_launched is not None:
            plan.on_launched()
        return dx, None, None, None


class DotInteraction:
    """``DotInteraction`` (src/model/interact.jl:369-411).

    ``dot(x, T)``: x [B][d] bottom-MLP output, T [B][F][d] the PreallocationStrategy lookup
    buffer whose slot 0 is reserved for x.  Returns [B][d + F(F-1)/2 (+pad)].
    """

    def __init__(self, pad_to_mul: int = POST_INTERACTION_PAD_TO_MUL):
        self.pad_to_mul = pad_to_mul

    def __call__(self, x: torch.Tensor, T: torch.Tensor, scatter: "ScatterPlan" = None) -> torch.Tensor:
        if scatter is not None:
            return _DotInteractionScatterFn.apply(x, T, self.pad_to_mul, scatter)
        return _DotInteractionFn.apply(x, T, self.pad_to_mul)


def dot_interaction(x: torch.Tensor, ys: Sequence[torch.Tensor]) -> torch.Tensor:
    """Implementation-2 entry point (src/model/interact.jl:503-513): ``ys`` is a vector of
    [B][D] matrices (DefaultStrategy).  Same kernels; the concat is one torch.stack."""
    T = torch.stack([x, *ys], dim=1).contiguous()
    return _DotInteractionFn.apply(None, T, POST_INTERACTION_PAD_TO_MUL)


def interaction_fwd(T: torch.Tensor, x: torch.Tensor = None, pad_to_mul: int = 1) -> torch.Tensor:
    """Raw forward launch (no autograd)."""
    with torch.no_grad():
        return _DotInteractionFn.apply(x, T, pad_to_mul)


def interaction_bwd(dOut: torch.Tensor, T: torch.Tensor, pad_to_mul: int = 1):
    """Raw backward launch: returns (dx, dT) as dot_back does (src/model/interact.jl:424-436)."""
    _require_cuda(dOut, T)
    B, F, d = T.shape
    dT = torch.empty_like(T)
    dx = torch.empty((B, d), dtype=torch.float32, device=T.device)
    lib = _lib.load()
    _lib.check(lib.dlrmb_interaction_bwd(
        T.device.index or 0, dOut.contiguous().data_ptr(), T.data_ptr(), B, F, d, pad_to_mul,
        dT.data_ptr(), dx.data_ptr(), _stream(T)))
    return dx, dT


__all__ = ["DotInteraction", "dot_interaction", "interaction_fwd", "interaction_bwd",
           "interaction_width", "POST_INTERACTION_PAD_TO_MUL"]
