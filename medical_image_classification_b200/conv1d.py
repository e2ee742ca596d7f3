"""Causal depth-wise conv1d -- host side of causal-conv1d's `causal_conv1d_fn` (the conv of the Mamba-2 mixer):

    causal_conv1d_fn(x, weight, bias=None, seq_idx=None, initial_states=None, return_final_states=False,
                     final_states_out=None, activation=None)

x (batch, dim, L); weight (dim, width), width 2..4; bias (dim); seq_idx (batch, L) integers: no tap crosses a change of id.
out[:, c, t] = act(bias[c] + sum_k weight[c, k] x[:, c, t - (width-1) + k]), act = SiLU for "silu" / "swish".  Returns out
(batch, dim, L) in x's dtype, channel-last in memory (out.stride(1) == 1).  x is read in place when it is channel-last
(x.stride(1) == 1, e.g. a transposed slice of in_proj's output); otherwise one channel-last copy is made.  Differentiable in x,
weight and bias.  The conv states (initial_states, return_final_states, final_states_out) are not implemented.

    causal_conv1d_update(x, conv_state, weight, bias=None, activation=None, cache_seqlens=None)

is causal-conv1d's decoding step: the conv over cat(conv_state, x) for the new tokens, with conv_state shifted in place.

The work is done by csrc/conv1d.cu through b200_causal_conv1d_fwd / _bwd / _update; there is no CPU path.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import no_autocast as _no_autocast


def act_is_silu(activation) -> bool:
    if activation not in (None, "silu", "swish"):
        raise RuntimeError(f"activation must be None, 'silu' or 'swish', got {activation!r}")
    return activation is not None


def check_weight(weight, bias, dim, what):
    if weight.dim() != 2 or weight.shape[0] != dim:
        raise RuntimeError(f"{what}: conv1d weight must be ({dim}, width), got {tuple(weight.shape)}")
    if not 2 <= weight.shape[1] <= 4:
        raise RuntimeError(f"{what}: conv1d width {weight.shape[1]} is outside 2..4")
    if bias is not None and tuple(bias.shape) != (dim,):
        raise RuntimeError(f"{what}: conv1d bias must be ({dim},), got {tuple(bias.shape)}")


def _seq(seq_idx):
    return (None, 0, 0) if seq_idx is None else (seq_idx.data_ptr(), seq_idx.stride(0), seq_idx.stride(1))


def conv_fwd(x, w32, b32, seq_idx, silu, out):
    """out (batch, L, C) = act(causal conv of x (batch, L, C)), both channel-last views with unit channel stride, any batch / time
    strides; w32 (C, width) / b32 (C) contiguous fp32; seq_idx int32 (batch, L) or None."""
    batch, L, C = x.shape
    sp, ssb, ssl = _seq(seq_idx)
    _lib.launch("b200_causal_conv1d_fwd", x.device, x.data_ptr(), _lib.dtype_code(x.dtype), x.stride(0), x.stride(1), w32.data_ptr(),
                _lib.ptr(b32), sp, ssb, ssl, out.data_ptr(), _lib.dtype_code(out.dtype), out.stride(0), out.stride(1), batch, L, C,
                w32.shape[1], int(silu))
    return out


def conv_bwd(g, x, w32, b32, seq_idx, silu, dx):
    """From g (batch, L, C) fp32, the gradient of conv_fwd's output, write dx (x's dtype, its own strides) in place and return
    (dweight (C, width), dbias (C) or None), fp32.  The partial sums of the kernel are added up here in a fixed order."""
    batch, L, C = x.shape
    width = w32.shape[1]
    rows = _lib.load().b200_causal_conv1d_partials(batch, L, C, width)
    if rows < 0:
        _lib.check(rows, "b200_causal_conv1d_partials")
    dwp = torch.empty((rows, C, width), dtype=torch.float32, device=x.device)
    dbp = torch.empty((rows, C), dtype=torch.float32, device=x.device) if b32 is not None else None
    sp, ssb, ssl = _seq(seq_idx)
    _lib.launch("b200_causal_conv1d_bwd", x.device, g.data_ptr(), g.stride(0), g.stride(1), x.data_ptr(), _lib.dtype_code(x.dtype),
                x.stride(0), x.stride(1), w32.data_ptr(), _lib.ptr(b32), sp, ssb, ssl, dx.data_ptr(), dx.stride(0), dx.stride(1),
                dwp.data_ptr(), _lib.ptr(dbp), batch, L, C, width, int(silu))
    return dwp.sum(0), None if dbp is None else dbp.sum(0)


def channel_last_f32(t):
    """t (batch, L, C) as fp32 with a unit channel stride (in place when it already is)."""
    t = t.to(torch.float32)
    return t if t.stride(-1) == 1 else t.contiguous()


class CausalConv1dFn(torch.autograd.Function):
    """x (batch, L, C) channel-last view -> act(conv) (batch, L, C) contiguous, x's dtype."""

    @staticmethod
    @_no_autocast
    def forward(ctx, x, weight, bias, seq_idx, silu):
        w32, b32 = _lib.f32c(weight), _lib.f32c(bias)
        out = conv_fwd(x, w32, b32, seq_idx, silu, torch.empty(x.shape, dtype=x.dtype, device=x.device))
        ctx.save_for_backward(x, w32, b32, seq_idx)
        ctx.silu = silu
        ctx.dtypes = (weight.dtype, None if bias is None else bias.dtype)
        return out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout):
        x, w32, b32, seq_idx = ctx.saved_tensors
        dx = torch.empty(x.shape, dtype=x.dtype, device=x.device)
        dw, db = conv_bwd(channel_last_f32(dout), x, w32, b32, seq_idx, ctx.silu, dx)
        t_w, t_b = ctx.dtypes
        return dx, dw.to(t_w), None if db is None else db.to(t_b), None, None


def causal_conv1d_fn(x, weight, bias=None, seq_idx=None, initial_states=None, return_final_states=False, final_states_out=None,
                     activation=None):
    """causal-conv1d's causal_conv1d_fn: x (batch, dim, L), weight (dim, width), bias (dim,) or None, seq_idx (batch, L) or None.
    Returns out (batch, dim, L) in x's dtype."""
    if initial_states is not None or return_final_states or final_states_out is not None:
        raise NotImplementedError("causal_conv1d_fn: the conv states (initial_states, return_final_states, final_states_out) are "
                                  "not implemented")
    silu = act_is_silu(activation)
    _lib.require_cuda(x, weight, bias, seq_idx)
    if x.dim() != 3:
        raise RuntimeError(f"causal_conv1d_fn: x must be (batch, dim, L), got {tuple(x.shape)}")
    batch, dim, L = x.shape
    check_weight(weight, bias, dim, "causal_conv1d_fn")
    _lib.dtype_code(x.dtype)
    from .ssd_combined import _index_tensor
    seq_idx = _index_tensor(seq_idx, "seq_idx", x.device, (batch, L), "causal_conv1d_fn")
    xt = x.transpose(1, 2)
    if xt.stride(2) != 1:
        xt = xt.contiguous()
    return CausalConv1dFn.apply(xt, weight, bias, seq_idx, silu).transpose(1, 2)


@torch.no_grad()
def causal_conv1d_update(x, conv_state, weight, bias=None, activation=None, cache_seqlens=None):
    """causal-conv1d's causal_conv1d_update (one decoding step): x (batch, dim) or (batch, dim, seqlen), conv_state (batch, dim,
    state_len) with state_len >= width - 1, in x's dtype.  Over cat(conv_state, x) along time, returns the conv (+ SiLU for
    "silu" / "swish") of the last seqlen steps, shaped and typed like x, and overwrites conv_state in place with the last
    state_len columns.  Every tensor is read through its strides in its own dtype; one kernel launch, not differentiable.
    cache_seqlens (the circular-buffer mode) is not implemented."""
    if cache_seqlens is not None:
        raise NotImplementedError("causal_conv1d_update: cache_seqlens (the circular-buffer conv state) is not implemented")
    silu = act_is_silu(activation)
    _lib.require_cuda(x, conv_state, weight, bias)
    if x.dim() not in (2, 3):
        raise RuntimeError(f"causal_conv1d_update: x must be (batch, dim) or (batch, dim, seqlen), got {tuple(x.shape)}")
    x3 = x.unsqueeze(-1) if x.dim() == 2 else x
    batch, dim, seqlen = x3.shape
    check_weight(weight, bias, dim, "causal_conv1d_update")
    width = weight.shape[1]
    if conv_state.dim() != 3 or tuple(conv_state.shape[:2]) != (batch, dim):
        raise RuntimeError(f"causal_conv1d_update: conv_state must be ({batch}, {dim}, state_len), got {tuple(conv_state.shape)}")
    state_len = conv_state.shape[2]
    if state_len < width - 1:
        raise RuntimeError(f"causal_conv1d_update: conv_state has state_len {state_len} < width - 1 = {width - 1}")
    if conv_state.dtype != x.dtype:
        raise RuntimeError(f"causal_conv1d_update: conv_state dtype {conv_state.dtype} differs from x's {x.dtype}")
    if any(st == 0 and sz > 1 for sz, st in zip(conv_state.shape, conv_state.stride())):
        raise RuntimeError("causal_conv1d_update: conv_state has a stride-0 (expanded) dimension and cannot be updated in place")
    out = torch.empty(x3.shape, dtype=x.dtype, device=x.device)
    code = _lib.dtype_code(x.dtype)
    _lib.launch("b200_causal_conv1d_update", x.device, x3.data_ptr(), code, *x3.stride(), conv_state.data_ptr(), *conv_state.stride(),
                weight.data_ptr(), _lib.dtype_code(weight.dtype), *weight.stride(), _lib.ptr(bias),
                0 if bias is None else _lib.dtype_code(bias.dtype), 0 if bias is None else bias.stride(0), out.data_ptr(), *out.stride(),
                batch, dim, seqlen, state_len, width, int(silu))
    return out if x.dim() == 3 else out.squeeze(-1)
