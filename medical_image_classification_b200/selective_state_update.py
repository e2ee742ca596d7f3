"""One recurrent step of a Mamba state -- host side of mamba_ssm 2.2.2's `selective_state_update`, the decode step that
mamba_ssm's `Mamba2.step` and transformers' `Mamba2Mixer.cuda_kernels_forward` call for every generated token:

    selective_state_update(state, x, dt, A, B, C, D=None, z=None, dt_bias=None, dt_softplus=False) -> out

Mamba-2 form: state (batch, nheads, headdim, dstate); x, dt, z (batch, nheads, headdim); A (nheads, headdim, dstate); B, C
(batch, ngroups, dstate); D, dt_bias (nheads, headdim).  Mamba-1 form: the same without the head dimension (state (batch, dim,
dstate), A (dim, dstate), B, C (batch, dstate), D, dt_bias (dim,)).  Head h reads group h // (nheads / ngroups); dstate <= 256.

In fp32:  dt' = softplus?(dt + dt_bias) (threshold 20),  state <- state * exp(A dt') + (B dt') x,  out = sum_n state C + D x,
then out *= silu(z).  `state` is updated in place in its own dtype; the sum uses the fp32 updated state before that rounding.
`out` has x's shape and dtype.  Nothing here is differentiable, as in mamba_ssm.

Every tensor is read in place through its strides in its own dtype (f32, bf16, f16), including stride-0 `expand`ed views and
column slices of a wider buffer, so transformers' argument sets run as one kernel launch with no copies; when A, dt and dt_bias
are constant over (headdim, dstate), exp(A dt') is formed once per (batch, head).  The work is done by csrc/state_update.cu through
b200_selective_state_update; there is no CPU path.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib


def _set(p, name, t, shape):
    """Point field `name` of p at t (None leaves it NULL), after checking t's shape, with its dtype code and strides."""
    if t is None:
        return
    if tuple(t.shape) != tuple(shape):
        raise RuntimeError(f"selective_state_update: {name} must be {tuple(shape)}, got {tuple(t.shape)}")
    setattr(p, name, t.data_ptr())
    setattr(p, name + "_dtype", _lib.dtype_code(t.dtype))
    setattr(p, name + "_stride", type(getattr(p, name + "_stride"))(*t.stride()))


@torch.no_grad()
def selective_state_update(state, x, dt, A, B, C, D=None, z=None, dt_bias=None, dt_softplus=False):
    """mamba_ssm's selective_state_update: advances `state` by one token in place and returns out (x's shape and dtype)."""
    _lib.require_cuda(state, x, dt, A, B, C, D, z, dt_bias)
    has_heads = state.dim() > 3
    if state.dim() not in (3, 4):
        raise RuntimeError(f"selective_state_update: state must be (batch, nheads, headdim, dstate) or (batch, dim, dstate), "
                           f"got {tuple(state.shape)}")
    if not has_heads:
        state = state.unsqueeze(1)
        x, dt, B, C = x.unsqueeze(1), dt.unsqueeze(1), B.unsqueeze(1), C.unsqueeze(1)
        A = A.unsqueeze(0)
        D = None if D is None else D.unsqueeze(0)
        z = None if z is None else z.unsqueeze(1)
        dt_bias = None if dt_bias is None else dt_bias.unsqueeze(0)
    batch, nheads, headdim, dstate = state.shape
    if B.dim() != 3:
        raise RuntimeError(f"selective_state_update: B must be (batch, ngroups, dstate), got {tuple(B.shape)}")
    ngroups = B.shape[1]
    if ngroups < 1 or nheads % ngroups:
        raise RuntimeError(f"selective_state_update: nheads = {nheads} is not a multiple of ngroups = {ngroups}")
    if dstate > 256:
        raise RuntimeError(f"selective_state_update: dstate = {dstate} exceeds 256")
    # a stride-0 dimension of the state would make several elements one memory location: the in-place update cannot be written
    if any(st == 0 and sz > 1 for sz, st in zip(state.shape, state.stride())):
        raise RuntimeError("selective_state_update: state has a stride-0 (expanded) dimension and cannot be updated in place")
    out = torch.empty(x.shape, dtype=x.dtype, device=x.device)
    p = _lib.SsuParams(batch=batch, nheads=nheads, headdim=headdim, ngroups=ngroups, dstate=dstate, dt_softplus=int(bool(dt_softplus)))
    _set(p, "state", state, (batch, nheads, headdim, dstate))
    _set(p, "x", x, (batch, nheads, headdim))
    _set(p, "dt", dt, (batch, nheads, headdim))
    _set(p, "A", A, (nheads, headdim, dstate))
    _set(p, "B", B, (batch, ngroups, dstate))
    _set(p, "C", C, (batch, ngroups, dstate))
    _set(p, "D", D, (nheads, headdim))
    _set(p, "z", z, (batch, nheads, headdim))
    _set(p, "dt_bias", dt_bias, (nheads, headdim))
    _set(p, "out", out, (batch, nheads, headdim))
    _lib.launch("b200_selective_state_update", state.device, ctypes.byref(p))
    return out if has_heads else out.squeeze(1)
