"""Mamba-1 selective scan operator -- host-side mirror of the reference's
`mamba_ssm.ops.selective_scan_interface` (reference
CrossMamba/FusionMamba/mamba_ssm/ops/selective_scan_interface.py:20-89): same function name,
argument meaning, return values and error behaviour (RuntimeError on bad input), but the work is
done by libb200ssm.so (hand-written sm_100a kernels, csrc/sscan.cu) through its C ABI
(include/b200_ssm.h).  There is no CPU path: CPU tensors raise.

    selective_scan_fn(u, delta, A, B, C, D=None, z=None, delta_bias=None,
                      delta_softplus=False, return_last_state=False)

u, delta: (batch, dim, L); A: (dim, N) real; B, C: (batch, N, L) or (batch, G, N, L);
D, delta_bias: (dim) fp32; z: (batch, dim, L).  Returns out (batch, dim, L) in u's dtype,
or (out, last_state (batch, dim, N) fp32).  last_state receives no gradient (interface.py:85-88).

`selective_scan_dirs_fn` is the same operator with the two SS2D extensions of the C ABI
(per-group time reversal and shared u rows), used by ss2d.SS2D.
"""
from __future__ import annotations

import ctypes as C

import torch


from ._lib import no_autocast as _no_autocast
from . import _lib

CKPT_EVERY = 8  # steps between state checkpoints written by the forward for the recompute backward

# Optional per-launch profiler (bench.py): an object with begin() -> token and
# end(token, kind, u, delta, Bm, algo_len), called immediately around the C-ABI launch on the current stream; algo_len is the
# caller's true sequence length when it runs the scan over rows padded to a 16-byte pitch (None otherwise).
_profiler = None


def set_profiler(p) -> None:
    global _profiler
    _profiler = p


def _last_contig(t):
    return t if t is None or t.stride(-1) == 1 else t.contiguous()


def _row_strides(t, rpg):
    """(batch, group, row) element strides of an activation given as (B, dim, L) or as a (B, G', rows, L) view."""
    if t.dim() == 4:
        return t.stride(0), t.stride(1), t.stride(2)
    return t.stride(0), rpg * t.stride(1), t.stride(1)


def _fill_fwd(p, u, delta, A, Bm, Cm, D, z, delta_bias, delta_softplus, rev_mask, u_group_div):
    """u, delta: (batch, dim, L), or 4-D views (batch, groups, rows per group, L) with arbitrary leading strides."""
    batch, L, dim = delta.shape[0], delta.shape[-1], A.shape[0]
    G, N = Bm.shape[1], Bm.shape[2]
    rpg = dim // G
    p.batch, p.dim, p.seqlen, p.dstate, p.n_groups = batch, dim, L, N, G
    p.io_dtype = _lib.dtype_code(u.dtype)
    p.delta_softplus = int(bool(delta_softplus))
    p.rev_mask = int(rev_mask)
    p.u_group_div = int(u_group_div)
    p.u_batch_stride, p.u_group_stride, p.u_row_stride = _row_strides(u, rpg)
    p.delta_batch_stride, p.delta_group_stride, p.delta_row_stride = _row_strides(delta, rpg)
    p.B_batch_stride, p.B_group_stride, p.B_state_stride = Bm.stride(0), Bm.stride(1), Bm.stride(2)
    p.C_batch_stride, p.C_group_stride, p.C_state_stride = Cm.stride(0), Cm.stride(1), Cm.stride(2)
    if z is not None:
        p.z_batch_stride, p.z_row_stride = z.stride(0), z.stride(1)
    p.u, p.delta, p.A, p.B, p.C = u.data_ptr(), delta.data_ptr(), A.data_ptr(), Bm.data_ptr(), Cm.data_ptr()
    p.D, p.z, p.delta_bias = _lib.ptr(D), _lib.ptr(z), _lib.ptr(delta_bias)


def _check_inputs(u, delta, A, B, C, D, z, delta_bias, u_group_div):
    _lib.require_cuda(u, delta, A, B, C, D, z, delta_bias)
    if u.dim() != 3 or delta.dim() != 3:
        raise RuntimeError(f"selective_scan: u and delta must be (batch, dim, L), got {tuple(u.shape)} / {tuple(delta.shape)}")
    if A.is_complex():
        raise RuntimeError("selective_scan: complex A is not supported by the B200 kernels (unused by the reference models)")
    batch, dim, L = delta.shape
    if A.dim() != 2 or A.shape[0] != dim:
        raise RuntimeError(f"selective_scan: A must be (dim={dim}, dstate), got {tuple(A.shape)}")
    if B.dim() not in (3, 4) or C.dim() not in (3, 4):
        raise RuntimeError("selective_scan: only input-dependent B/C of shape (batch, [groups,] dstate, L) are supported")
    if u.dtype != delta.dtype:
        raise RuntimeError(f"selective_scan: u ({u.dtype}) and delta ({delta.dtype}) must share a dtype")
    if u.shape[0] != batch or u.shape[2] != L or u.shape[1] * u_group_div != dim:
        raise RuntimeError(f"selective_scan: u {tuple(u.shape)} does not match delta {tuple(delta.shape)}")
    for name, t in (("D", D), ("delta_bias", delta_bias)):
        if t is not None and tuple(t.shape) != (dim,):
            raise RuntimeError(f"selective_scan: {name} must have shape ({dim},), got {tuple(t.shape)}")
    if z is not None and tuple(z.shape) != (batch, dim, L):
        raise RuntimeError(f"selective_scan: z must be {(batch, dim, L)}, got {tuple(z.shape)}")


def launch_fwd(u, delta, A32, Bm, Cm, D32, z, bias32, delta_softplus, rev_mask=0, u_group_div=1,
               want_ckpt=False, want_last_state=False, algo_len=None):
    """One b200_sscan_fwd call on prepared tensors (last stride 1, B/C 4-D, A/D/bias fp32 contiguous).
    Returns (out, last_state | None, ckpt | None)."""
    batch, L, dim = delta.shape[0], delta.shape[-1], A32.shape[0]
    G, N = Bm.shape[1], Bm.shape[2]
    out = torch.empty((batch, dim, L), dtype=u.dtype, device=u.device)
    ckpt = None
    if want_ckpt:
        nbytes = _lib.load().b200_sscan_ckpt_bytes(batch, dim, L, N, G, CKPT_EVERY)
        ckpt = torch.empty(nbytes // 4, dtype=torch.float32, device=u.device)
    last_state = torch.empty((batch, dim, N), dtype=torch.float32, device=u.device) if want_last_state else None
    p = _lib.SScanFwdParams()
    _fill_fwd(p, u, delta, A32, Bm, Cm, D32, z, bias32, delta_softplus, rev_mask, u_group_div)
    p.ckpt_every = CKPT_EVERY
    p.out_batch_stride, p.out_row_stride = out.stride(0), out.stride(1)
    p.out, p.last_state, p.ckpt = out.data_ptr(), _lib.ptr(last_state), _lib.ptr(ckpt)
    prof = _profiler
    with torch.cuda.device(u.device):
        tok = prof.begin() if prof is not None else None
        _lib.launch("b200_sscan_fwd", u.device, C.byref(p))
        if prof is not None:
            prof.end(tok, "fwd", u, delta, Bm, algo_len)
    return out, last_state, ckpt


def launch_bwd(u, delta, A32, Bm, Cm, D32, z, bias32, delta_softplus, ckpt, dout, rev_mask=0,
               u_group_div=1, dout_group_div=1, has_D=True, has_bias=True, ddelta=None, dB=None, dC=None, algo_len=None):
    """One b200_sscan_bwd call.  `dout` is (batch, dim / dout_group_div, L).
    Returns du (batch, dim, L), ddelta, dA, dB, dC (fp32), dD, ddelta_bias, dz.
    ddelta (batch, G, rows per group, L) and dB, dC (batch, G, N, L; fp32, ZERO-FILLED by the caller) may be passed as
    views into a wider buffer (last stride 1); they are then written / accumulated in place."""
    batch, L, dim = delta.shape[0], delta.shape[-1], A32.shape[0]
    G, N = Bm.shape[1], Bm.shape[2]
    rpg = dim // G
    dev = u.device
    du = torch.empty((batch, dim, L), dtype=u.dtype, device=dev)
    if ddelta is None:
        ddelta = torch.empty((batch, dim, L), dtype=u.dtype, device=dev)
    dz = torch.empty((batch, dim, L), dtype=u.dtype, device=dev) if z is not None else None
    # fp32 accumulators for everything reduced with atomics (selective_scan.cpp:460-466)
    if dB is None:
        dB = torch.zeros((batch, G, N, L), dtype=torch.float32, device=dev)
    if dC is None:
        dC = torch.zeros((batch, G, N, L), dtype=torch.float32, device=dev)
    dA = torch.zeros((dim, N), dtype=torch.float32, device=dev)
    dD = torch.zeros(dim, dtype=torch.float32, device=dev) if has_D else None
    dbias = torch.zeros(dim, dtype=torch.float32, device=dev) if has_bias else None
    q = _lib.SScanBwdParams()
    _fill_fwd(q.f, u, delta, A32, Bm, Cm, D32, z, bias32, delta_softplus, rev_mask, u_group_div)
    q.f.ckpt_every = CKPT_EVERY
    q.f.ckpt = ckpt.data_ptr()
    q.dout_batch_stride, q.dout_row_stride = dout.stride(0), dout.stride(1)
    q.dout_group_stride, q.dout_group_div = rpg * dout.stride(1), int(dout_group_div)
    q.du_batch_stride, q.du_row_stride = du.stride(0), du.stride(1)
    q.ddelta_batch_stride, q.ddelta_group_stride, q.ddelta_row_stride = _row_strides(ddelta, rpg)
    q.dB_batch_stride, q.dB_group_stride, q.dB_state_stride = dB.stride(0), dB.stride(1), dB.stride(2)
    q.dC_batch_stride, q.dC_group_stride, q.dC_state_stride = dC.stride(0), dC.stride(1), dC.stride(2)
    if dz is not None:
        q.dz_batch_stride, q.dz_row_stride = dz.stride(0), dz.stride(1)
    q.dout, q.du, q.ddelta, q.dz = dout.data_ptr(), du.data_ptr(), ddelta.data_ptr(), _lib.ptr(dz)
    q.dA, q.dB, q.dC, q.dD, q.ddelta_bias = dA.data_ptr(), dB.data_ptr(), dC.data_ptr(), _lib.ptr(dD), _lib.ptr(dbias)
    prof = _profiler
    with torch.cuda.device(dev):
        tok = prof.begin() if prof is not None else None
        _lib.launch("b200_sscan_bwd", dev, C.byref(q))
        if prof is not None:
            prof.end(tok, "bwd", u, delta, Bm, algo_len)
    return du, ddelta, dA, dB, dC, dD, dbias, dz


class SelectiveScanFn(torch.autograd.Function):
    """Mirror of reference SelectiveScanFn (selective_scan_interface.py:20-80)."""

    @staticmethod
    @_no_autocast
    def forward(ctx, u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False,
                return_last_state=False, rev_mask=0, u_group_div=1):
        _check_inputs(u, delta, A, B, C, D, z, delta_bias, u_group_div)
        u, delta, z = _last_contig(u), _last_contig(delta), _last_contig(z)
        ctx.squeeze_B = B.dim() == 3
        ctx.squeeze_C = C.dim() == 3
        Bm = B.unsqueeze(1) if B.dim() == 3 else B
        Cm = C.unsqueeze(1) if C.dim() == 3 else C
        ctx.B_dtype, ctx.C_dtype = B.dtype, C.dtype
        Bm = _last_contig(Bm.to(u.dtype))
        Cm = _last_contig(Cm.to(u.dtype))
        if z is not None:
            z = z.to(u.dtype)
        batch, dim, L = delta.shape
        G, N = Bm.shape[1], Bm.shape[2]
        if Bm.shape != Cm.shape or Bm.shape[0] != batch or Bm.shape[3] != L or dim % G != 0 or A.shape[1] != N:
            raise RuntimeError(f"selective_scan: B {tuple(B.shape)} / C {tuple(C.shape)} do not match "
                               f"delta {tuple(delta.shape)} and A {tuple(A.shape)}")
        A32, D32, bias32 = _lib.f32c(A), _lib.f32c(D), _lib.f32c(delta_bias)
        need_grad = any(ctx.needs_input_grad)
        out, last_state, ckpt = launch_fwd(u, delta, A32, Bm, Cm, D32, z, bias32, delta_softplus, rev_mask,
                                           u_group_div, want_ckpt=need_grad, want_last_state=return_last_state)
        ctx.delta_softplus = bool(delta_softplus)
        ctx.rev_mask, ctx.u_group_div = int(rev_mask), int(u_group_div)
        ctx.has_D, ctx.has_bias = D is not None, delta_bias is not None
        ctx.A_dtype = A.dtype
        ctx.D_dtype = D.dtype if D is not None else None
        ctx.bias_dtype = delta_bias.dtype if delta_bias is not None else None
        if need_grad:
            ctx.save_for_backward(u, delta, A32, Bm, Cm, D32, z, bias32, ckpt)
        if return_last_state:
            ctx.mark_non_differentiable(last_state)
            return out, last_state
        return out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout, *args):
        u, delta, A32, Bm, Cm, D32, z, bias32, ckpt = ctx.saved_tensors
        dout = _last_contig(dout.to(u.dtype))
        batch, dim, L = delta.shape
        G = Bm.shape[1]
        du, ddelta, dA, dB, dC, dD, dbias, dz = launch_bwd(
            u, delta, A32, Bm, Cm, D32, z, bias32, ctx.delta_softplus, ckpt, dout, ctx.rev_mask,
            ctx.u_group_div, 1, ctx.has_D, ctx.has_bias)
        if ctx.u_group_div > 1:  # directions sharing one u row: their du add up
            rpg = dim // G
            du = du.view(batch, G // ctx.u_group_div, ctx.u_group_div, rpg, L).sum(2).view(batch, -1, L)
        dB = dB.to(ctx.B_dtype)
        dC = dC.to(ctx.C_dtype)
        if ctx.squeeze_B:
            dB = dB.squeeze(1)
        if ctx.squeeze_C:
            dC = dC.squeeze(1)
        return (du, ddelta, dA.to(ctx.A_dtype), dB, dC,
                dD.to(ctx.D_dtype) if dD is not None else None,
                dz,
                dbias.to(ctx.bias_dtype) if dbias is not None else None,
                None, None, None, None)


MAX_DSTATE_PER_CALL = 16     # one kernel call carries 16 states per row in registers (csrc/sscan*.cu)
MAX_DSTATE = 256             # the reference's limit (selective_scan.cpp:262)


def selective_scan_fn(u, delta, A, B, C, D=None, z=None, delta_bias=None, delta_softplus=False,
                      return_last_state=False):
    """if return_last_state is True, returns (out, last_state); last_state has shape
    (batch, dim, dstate) and gets no gradient (reference selective_scan_interface.py:83-89).

    dstate up to 256 like the reference (selective_scan.cpp:262).  The recurrence is independent per state and y is a sum over
    states, so wider state spaces (no model of the reference repo uses one: every SS2D has d_state 16) run as ceil(dstate / 16)
    calls on 16-state slices of A, B and C whose outputs add up; D u, the z gate and the concatenation of last_state are applied
    once around them with tensor ops, and autograd sums the slices' gradients of u, delta and delta_bias."""
    N = A.shape[1] if hasattr(A, "shape") and A.dim() == 2 else 0
    if N <= MAX_DSTATE_PER_CALL:
        return SelectiveScanFn.apply(u, delta, A, B, C, D, z, delta_bias, delta_softplus, return_last_state)
    if N > MAX_DSTATE:
        raise RuntimeError(f"selective_scan: dstate {N} > {MAX_DSTATE} (the reference's limit, selective_scan.cpp:262)")
    sdim = B.dim() - 2                                       # the state dimension of B / C: (b, n, l) or (b, g, n, l)
    y, lasts = None, []
    for n0 in range(0, N, MAX_DSTATE_PER_CALL):
        n1 = min(N, n0 + MAX_DSTATE_PER_CALL)
        r = SelectiveScanFn.apply(u, delta, A[:, n0:n1], B.narrow(sdim, n0, n1 - n0), C.narrow(sdim, n0, n1 - n0), None, None,
                                  delta_bias, delta_softplus, return_last_state)
        if return_last_state:
            r, last = r
            lasts.append(last)
        y = r if y is None else y + r
    if D is not None:
        y = y + (u * D.to(u.dtype).view(1, -1, 1)).to(y.dtype)
    if z is not None:
        y = y * torch.nn.functional.silu(z.to(y.dtype))
    return (y, torch.cat(lasts, dim=-1)) if return_last_state else y


def selective_scan_dirs_fn(u, delta, A, B, C, D=None, delta_bias=None, delta_softplus=False,
                           rev_mask=0, u_group_div=1):
    """The same operator with per-group time reversal (`rev_mask`, bit g) and `u_group_div`
    consecutive groups reading the same u rows: u is (batch, dim / u_group_div, L)."""
    return SelectiveScanFn.apply(u, delta, A, B, C, D, None, delta_bias, delta_softplus, False,
                                 rev_mask, u_group_div)


# The reference file also exports its pure-PyTorch oracle under this name; the product package
# deliberately has none (no CPU fallback) -- tests use the separate `oracle` package.
def selective_scan_ref(*args, **kwargs):  # pragma: no cover
    raise RuntimeError("medical_image_classification_b200 ships no CPU reference path; "
                       "use oracle.sscan_fwd / the reference's selective_scan_ref for checking")
