"""Mamba-2 SSD chunked scan -- host-side mirror of `mamba_ssm.ops.triton.ssd_combined`
(mamba_ssm==2.2.2, not vendored in the reference; call contract: reference SSD/MedSSD.py:41,361-375):

    mamba_chunk_scan_combined(x, dt, A, B, C, chunk_size, D=None, z=None, dt_bias=None,
                              initial_states=None, seq_idx=None, cu_seqlens=None, dt_softplus=False,
                              dt_limit=(0.0, inf), return_final_states=False, return_varlen_states=False)

x (batch, L, H, P); dt (batch, L, H); A (H); B, C (batch, L, G, N); D (H) or (H, P); z like x;
dt_bias (H); initial_states (batch, H, P, N).  Returns out (batch, L, H, P) in x's dtype
[, final_states (batch, H, P, N) fp32][, varlen_states (nseq, H, P, N) fp32].  Tensors are taken with
whatever strides they have (the reference passes (b, l, .) views of channel-major storage, L stride 1)
-- nothing is copied.

Gradients flow into initial_states (in its dtype) and out of final_states, as in mamba_ssm 2.2.2, so a
long sequence can be trained over several calls that pass the state along; varlen_states carries none.
A backward that needs neither runs exactly the kernels it would without them.

Packed sequences: seq_idx (batch, L) integers, non-decreasing along L (the caller's contract, not
checked: that would need a host sync), restarts the recurrence wherever it changes, in the forward
and in the backward; initial_states[b] reach row b's first sequence only when its id is 0 (so only
such a row gets a non-zero initial_states gradient), and the final_states gradient reaches only the
row's last sequence.
return_varlen_states (batch 1, cu_seqlens (nseq + 1,) giving the same boundaries) also returns the
state after each sequence's last token.  It differs from mamba_ssm in one case: a first sequence that
ends inside the first chunk includes initial_states, as out and final_states do.

The work is done by libb200ssm.so (csrc/ssd.cu, sm_100a tensor-core kernels) through its C ABI
(include/b200_ssm.h: b200_ssd_fwd / b200_ssd_bwd / b200_ssd_varlen_states).  There is no CPU path:
CPU tensors raise.
"""
from __future__ import annotations

import ctypes

import torch

import torch.nn.functional as F

from ._lib import no_autocast as _no_autocast
from . import _lib
from .conv1d import act_is_silu, check_weight, conv_bwd, conv_fwd

# 0: fp32-accurate tensor-core products (3xTF32 split, default); 1: single-pass TF32 (the arithmetic
# of the reference's Triton kernels on fp32 inputs: tl.dot with its default allow_tf32).  Under bf16 autocast --
# BASELINE.json configs[2], where everything around the operator is bf16 -- the single-pass mode is used unless
# set_precision() was called explicitly: it is exactly the reference's own arithmetic for this call.
_precision = 0
_explicit = False

# Optional per-call profiler (bench.py --model medssd): an object with begin() -> token and end(token, kind, shape), called
# immediately around the C-ABI call on the current stream; shape = (batch, L, H, P, G, N, chunk, precision).
_profiler = None


def set_profiler(p) -> None:
    global _profiler
    _profiler = p


def _effective_precision() -> int:
    if not _explicit and torch.is_autocast_enabled():
        return 1
    return _precision


def set_precision(mode) -> None:
    """0 / 1 fix the mode; None returns to the default policy (fp32-accurate, single-pass TF32 under autocast)."""
    global _precision, _explicit
    if mode is None:
        _precision, _explicit = 0, False
        return
    if mode not in (0, 1):
        raise ValueError("precision must be 0 (3xTF32, fp32-accurate) or 1 (single-pass TF32)")
    _precision = mode
    _explicit = True


def _fill_fwd(p, x, dt, A, Bm, Cm, D, dt_bias, chunk_size, dt_softplus, dt_limit, initial_states, precision, seq_idx):
    batch, L, H, P = x.shape
    G, N = Bm.shape[2], Bm.shape[3]
    p.batch, p.seqlen, p.nheads, p.headdim, p.n_groups, p.dstate, p.chunk_size = batch, L, H, P, G, N, chunk_size
    p.io_dtype = _lib.dtype_code(x.dtype)
    p.dt_softplus = int(bool(dt_softplus))
    p.precision = int(precision)
    p.dt_min, p.dt_max = float(dt_limit[0]), float(min(dt_limit[1], 3.0e38))
    for name, t in (("x_stride", x), ("B_stride", Bm), ("C_stride", Cm)):
        getattr(p, name)[:] = list(t.stride())
    p.dt_stride[:] = list(dt.stride())
    p.x, p.dt, p.A, p.B, p.C = x.data_ptr(), dt.data_ptr(), A.data_ptr(), Bm.data_ptr(), Cm.data_ptr()
    p.D, p.dt_bias, p.initial_states = _lib.ptr(D), _lib.ptr(dt_bias), _lib.ptr(initial_states)
    if seq_idx is not None:
        p.seq_idx = seq_idx.data_ptr()
        p.seq_idx_stride[:] = list(seq_idx.stride())


def _empty_like_layout(t):
    """fp32 tensor of t's shape with t's strides when t is dense (any dimension order), contiguous otherwise."""
    if _lib.is_dense(t):
        return torch.empty_strided(t.shape, t.stride(), dtype=torch.float32, device=t.device)
    return torch.empty(t.shape, dtype=torch.float32, device=t.device)


def _ssd_fwd(x, dt_, A32, B_, C_, D32, bias32, init32, seq_idx, chunk_size, dt_softplus, dt_limit, prec, out, fin):
    """Run b200_ssd_fwd into out (and fin when given); returns (workspace, params)."""
    batch, L, H, P = x.shape
    G, N = B_.shape[2], B_.shape[3]
    dev = x.device
    nbytes = _lib.load().b200_ssd_workspace_bytes(batch, L, H, P, G, N, chunk_size)
    ws = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    p = _lib.SsdFwdParams()
    _fill_fwd(p, x, dt_, A32, B_, C_, D32, bias32, chunk_size, dt_softplus, dt_limit, init32, prec, seq_idx)
    p.out_stride[:] = list(out.stride())
    p.out, p.final_states, p.workspace = out.data_ptr(), _lib.ptr(fin), ws.data_ptr()
    prof = _profiler
    with torch.cuda.device(dev):
        tok = prof.begin() if prof is not None else None
        _lib.launch("b200_ssd_fwd", dev, ctypes.byref(p))
        if prof is not None:
            prof.end(tok, "fwd", (batch, L, H, P, G, N, chunk_size, prec))
    return ws, p


def _ssd_bwd(x, dt_, A32, B_, C_, D32, bias32, init32, seq_idx, out, ws, fin, cfg, dout, dfin, dx, ddt, dB, dC, dinit):
    """Run b200_ssd_bwd, writing dx / ddt / dB / dC (fp32, any strides) and dinit (or None) in place; returns (dA, dD, ddt_bias),
    fp32, None where the primal is None."""
    chunk_size, dt_softplus, dt_limit, precision = cfg
    batch, L, H, P = x.shape
    G, N = B_.shape[2], B_.shape[3]
    dev = x.device
    dA = torch.zeros(H, dtype=torch.float32, device=dev)
    dD = torch.zeros(H, dtype=torch.float32, device=dev) if D32 is not None else None
    dbias = torch.zeros(H, dtype=torch.float32, device=dev) if bias32 is not None else None
    nbytes = _lib.load().b200_ssd_bwd_scratch_bytes(batch, L, H, P, G, N, chunk_size)
    scratch = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    q = _lib.SsdBwdParams()
    _fill_fwd(q.f, x, dt_, A32, B_, C_, D32, bias32, chunk_size, dt_softplus, dt_limit, init32, precision, seq_idx)
    q.f.out_stride[:] = list(out.stride())
    q.f.out, q.f.workspace = out.data_ptr(), ws.data_ptr()
    q.dout_stride[:] = list(dout.stride())
    q.dout, q.dx, q.ddt, q.dB, q.dC = dout.data_ptr(), dx.data_ptr(), ddt.data_ptr(), dB.data_ptr(), dC.data_ptr()
    q.dx_stride[:], q.ddt_stride[:] = list(dx.stride()), list(ddt.stride())
    q.dB_stride[:], q.dC_stride[:] = list(dB.stride()), list(dC.stride())
    q.dA, q.dD, q.ddt_bias, q.scratch = dA.data_ptr(), _lib.ptr(dD), _lib.ptr(dbias), scratch.data_ptr()
    q.final_states, q.dfinal_states, q.dinitial_states = _lib.ptr(fin), _lib.ptr(dfin), _lib.ptr(dinit)
    prof = _profiler
    with torch.cuda.device(dev):
        tok = prof.begin() if prof is not None else None
        _lib.launch("b200_ssd_bwd", dev, ctypes.byref(q))
        if prof is not None:
            prof.end(tok, "bwd", (batch, L, H, P, G, N, chunk_size, precision))
    return dA, dD, dbias


class SsdChunkScanFn(torch.autograd.Function):
    @staticmethod
    @_no_autocast
    def forward(ctx, x, dt, A, B, C, D, dt_bias, initial_states, seq_idx, cu_seqlens, chunk_size, dt_softplus, dt_limit,
                return_final_states, prec):
        batch, L, H, P = x.shape
        N = B.shape[3]
        dev = x.device
        dt_, B_, C_ = dt.to(x.dtype), B.to(x.dtype), C.to(x.dtype)
        A32, D32, bias32, init32 = _lib.f32c(A), _lib.f32c(D), _lib.f32c(dt_bias), _lib.f32c(initial_states)
        out = torch.empty((batch, L, H, P), dtype=x.dtype, device=dev)
        fin = torch.empty((batch, H, P, N), dtype=torch.float32, device=dev) if return_final_states else None
        ws, p = _ssd_fwd(x, dt_, A32, B_, C_, D32, bias32, init32, seq_idx, chunk_size, dt_softplus, dt_limit, prec, out, fin)
        extra = (fin,) if return_final_states else ()
        if cu_seqlens is not None:      # return_varlen_states: reads this call's workspace
            nseq = cu_seqlens.shape[0] - 1
            varlen = torch.empty((nseq, H, P, N), dtype=torch.float32, device=dev)
            if nseq > 0:
                _lib.launch("b200_ssd_varlen_states", dev, ctypes.byref(p), cu_seqlens.data_ptr(), nseq, varlen.data_ptr())
            extra += (varlen,)
        ctx.save_for_backward(x, dt_, A32, B_, C_, D32, bias32, init32, seq_idx, out, ws, fin)
        ctx.cfg = (chunk_size, bool(dt_softplus), tuple(dt_limit), prec)
        ctx.dtypes = (dt.dtype, A.dtype, B.dtype, C.dtype, None if D is None else D.dtype,
                      None if dt_bias is None else dt_bias.dtype, None if initial_states is None else initial_states.dtype)
        # an output the loss does not use arrives in backward as None (not a zero tensor), so a final_states that takes
        # no part in the loss costs nothing
        ctx.set_materialize_grads(False)
        if cu_seqlens is not None:
            ctx.mark_non_differentiable(extra[-1])
        return (out,) + extra if extra else out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout, *dextra):
        x, dt_, A32, B_, C_, D32, bias32, init32, seq_idx, out, ws, fin = ctx.saved_tensors
        dfin = dextra[0] if fin is not None else None
        dout = torch.zeros_like(out) if dout is None else dout.to(x.dtype)
        dfin = None if dfin is None else _lib.f32c(dfin)
        dinit = torch.empty_like(init32) if ctx.needs_input_grad[7] else None
        # every gradient in the layout of its primal (the models pass sequence-contiguous views of channel-major storage,
        # SSD/MedSSD.py:344-347): the cross-scan adjoint then reads them in place -- no strided copy after the kernels
        dx, ddt, dB, dC = (_empty_like_layout(t) for t in (x, dt_, B_, C_))
        dA, dD, dbias = _ssd_bwd(x, dt_, A32, B_, C_, D32, bias32, init32, seq_idx, out, ws, fin, ctx.cfg, dout, dfin, dx, ddt, dB,
                                 dC, dinit)
        t_dt, t_A, t_B, t_C, t_D, t_bias, t_init = ctx.dtypes
        return (dx.to(x.dtype), ddt.to(t_dt), dA.to(t_A), dB.to(t_B), dC.to(t_C),
                None if dD is None else dD.to(t_D), None if dbias is None else dbias.to(t_bias),
                None if dinit is None else dinit.to(t_init), None, None, None, None, None, None, None)


def mamba_chunk_scan_combined(x, dt, A, B, C, chunk_size, D=None, z=None, dt_bias=None, initial_states=None,
                              seq_idx=None, cu_seqlens=None, dt_softplus=False, dt_limit=(0.0, float("inf")),
                              return_final_states=False, return_varlen_states=False):
    """Argument:
        x: (batch, seqlen, nheads, headdim)    dt: (batch, seqlen, nheads)    A: (nheads)
        B, C: (batch, seqlen, ngroups, dstate)  chunk_size: int
        D: (nheads, headdim) or (nheads,)       z: (batch, seqlen, nheads, headdim)
        dt_bias: (nheads,)                      initial_states: (batch, nheads, headdim, dstate)
        seq_idx: (batch, seqlen) integers, non-decreasing along seqlen: the recurrence restarts where it changes
        cu_seqlens: (nseq + 1,) integers, sequence boundaries of the packed row; used by return_varlen_states (batch 1)
        dt_softplus: whether to apply softplus to dt
    Return:
        out: (batch, seqlen, nheads, headdim) [, final_states (batch, nheads, headdim, dstate)]
        [, varlen_states (nseq, nheads, headdim, dstate): the state after each sequence's last token]
    final_states and varlen_states are fp32.  initial_states receives a gradient in its own dtype, and final_states
    passes one back (with seq_idx: to row b's leading id-0 sequence and from its last sequence); varlen_states carries none.
    """
    _lib.require_cuda(x, dt, A, B, C, D, z, dt_bias, initial_states, seq_idx)
    if x.dim() != 4 or dt.dim() != 3 or B.dim() != 4 or C.dim() != 4:
        raise RuntimeError(f"mamba_chunk_scan_combined: expected x (b,l,h,p), dt (b,l,h), B/C (b,l,g,n); got "
                           f"{tuple(x.shape)}, {tuple(dt.shape)}, {tuple(B.shape)}, {tuple(C.shape)}")
    batch, L, H, P = x.shape
    G, N = B.shape[2], B.shape[3]
    if tuple(dt.shape) != (batch, L, H) or tuple(A.shape) != (H,) or tuple(C.shape) != tuple(B.shape) \
            or B.shape[:2] != (batch, L) or H % G != 0:
        raise RuntimeError("mamba_chunk_scan_combined: inconsistent shapes "
                           f"x {tuple(x.shape)} dt {tuple(dt.shape)} A {tuple(A.shape)} B {tuple(B.shape)} C {tuple(C.shape)}")
    if dt_bias is not None and tuple(dt_bias.shape) != (H,):
        raise RuntimeError(f"mamba_chunk_scan_combined: dt_bias must be ({H},), got {tuple(dt_bias.shape)}")
    if initial_states is not None:
        if tuple(initial_states.shape) != (batch, H, P, N):
            raise RuntimeError(f"mamba_chunk_scan_combined: initial_states must be {(batch, H, P, N)}")
    seq_idx = _index_tensor(seq_idx, "seq_idx", x.device, (batch, L))
    if return_varlen_states:
        if cu_seqlens is None:
            raise RuntimeError("mamba_chunk_scan_combined: return_varlen_states needs cu_seqlens")
        if batch != 1:
            raise RuntimeError(f"mamba_chunk_scan_combined: return_varlen_states needs batch == 1 (packed sequences), got {batch}")
        if cu_seqlens.dim() != 1 or cu_seqlens.shape[0] < 1:
            raise RuntimeError(f"mamba_chunk_scan_combined: cu_seqlens must be 1-D (nseq + 1,), got {tuple(cu_seqlens.shape)}")
        cu_seqlens = _index_tensor(cu_seqlens, "cu_seqlens", x.device, tuple(cu_seqlens.shape))
    else:
        cu_seqlens = None          # accepted and unused, as in mamba_ssm
    D_head = None
    if D is not None:
        if tuple(D.shape) == (H,):
            D_head = D
        elif tuple(D.shape) != (H, P):
            raise RuntimeError(f"mamba_chunk_scan_combined: D must be ({H},) or ({H}, {P}), got {tuple(D.shape)}")
    chunk_size = int(chunk_size)
    if chunk_size < 1:
        raise RuntimeError(f"mamba_chunk_scan_combined: chunk_size must be positive, got {chunk_size}")
    # The result does not depend on the chunk length (it only decides where the recurrence is cut: tests' chunk-size invariance),
    # so every chunk_size mamba_ssm accepts (any power of two >= 16; the reference passes 256, SSD/MedSSD.py:365) is honoured by
    # running the kernels on the nearest length they tile: a multiple of 32 in [32, 256].
    chunk_size = min(256, (chunk_size + 31) // 32 * 32)
    res = SsdChunkScanFn.apply(x, dt, A, B, C, D_head, dt_bias, initial_states, seq_idx, cu_seqlens, chunk_size, dt_softplus,
                               (float(dt_limit[0]), float(dt_limit[1])), return_final_states,
                               _effective_precision())   # read here: autocast is off inside the Function
    out, extra = (res[0], res[1:]) if isinstance(res, tuple) else (res, ())
    if D is not None and D_head is None:      # D with a head dimension: plain PyTorch on the side (unused by the models)
        out = out + x * D.to(x.dtype)
    if z is not None:                         # out * silu(z), as mamba_ssm does when no norm is fused
        out = out * F.silu(z)
    return (out,) + extra if extra else out


def _index_tensor(t, name, device, shape, op="mamba_chunk_scan_combined"):
    """t as the int32 tensor the kernels read (in place when it already is int32 with a unit last stride); None stays None."""
    if t is None:
        return None
    if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool:
        raise RuntimeError(f"{op}: {name} must hold integers, got {t.dtype}")
    if tuple(t.shape) != shape:
        raise RuntimeError(f"{op}: {name} must be {shape}, got {tuple(t.shape)}")
    if t.device != device:
        raise RuntimeError(f"{op}: {name} is on {t.device}, x on {device}")
    if t.dtype != torch.int32 or (t.shape[-1] > 1 and t.stride(-1) != 1):
        t = t.to(torch.int32).contiguous()
    return t


# ------------------------------------------------------------------------------------------------
# gated RMSNorm (mamba_ssm.ops.triton.layernorm_gated.RMSNorm / rmsnorm_fn, mamba_ssm 2.2.2, as used at
# SSD/MedSSD.py:268-269,393-394): csrc/rmsnorm.cu through b200_rmsnorm_fwd / _bwd
# ------------------------------------------------------------------------------------------------
_IO_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


def _rows_io(t, dim):
    """(tensor, row stride) of t as the kernels read it: in place when its dtype is one they read and its rows are contiguous."""
    return _lib.rows_view(t if t.dtype in _IO_DTYPES else t.float(), dim)


def _rmsnorm_launch_fwd(x2, xs, z2, zs, w32, b32, rows, dim, eps, group_size, nbg, out_dtype):
    """b200_rmsnorm_fwd on rows of x2 / z2 (row strides xs / zs): returns out (rows, dim) out_dtype and rstd (rows, groups)."""
    out = torch.empty((rows, dim), dtype=out_dtype, device=x2.device)
    rstd = torch.empty((rows, dim // group_size), dtype=torch.float32, device=x2.device)
    _lib.launch("b200_rmsnorm_fwd", x2.device, x2.data_ptr(), _lib.dtype_code(x2.dtype), xs, _lib.ptr(z2),
                _lib.dtype_code(z2.dtype) if z2 is not None else 0, zs, w32.data_ptr(), _lib.ptr(b32), out.data_ptr(),
                _lib.dtype_code(out_dtype), rstd.data_ptr(), rows, dim, group_size, int(nbg), float(eps))
    return out, rstd


def _rmsnorm_launch_bwd(dy2, dys, x2, xs, z2, zs, w32, b32, rstd, rows, dim, group_size, nbg):
    """b200_rmsnorm_bwd: returns dx (rows, dim) in x2's dtype, dz in z2's (or None) and the summed (dweight[, dbias]) fp32."""
    dev = dy2.device
    dx = torch.empty((rows, dim), dtype=x2.dtype, device=dev)
    dz = torch.empty((rows, dim), dtype=z2.dtype, device=dev) if z2 is not None else None
    grid = _lib.load().b200_rmsnorm_grid(rows, dim, group_size)
    if grid < 0:
        _lib.check(grid, "b200_rmsnorm_grid")
    part = torch.empty((1 if b32 is None else 2, grid, dim), dtype=torch.float32, device=dev)
    _lib.launch("b200_rmsnorm_bwd", dev, dy2.data_ptr(), _lib.dtype_code(dy2.dtype), dys, x2.data_ptr(), _lib.dtype_code(x2.dtype),
                xs, _lib.ptr(z2), _lib.dtype_code(z2.dtype) if z2 is not None else 0, zs, w32.data_ptr(), _lib.ptr(b32),
                rstd.data_ptr(), dx.data_ptr(), _lib.ptr(dz), part[0].data_ptr(), part[1].data_ptr() if b32 is not None else None,
                rows, dim, group_size, int(nbg))
    return dx, dz, part.sum(1)


class RmsNormGatedFn(torch.autograd.Function):
    """out = rmsnorm_g(x * silu(z)) * w + b (norm_before_gate=False), (rmsnorm_g(x) * w + b) * silu(z) (True), or
    rmsnorm_g(x) * w + b (z None), each group of group_size columns normalised on its own.  x, z and dy are read in place when
    their rows are contiguous (z is a column slice of in_proj's output); out is out_dtype; gradients come back in the primals'
    dtypes."""

    @staticmethod
    @_no_autocast
    def forward(ctx, x, z, weight, bias, eps, group_size, norm_before_gate, out_dtype):
        _lib.require_cuda(x, z, weight, bias)
        dim = x.shape[-1]
        rows = x.numel() // dim
        x2, xs = _rows_io(x, dim)
        z2, zs = _rows_io(z, dim) if z is not None else (None, 0)
        w32, b32 = _lib.f32c(weight), _lib.f32c(bias)
        out, rstd = _rmsnorm_launch_fwd(x2, xs, z2, zs, w32, b32, rows, dim, eps, group_size, norm_before_gate, out_dtype)
        ctx.save_for_backward(x2, z2, w32, b32, rstd)
        ctx.cfg = (xs, zs, rows, group_size, int(norm_before_gate))
        ctx.dtypes = (x.dtype, None if z is None else z.dtype, weight.dtype, None if bias is None else bias.dtype)
        return out.view(x.shape)

    @staticmethod
    @_no_autocast
    def backward(ctx, dy):
        x2, z2, w32, b32, rstd = ctx.saved_tensors
        xs, zs, rows, group_size, nbg = ctx.cfg
        t_x, t_z, t_w, t_b = ctx.dtypes
        shape, dim, dev = dy.shape, dy.shape[-1], dy.device
        dy2, dys = _rows_io(dy, dim)
        dx, dz, dwb = _rmsnorm_launch_bwd(dy2, dys, x2, xs, z2, zs, w32, b32, rstd, rows, dim, group_size, nbg)
        return (dx.view(shape).to(t_x), None if dz is None else dz.view(shape).to(t_z), dwb[0].to(t_w),
                None if b32 is None else dwb[1].to(t_b), None, None, None, None)


def _rmsnorm(x, z, weight, bias, eps, group_size, norm_before_gate, out_dtype):
    dim = x.shape[-1]
    group_size = dim if group_size is None else int(group_size)
    if z is not None and z.shape != x.shape:
        raise RuntimeError(f"rmsnorm: z {tuple(z.shape)} must have the shape of x {tuple(x.shape)}")
    if tuple(weight.shape) != (dim,) or (bias is not None and tuple(bias.shape) != (dim,)):
        raise RuntimeError(f"rmsnorm: weight / bias must be ({dim},)")
    if group_size < 1 or dim % group_size:
        raise RuntimeError(f"rmsnorm: group_size {group_size} does not divide the last dimension {dim}")
    return RmsNormGatedFn.apply(x, z, weight, bias, eps, group_size, bool(norm_before_gate), out_dtype)


def rmsnorm_fn(x, weight, bias, z=None, eps=1e-6, group_size=None, norm_before_gate=True):
    """mamba_ssm.ops.triton.layernorm_gated.rmsnorm_fn (mamba_ssm 2.2.2): the gated, grouped RMSNorm of rms_norm_ref; out in
    x's dtype."""
    return _rmsnorm(x, z, weight, bias, eps, group_size, norm_before_gate, x.dtype)


class RMSNormGated(torch.nn.Module):
    """Mirror of mamba_ssm's gated RMSNorm module (layernorm_gated.RMSNorm): rmsnorm_fn with this module's weight, group_size
    (None: one group of hidden_size) and norm_before_gate; z may be None."""

    def __init__(self, hidden_size, eps=1e-5, group_size=None, norm_before_gate=False, device=None, dtype=None):
        super().__init__()
        if group_size is not None and (group_size < 1 or hidden_size % group_size):
            raise ValueError(f"RMSNormGated: group_size {group_size} does not divide hidden_size {hidden_size}")
        self.eps = eps
        self.weight = torch.nn.Parameter(torch.ones(hidden_size, device=device, dtype=dtype))
        self.register_parameter("bias", None)
        self.group_size = group_size
        self.norm_before_gate = norm_before_gate

    def forward(self, x, z=None, out_dtype=None):
        """out_dtype (default x.dtype, mamba_ssm's contract) lets a caller ask for what its next Linear casts to under autocast."""
        return _rmsnorm(x, z, self.weight, self.bias, self.eps, self.group_size, self.norm_before_gate,
                        x.dtype if out_dtype is None else out_dtype)


# ------------------------------------------------------------------------------------------------
# the fused Mamba-2 mixer (mamba_ssm.ops.triton.ssd_combined.mamba_split_conv1d_scan_combined, mamba_ssm 2.2.2):
# csrc/conv1d.cu -> csrc/ssd.cu -> csrc/rmsnorm.cu -> out_proj, one autograd node that recomputes the conv in its backward
# ------------------------------------------------------------------------------------------------
def _silu_grad(z):
    s = torch.sigmoid(z)
    return s * (1 + z * (1 - s))


class SplitConv1dScanFn(torch.autograd.Function):
    """Saves zxbcdt, the SSD output y, the SSD workspace, the RMSNorm rstd, seq_idx, final_states (when returned) and the
    parameters; no (batch, L, .) activation besides zxbcdt and y.  The backward re-runs the conv forward (and the RMSNorm forward
    when out_proj needs its input) and writes every slice of one dzxbcdt."""

    @staticmethod
    @_no_autocast
    def forward(ctx, zxbcdt, conv_w, conv_b, dt_bias, A, D, initial_states, rms_w, outproj_w, outproj_b, seq_idx, cfg):
        dims, chunk_size, dt_limit, silu, eps, nbg, return_final_states, prec, lin_dtype = cfg
        d_nonssm, H, P, G, N = dims
        batch, L, _ = zxbcdt.shape
        dim, dev = H * P, zxbcdt.device
        z0, x0, z, xBC, dt = zxbcdt.split([d_nonssm, d_nonssm, dim, dim + 2 * G * N, H], dim=-1)
        w32, b32 = _lib.f32c(conv_w), _lib.f32c(conv_b)
        xbc = conv_fwd(xBC, w32, b32, seq_idx, silu, torch.empty(xBC.shape, dtype=zxbcdt.dtype, device=dev))
        x, Bm, Cm = _xbc_views(xbc, H, P, G, N)
        A32, bias32, init32 = _lib.f32c(A), _lib.f32c(dt_bias), _lib.f32c(initial_states)
        D32 = _lib.f32c(D) if D is not None and D.dim() == 1 else None
        y = torch.empty((batch, L, H, P), dtype=zxbcdt.dtype, device=dev)
        fin = torch.empty((batch, H, P, N), dtype=torch.float32, device=dev) if return_final_states else None
        ws, _ = _ssd_fwd(x, dt, A32, Bm, Cm, D32, bias32, init32, seq_idx, chunk_size, True, dt_limit, prec, y, fin)
        # D with a head dimension: plain PyTorch on the side, as in mamba_chunk_scan_combined.  y stays the kernel's output (its
        # backward derives the dt gradients from it); the norm reads y + x D, recomputed in the backward
        Dhp = D.detach() if D is not None and D.dim() == 2 else None
        yn = _add_dx(y, x, Dhp)
        del xbc, x, Bm, Cm
        rw32 = _lib.f32c(rms_w)
        out, rstd = _norm_gate(yn, z, rw32, eps, dim // G, nbg)
        del yn
        if d_nonssm:
            out = torch.cat([F.silu(z0) * x0, out], -1)
        if outproj_w is not None:
            out = F.linear(out.to(lin_dtype), outproj_w.detach().to(lin_dtype),
                           None if outproj_b is None else outproj_b.detach().to(lin_dtype))
        ctx.save_for_backward(zxbcdt, w32, b32, A32, bias32, init32, D32, Dhp, rw32, outproj_w, outproj_b, seq_idx, y, ws, rstd,
                              fin)
        ctx.cfg = cfg
        ctx.dtypes = tuple(None if t is None else t.dtype for t in (conv_w, conv_b, dt_bias, A, D, initial_states, rms_w))
        ctx.set_materialize_grads(False)
        return (out, fin) if return_final_states else out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout, *dextra):
        zxbcdt, w32, b32, A32, bias32, init32, D32, Dhp, rw32, outproj_w, outproj_b, seq_idx, y, ws, rstd, fin = ctx.saved_tensors
        dims, chunk_size, dt_limit, silu, eps, nbg, return_final_states, prec, lin_dtype = ctx.cfg
        d_nonssm, H, P, G, N = dims
        batch, L, _ = zxbcdt.shape
        dim, gn, dev = H * P, G * N, zxbcdt.device
        dfin = _lib.f32c(dextra[0]) if return_final_states and dextra[0] is not None else None
        z0, x0, z, xBC, dt = zxbcdt.split([d_nonssm, d_nonssm, dim, dim + 2 * gn, H], dim=-1)
        dz_all = torch.empty_like(zxbcdt)
        dz0, dx0, dz, dxBC, ddt_slice = dz_all.split([d_nonssm, d_nonssm, dim, dim + 2 * gn, H], dim=-1)
        d_ow = d_ob = d_rw = None
        if dout is None:
            dout = torch.zeros((batch, L, outproj_w.shape[0] if outproj_w is not None else d_nonssm + dim), dtype=y.dtype, device=dev)
        # the conv output again (for the SSD backward, and for y + x D)
        xbc = conv_fwd(xBC, w32, b32, seq_idx, silu, torch.empty(xBC.shape, dtype=zxbcdt.dtype, device=dev))
        x, Bm, Cm = _xbc_views(xbc, H, P, G, N)
        yn = _add_dx(y, x, Dhp)
        if outproj_w is not None:      # its input, recomputed: RMSNorm forward (kernel) and the SwiGLU branch
            normed, _ = _norm_gate(yn, z, rw32, eps, dim // G, nbg)
            if d_nonssm:
                normed = torch.cat([F.silu(z0) * x0, normed], -1)
            g2 = dout.to(lin_dtype).flatten(0, 1)
            d_ow = (g2.t() @ normed.to(lin_dtype).flatten(0, 1)).to(outproj_w.dtype)
            d_ob = None if outproj_b is None else g2.float().sum(0).to(outproj_b.dtype)
            dout = (g2 @ outproj_w.to(lin_dtype)).view(batch, L, -1)
            del normed
        if d_nonssm:
            d_sw, dout = dout[..., :d_nonssm].float(), dout[..., d_nonssm:]
            z0f, x0f = z0.float(), x0.float()
            dz0.copy_(d_sw * x0f * _silu_grad(z0f))
            dx0.copy_(d_sw * F.silu(z0f))
        if rw32 is not None:
            g_, gs_ = _rows_io(dout, dim)
            z_, zs = _rows_io(z, dim)
            dy, dzn, dwb = _rmsnorm_launch_bwd(g_, gs_, yn.view(-1, dim), dim, z_, zs, rw32, None, rstd, batch * L, dim, dim // G, nbg)
            dz.copy_(dzn.view(batch, L, dim))
            d_rw = dwb[0]
        else:
            g, zf = dout.float(), z.float()
            dz.copy_(g * yn.view(batch, L, dim).float() * _silu_grad(zf))
            dy = (g * F.silu(zf)).to(y.dtype)
        dy = dy.reshape(batch, L, H, P)
        del yn
        # the SSD backward into one fp32 (batch, L, conv_dim) buffer that the conv backward reads
        gbuf = torch.empty(xBC.shape, dtype=torch.float32, device=dev)
        gx, gB, gC = _xbc_views(gbuf, H, P, G, N)
        ddt = ddt_slice if zxbcdt.dtype == torch.float32 else torch.empty((batch, L, H), dtype=torch.float32, device=dev)
        dinit = torch.empty_like(init32) if ctx.needs_input_grad[6] else None
        dA, dD, dbias = _ssd_bwd(x, dt, A32, Bm, Cm, D32, bias32, init32, seq_idx, y, ws, fin, (chunk_size, True, dt_limit, prec), dy,
                                 dfin, gx, ddt, gB, gC, dinit)
        if ddt is not ddt_slice:
            ddt_slice.copy_(ddt)
        if Dhp is not None:
            dyf = dy.float()
            gx.add_(dyf * Dhp.float())
            dD = (dyf * x.float()).sum((0, 1))
        del xbc, x, Bm, Cm
        dw, db = conv_bwd(gbuf, xBC, w32, b32, seq_idx, silu, dxBC)
        t_w, t_b, t_bias, t_A, t_D, t_init, t_rw = ctx.dtypes
        cast = lambda t, dt_: None if t is None or dt_ is None else t.to(dt_)
        return (dz_all, cast(dw, t_w), cast(db, t_b), cast(dbias, t_bias), dA.to(t_A), cast(dD, t_D), cast(dinit, t_init),
                cast(d_rw, t_rw), d_ow, d_ob, None, None)


def _add_dx(y, x, Dhp):
    """y + x * D for D (H, P), in y's dtype; y itself when there is no such D."""
    return y if Dhp is None else (y.float() + x.float() * Dhp.float()).to(y.dtype)


def _xbc_views(t, H, P, G, N):
    """x (b, l, H, P), B and C (b, l, G, N): views of the columns of a (b, l, H P + 2 G N) tensor."""
    dim = H * P
    return (t[..., :dim].unflatten(-1, (H, P)), t[..., dim:dim + G * N].unflatten(-1, (G, N)),
            t[..., dim + G * N:].unflatten(-1, (G, N)))


def _norm_gate(y, z, rw32, eps, group_size, nbg):
    """(out, rstd): the grouped gated RMSNorm of y (b, l, H, P) with z read in place (kernel), or y * silu(z) without a weight."""
    batch, L, H, P = y.shape
    y2 = y.view(batch, L, H * P)
    if rw32 is None:
        return y2 * F.silu(z), None
    rows, dim = batch * L, H * P
    y_, ys = _rows_io(y2, dim)
    z_, zs = _rows_io(z, dim)
    out, rstd = _rmsnorm_launch_fwd(y_, ys, z_, zs, rw32, None, rows, dim, eps, group_size, nbg, y.dtype)
    return out.view(batch, L, dim), rstd


def mamba_split_conv1d_scan_combined(zxbcdt, conv1d_weight, conv1d_bias, dt_bias, A, D, chunk_size, initial_states=None, seq_idx=None,
                                     dt_limit=(0.0, float("inf")), return_final_states=False, activation="silu", rmsnorm_weight=None,
                                     rmsnorm_eps=1e-6, outproj_weight=None, outproj_bias=None, headdim=None, ngroups=1,
                                     norm_before_gate=True):
    """Argument:
        zxbcdt: (batch, seqlen, 2 * d_nonssm + 2 * dim + 2 * ngroups * dstate + nheads), split into [z0, x0, z, xBC, dt]
        conv1d_weight: (dim + 2 * ngroups * dstate, width)   conv1d_bias: (dim + 2 * ngroups * dstate,) or None
        dt_bias: (nheads,)   A: (nheads)   D: (nheads, headdim) or (nheads,) with headdim given
        initial_states: (batch, nheads, headdim, dstate)   seq_idx: (batch, seqlen) integers, non-decreasing along seqlen
        rmsnorm_weight: (dim,) or None   outproj_weight: (dim_out, d_nonssm + dim) or None   outproj_bias: (dim_out,) or None
    Return:
        out: (batch, seqlen, d_nonssm + dim) or (batch, seqlen, dim_out) with out_proj [, final_states (batch, nheads, headdim,
        dstate) fp32]
    act(causal conv1d(xBC)) is split into x, B, C for the SSD (dt_softplus, dt_bias, D, dt_limit); its output y is gated by z
    (y * silu(z), or the grouped gated RMSNorm of group size dim // ngroups), the SwiGLU silu(z0) * x0 is prepended when
    d_nonssm > 0, and out_proj applied (in the autocast dtype under autocast).  Every tensor argument gets a gradient in its
    own dtype; final_states passes one back.  The backward recomputes the conv output instead of keeping it."""
    what = "mamba_split_conv1d_scan_combined"
    _lib.require_cuda(zxbcdt, conv1d_weight, conv1d_bias, dt_bias, A, D, initial_states, seq_idx, rmsnorm_weight, outproj_weight,
                      outproj_bias)
    silu = act_is_silu(activation)
    if zxbcdt.dim() != 3:
        raise RuntimeError(f"{what}: zxbcdt must be (batch, seqlen, channels), got {tuple(zxbcdt.shape)}")
    if D.dim() == 1:
        if headdim is None:
            raise RuntimeError(f"{what}: D of shape (nheads,) needs headdim")
        H, P = D.shape[0], int(headdim)
    elif D.dim() == 2:
        H, P = D.shape
    else:
        raise RuntimeError(f"{what}: D must be (nheads,) or (nheads, headdim), got {tuple(D.shape)}")
    dim, G = H * P, int(ngroups)
    if G < 1 or H % G:
        raise RuntimeError(f"{what}: nheads {H} is not a multiple of ngroups {G}")
    if conv1d_weight.dim() != 2:
        raise RuntimeError(f"{what}: conv1d_weight must be (channels, width), got {tuple(conv1d_weight.shape)}")
    N = (conv1d_weight.shape[0] - dim) // G // 2
    conv_dim = dim + 2 * G * N
    batch, L, width_all = zxbcdt.shape
    d_nonssm = (width_all - 2 * dim - 2 * G * N - H) // 2
    if N < 1 or conv1d_weight.shape[0] != conv_dim or d_nonssm < 0 or 2 * d_nonssm + dim + conv_dim + H != width_all:
        raise RuntimeError(f"{what}: zxbcdt {tuple(zxbcdt.shape)} and conv1d_weight {tuple(conv1d_weight.shape)} do not split into "
                           f"[z0, x0, z, xBC, dt] with nheads {H}, headdim {P}, ngroups {G}")
    check_weight(conv1d_weight, conv1d_bias, conv_dim, what)
    if tuple(A.shape) != (H,) or tuple(dt_bias.shape) != (H,):
        raise RuntimeError(f"{what}: A and dt_bias must be ({H},), got {tuple(A.shape)}, {tuple(dt_bias.shape)}")
    if initial_states is not None and tuple(initial_states.shape) != (batch, H, P, N):
        raise RuntimeError(f"{what}: initial_states must be {(batch, H, P, N)}, got {tuple(initial_states.shape)}")
    if rmsnorm_weight is not None and tuple(rmsnorm_weight.shape) != (dim,):
        raise RuntimeError(f"{what}: rmsnorm_weight must be ({dim},), got {tuple(rmsnorm_weight.shape)}")
    if outproj_weight is None and outproj_bias is not None:
        raise RuntimeError(f"{what}: outproj_bias needs outproj_weight")
    if outproj_weight is not None:
        if outproj_weight.dim() != 2 or outproj_weight.shape[1] != d_nonssm + dim:
            raise RuntimeError(f"{what}: outproj_weight must be (dim_out, {d_nonssm + dim}), got {tuple(outproj_weight.shape)}")
        if outproj_bias is not None and tuple(outproj_bias.shape) != (outproj_weight.shape[0],):
            raise RuntimeError(f"{what}: outproj_bias must be ({outproj_weight.shape[0]},), got {tuple(outproj_bias.shape)}")
    if zxbcdt.stride(-1) != 1:
        zxbcdt = zxbcdt.contiguous()
    _lib.dtype_code(zxbcdt.dtype)
    seq_idx = _index_tensor(seq_idx, "seq_idx", zxbcdt.device, (batch, L), what)
    chunk_size = int(chunk_size)
    if chunk_size < 1:
        raise RuntimeError(f"{what}: chunk_size must be positive, got {chunk_size}")
    chunk_size = min(256, (chunk_size + 31) // 32 * 32)      # as in mamba_chunk_scan_combined
    autocast = torch.is_autocast_enabled()
    lin_dtype = torch.get_autocast_dtype("cuda") if autocast else zxbcdt.dtype
    cfg = ((d_nonssm, H, P, G, N), chunk_size, (float(dt_limit[0]), float(dt_limit[1])), silu, float(rmsnorm_eps),
           bool(norm_before_gate), bool(return_final_states), _effective_precision(), lin_dtype)
    return SplitConv1dScanFn.apply(zxbcdt, conv1d_weight, conv1d_bias, dt_bias, A, D, initial_states, rmsnorm_weight, outproj_weight,
                                   outproj_bias, seq_idx, cfg)
