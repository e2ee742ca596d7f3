"""Mamba-2 SSD chunked scan -- host-side mirror of `mamba_ssm.ops.triton.ssd_combined`
(mamba_ssm==2.2.2, not vendored in the reference; call contract: reference SSD/MedSSD.py:41,361-375):

    mamba_chunk_scan_combined(x, dt, A, B, C, chunk_size, D=None, z=None, dt_bias=None,
                              initial_states=None, seq_idx=None, cu_seqlens=None, dt_softplus=False,
                              dt_limit=(0.0, inf), return_final_states=False, return_varlen_states=False)

x (batch, L, H, P); dt (batch, L, H); A (H); B, C (batch, L, G, N); D (H) or (H, P); z like x;
dt_bias (H); initial_states (batch, H, P, N).  Returns out (batch, L, H, P) in x's dtype
[, final_states (batch, H, P, N) fp32].  Tensors are taken with whatever strides they have (the
reference passes (b, l, .) views of channel-major storage, L stride 1) -- nothing is copied.

The work is done by libb200ssm.so (csrc/ssd.cu, sm_100a tensor-core kernels) through its C ABI
(include/b200_ssm.h: b200_ssd_fwd / b200_ssd_bwd).  There is no CPU path: CPU tensors raise.
`seq_idx` / `cu_seqlens` (variable-length batches) are never passed by the reference models and
raise NotImplementedError.
"""
from __future__ import annotations

import ctypes

import torch

import torch.nn.functional as F

from ._lib import no_autocast as _no_autocast
from . import _lib

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


def _fill_fwd(p, x, dt, A, Bm, Cm, D, dt_bias, chunk_size, dt_softplus, dt_limit, initial_states, precision):
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


def _empty_like_layout(t):
    """fp32 tensor of t's shape with t's strides when t is dense (any dimension order), contiguous otherwise."""
    if _lib.is_dense(t):
        return torch.empty_strided(t.shape, t.stride(), dtype=torch.float32, device=t.device)
    return torch.empty(t.shape, dtype=torch.float32, device=t.device)


class SsdChunkScanFn(torch.autograd.Function):
    @staticmethod
    @_no_autocast
    def forward(ctx, x, dt, A, B, C, D, dt_bias, initial_states, chunk_size, dt_softplus, dt_limit, return_final_states, prec):
        batch, L, H, P = x.shape
        G, N = B.shape[2], B.shape[3]
        dev = x.device
        dt_, B_, C_ = dt.to(x.dtype), B.to(x.dtype), C.to(x.dtype)
        A32, D32, bias32, init32 = _lib.f32c(A), _lib.f32c(D), _lib.f32c(dt_bias), _lib.f32c(initial_states)
        out = torch.empty((batch, L, H, P), dtype=x.dtype, device=dev)
        fin = torch.empty((batch, H, P, N), dtype=torch.float32, device=dev) if return_final_states else None
        nbytes = _lib.load().b200_ssd_workspace_bytes(batch, L, H, P, G, N, chunk_size)
        ws = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
        p = _lib.SsdFwdParams()
        _fill_fwd(p, x, dt_, A32, B_, C_, D32, bias32, chunk_size, dt_softplus, dt_limit, init32, prec)
        p.out_stride[:] = list(out.stride())
        p.out, p.final_states, p.workspace = out.data_ptr(), _lib.ptr(fin), ws.data_ptr()
        prof = _profiler
        with torch.cuda.device(dev):
            tok = prof.begin() if prof is not None else None
            _lib.launch("b200_ssd_fwd", dev, ctypes.byref(p))
            if prof is not None:
                prof.end(tok, "fwd", (batch, L, H, P, G, N, chunk_size, prec))
        ctx.save_for_backward(x, dt_, A32, B_, C_, D32, bias32, init32, out, ws)
        ctx.cfg = (chunk_size, bool(dt_softplus), tuple(dt_limit), prec)
        ctx.dtypes = (dt.dtype, A.dtype, B.dtype, C.dtype, None if D is None else D.dtype,
                      None if dt_bias is None else dt_bias.dtype)
        if return_final_states:
            ctx.mark_non_differentiable(fin)
            return out, fin
        return out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout, *unused):
        x, dt_, A32, B_, C_, D32, bias32, init32, out, ws = ctx.saved_tensors
        chunk_size, dt_softplus, dt_limit, precision = ctx.cfg
        batch, L, H, P = x.shape
        G, N = B_.shape[2], B_.shape[3]
        dev = x.device
        dout = dout.to(x.dtype)
        # every gradient in the layout of its primal (the models pass sequence-contiguous views of channel-major storage,
        # SSD/MedSSD.py:344-347): the cross-scan adjoint then reads them in place -- no strided copy after the kernels
        dx, ddt, dB, dC = (_empty_like_layout(t) for t in (x, dt_, B_, C_))
        dA = torch.zeros(H, dtype=torch.float32, device=dev)
        dD = torch.zeros(H, dtype=torch.float32, device=dev) if D32 is not None else None
        dbias = torch.zeros(H, dtype=torch.float32, device=dev) if bias32 is not None else None
        nbytes = _lib.load().b200_ssd_bwd_scratch_bytes(batch, L, H, P, G, N, chunk_size)
        scratch = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
        q = _lib.SsdBwdParams()
        _fill_fwd(q.f, x, dt_, A32, B_, C_, D32, bias32, chunk_size, dt_softplus, dt_limit, init32, precision)
        q.f.out_stride[:] = list(out.stride())
        q.f.out, q.f.workspace = out.data_ptr(), ws.data_ptr()
        q.dout_stride[:] = list(dout.stride())
        q.dout, q.dx, q.ddt, q.dB, q.dC = dout.data_ptr(), dx.data_ptr(), ddt.data_ptr(), dB.data_ptr(), dC.data_ptr()
        q.dx_stride[:], q.ddt_stride[:] = list(dx.stride()), list(ddt.stride())
        q.dB_stride[:], q.dC_stride[:] = list(dB.stride()), list(dC.stride())
        q.dA, q.dD, q.ddt_bias, q.scratch = dA.data_ptr(), _lib.ptr(dD), _lib.ptr(dbias), scratch.data_ptr()
        prof = _profiler
        with torch.cuda.device(dev):
            tok = prof.begin() if prof is not None else None
            _lib.launch("b200_ssd_bwd", dev, ctypes.byref(q))
            if prof is not None:
                prof.end(tok, "bwd", (batch, L, H, P, G, N, chunk_size, precision))
        t_dt, t_A, t_B, t_C, t_D, t_bias = ctx.dtypes
        return (dx.to(x.dtype), ddt.to(t_dt), dA.to(t_A), dB.to(t_B), dC.to(t_C),
                None if dD is None else dD.to(t_D), None if dbias is None else dbias.to(t_bias),
                None, None, None, None, None, None)


def mamba_chunk_scan_combined(x, dt, A, B, C, chunk_size, D=None, z=None, dt_bias=None, initial_states=None,
                              seq_idx=None, cu_seqlens=None, dt_softplus=False, dt_limit=(0.0, float("inf")),
                              return_final_states=False, return_varlen_states=False):
    """Argument:
        x: (batch, seqlen, nheads, headdim)    dt: (batch, seqlen, nheads)    A: (nheads)
        B, C: (batch, seqlen, ngroups, dstate)  chunk_size: int
        D: (nheads, headdim) or (nheads,)       z: (batch, seqlen, nheads, headdim)
        dt_bias: (nheads,)                      initial_states: (batch, nheads, headdim, dstate)
        dt_softplus: whether to apply softplus to dt
    Return:
        out: (batch, seqlen, nheads, headdim) [, final_states (batch, nheads, headdim, dstate)]
    """
    if seq_idx is not None or cu_seqlens is not None or return_varlen_states:
        raise NotImplementedError("mamba_chunk_scan_combined: seq_idx / cu_seqlens (variable-length batches) are not "
                                  "supported by the B200 kernels (never passed by the reference models)")
    _lib.require_cuda(x, dt, A, B, C, D, z, dt_bias, initial_states)
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
        if initial_states.requires_grad:
            raise NotImplementedError("mamba_chunk_scan_combined: no gradient for initial_states in the B200 kernels")
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
    res = SsdChunkScanFn.apply(x, dt, A, B, C, D_head, dt_bias, initial_states, chunk_size, dt_softplus,
                               (float(dt_limit[0]), float(dt_limit[1])), return_final_states,
                               _effective_precision())   # read here: autocast is off inside the Function
    out, fin = res if return_final_states else (res, None)
    if D is not None and D_head is None:      # D with a head dimension: plain PyTorch on the side (unused by the models)
        out = out + x * D.to(x.dtype)
    if z is not None:                         # out * silu(z), as mamba_ssm does when no norm is fused
        out = out * F.silu(z)
    return (out, fin) if return_final_states else out


# ------------------------------------------------------------------------------------------------
# gated RMSNorm (mamba_ssm.ops.triton.layernorm_gated.RMSNorm / rmsnorm_fn, mamba_ssm 2.2.2, as used at
# SSD/MedSSD.py:268-269,393-394): csrc/rmsnorm.cu through b200_rmsnorm_fwd / _bwd
# ------------------------------------------------------------------------------------------------
_IO_DTYPES = (torch.float32, torch.bfloat16, torch.float16)


def _rows_io(t, dim):
    """(tensor, row stride) of t as the kernels read it: in place when its dtype is one they read and its rows are contiguous."""
    return _lib.rows_view(t if t.dtype in _IO_DTYPES else t.float(), dim)


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
        out = torch.empty((rows, dim), dtype=out_dtype, device=x.device)
        rstd = torch.empty((rows, dim // group_size), dtype=torch.float32, device=x.device)
        _lib.launch("b200_rmsnorm_fwd", x.device, x2.data_ptr(), _lib.dtype_code(x2.dtype), xs, _lib.ptr(z2),
                    _lib.dtype_code(z2.dtype) if z2 is not None else 0, zs, w32.data_ptr(), _lib.ptr(b32), out.data_ptr(),
                    _lib.dtype_code(out_dtype), rstd.data_ptr(), rows, dim, group_size, int(norm_before_gate), float(eps))
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
        dx = torch.empty((rows, dim), dtype=x2.dtype, device=dev)
        dz = torch.empty((rows, dim), dtype=z2.dtype, device=dev) if z2 is not None else None
        grid = _lib.load().b200_rmsnorm_grid(rows, dim, group_size)
        if grid < 0:
            _lib.check(grid, "b200_rmsnorm_grid")
        part = torch.empty((1 if b32 is None else 2, grid, dim), dtype=torch.float32, device=dev)
        _lib.launch("b200_rmsnorm_bwd", dev, dy2.data_ptr(), _lib.dtype_code(dy2.dtype), dys, x2.data_ptr(), _lib.dtype_code(x2.dtype),
                    xs, _lib.ptr(z2), _lib.dtype_code(z2.dtype) if z2 is not None else 0, zs, w32.data_ptr(), _lib.ptr(b32),
                    rstd.data_ptr(), dx.data_ptr(), _lib.ptr(dz), part[0].data_ptr(), part[1].data_ptr() if b32 is not None else None,
                    rows, dim, group_size, nbg)
        dwb = part.sum(1)
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
