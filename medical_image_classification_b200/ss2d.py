"""SS2D block (Mamba-1 four-direction 2-D selective scan) -- B200 mirror of the reference module
`SS2D` (reference MedMamba.py:253-483): same constructor arguments, same parameter names and shapes
(`in_proj.weight, conv2d.{weight,bias}, x_proj_weight (4,R+2N,D), dt_projs_weight (4,D,R),
dt_projs_bias (4,D), A_logs (4D,N), Ds (4D), out_norm.{weight,bias}, out_proj.weight`), so reference
checkpoints load with strict=True, and the same `forward((B,H,W,C)) -> (B,H,W,C)`.

What differs is how `forward_core` moves data (cross.py / csrc/sscan.cu / csrc/cross.cu): the four
permuted copies of the image, the flips and the four-way un-permute of the reference
(MedMamba.py:393-395, 420-424, 476-477) are replaced by one pack kernel, a scan kernel that walks
two of the directions backwards, and one merge kernel.  The x_proj / dt_proj contractions
(MedMamba.py:397-400) are point-wise in the sequence position, so they run on the un-permuted
[x, x^T] pair as plain batched GEMMs (cuBLAS).
"""
from __future__ import annotations

import math

import torch

import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from ._lib import no_autocast as _no_autocast
from .cross import ss2d_core
from .selective_scan_interface import selective_scan_fn


class SplitHalvesFn(torch.autograd.Function):
    """a, b = t.chunk(2, dim=-1) (MedMamba.py:467 `x, z = xz.chunk(2, dim=-1)`, :530 `left, right = input.chunk(...)`) with a
    one-pass backward: d(input) = cat(d left, d right)
    instead of two zero-filled full-size buffers, two slice copies and an add."""

    @staticmethod
    @_no_autocast
    def forward(ctx, inp):
        c = inp.shape[-1] // 2
        return inp[..., :c], inp[..., c:]

    @staticmethod
    @_no_autocast
    def backward(ctx, dl, dr):
        return torch.cat((dl, dr.to(dl.dtype)), dim=-1)


def split_halves(t):
    """t.chunk(2, dim=-1); with an even last dimension through SplitHalvesFn (one cat in the backward)."""
    if t.shape[-1] % 2 == 0 and t.requires_grad:
        return SplitHalvesFn.apply(t)
    return t.chunk(2, dim=-1)


class LnGateFn(torch.autograd.Function):
    """out = LayerNorm(y) [* silu(z)] in one pass over HBM (csrc/lngate.cu) -- reference MedMamba.py:478-479 (with z)
    and the block pre-norm `ln_1` (MedMamba.py:531, z = None).  y (..., D) fp32 (or bf16 when z is None: the bf16 residual
    stream of an autocast model), z (..., D) fp32 / bf16; both may be strided views with contiguous rows (halves of a
    chunk) and are read in place; returns out_dtype; dy comes back in y's dtype."""

    @staticmethod
    @_no_autocast
    def forward(ctx, y, z, weight, bias, eps, out_dtype):
        _lib.require_cuda(y, z, weight, bias)
        D = y.shape[-1]
        if y.dtype != torch.float32 and not (y.dtype == torch.bfloat16 and z is None):
            y = y.float()
        y2, ys = _lib.rows_view(y, D)
        z2, zs = (None, 0)
        if z is not None:
            if z.dtype not in (torch.float32, torch.bfloat16):
                z = z.float()
            z2, zs = _lib.rows_view(z, D)
        rows = y.numel() // D
        w32, b32 = weight.detach().float().contiguous(), bias.detach().float().contiguous()
        out = torch.empty((rows, D), dtype=out_dtype, device=y.device)
        mean = torch.empty(rows, dtype=torch.float32, device=y.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=y.device)
        zcode = _lib.dtype_code(z2.dtype) if z2 is not None else 0
        _lib.launch("b200_ln_gate_fwd", y.device, y2.data_ptr(), _lib.dtype_code(y2.dtype), ys, _lib.ptr(z2), zs, zcode, w32.data_ptr(),
                    b32.data_ptr(), out.data_ptr(), _lib.dtype_code(out_dtype), mean.data_ptr(), rstd.data_ptr(), rows, D, float(eps))
        ctx.save_for_backward(y2, z2, w32, b32, mean, rstd)
        ctx.ys, ctx.zs, ctx.shape, ctx.zshape, ctx.rows = ys, zs, y.shape, (z.shape if z is not None else None), rows
        ctx.wdtype, ctx.bdtype = weight.dtype, bias.dtype
        return out.view(*y.shape[:-1], D)

    @staticmethod
    @_no_autocast
    def backward(ctx, dout):
        y2, z2, w32, b32, mean, rstd = ctx.saved_tensors
        rows, D = ctx.rows, ctx.shape[-1]
        dout = dout.reshape(rows, D).contiguous()
        dev = dout.device
        dy = torch.empty((rows, D), dtype=y2.dtype, device=dev)
        dz = torch.empty((rows, D), dtype=z2.dtype, device=dev) if z2 is not None else None
        grid = _lib.load().b200_ln_gate_grid(rows)
        part = torch.empty((2, grid, D), dtype=torch.float32, device=dev)
        zcode = _lib.dtype_code(z2.dtype) if z2 is not None else 0
        _lib.launch("b200_ln_gate_bwd", dev, dout.data_ptr(), y2.data_ptr(), _lib.dtype_code(y2.dtype), ctx.ys, _lib.ptr(z2), ctx.zs, zcode,
                    w32.data_ptr(), b32.data_ptr(), _lib.dtype_code(dout.dtype), mean.data_ptr(), rstd.data_ptr(), dy.data_ptr(), _lib.ptr(dz),
                    part[0].data_ptr(), part[1].data_ptr(), rows, D)
        dwb = part.sum(1)
        return (dy.view(ctx.shape), dz.view(ctx.zshape) if dz is not None else None, dwb[0].to(ctx.wdtype), dwb[1].to(ctx.bdtype),
                None, None)


class DwConvSiluFn(torch.autograd.Function):
    """x (B, D, H, W) fp32 = SiLU(depthwise conv3x3(xin) + bias) with xin a channels-last (B, H, W, D) view read in
    place (csrc/dwconv.cu) -- reference MedMamba.py:470-473 + the .float() of :403."""

    @staticmethod
    @_no_autocast
    def forward(ctx, xin, weight, bias):
        _lib.require_cuda(xin, weight, bias)
        B, H, W, D = xin.shape
        ok = xin.stride(3) == 1 and xin.stride(1) == W * xin.stride(2) and xin.stride(0) == H * xin.stride(1)
        if not ok or xin.dtype not in (torch.float32, torch.bfloat16):
            xin = xin.contiguous() if xin.dtype in (torch.float32, torch.bfloat16) else xin.float().contiguous()
        w32 = weight.detach().float().reshape(D, 9).contiguous()
        b32 = bias.detach().float().contiguous() if bias is not None else None
        out = torch.empty((B, D, H, W), dtype=torch.float32, device=xin.device)
        _lib.launch("b200_dwconv_silu_fwd", xin.device, xin.data_ptr(), xin.stride(2), _lib.dtype_code(xin.dtype), w32.data_ptr(),
                    _lib.ptr(b32), out.data_ptr(), B, D, H, W)
        ctx.save_for_backward(xin, w32, b32)
        ctx.wshape, ctx.wdtype = weight.shape, weight.dtype
        ctx.bdtype = bias.dtype if bias is not None else None
        return out

    @staticmethod
    @_no_autocast
    def backward(ctx, g):
        xin, w32, b32 = ctx.saved_tensors
        B, H, W, D = xin.shape
        g = g.float().contiguous()
        dxin = torch.empty((B, H, W, D), dtype=xin.dtype, device=xin.device)
        acc_w = torch.zeros((D * 9 + D,), dtype=torch.float32, device=xin.device)   # weight taps | bias: one memset
        dw_buf, db_buf = acc_w[: D * 9], acc_w[D * 9:]
        _lib.launch("b200_dwconv_silu_bwd", xin.device, g.data_ptr(), xin.data_ptr(), xin.stride(2), _lib.dtype_code(xin.dtype),
                    w32.data_ptr(), _lib.ptr(b32), dxin.data_ptr(), dw_buf.data_ptr(), db_buf.data_ptr(), B, D, H, W)
        dweight = dw_buf.view(ctx.wshape).to(ctx.wdtype)
        dbias = db_buf.to(ctx.bdtype) if ctx.bdtype is not None else None
        return dxin, dweight, dbias


def _autocast_out_dtype():
    return torch.bfloat16 if (torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16) else torch.float32


def ln_gate(y, z, norm: nn.LayerNorm):
    """LayerNorm(y) * silu(z) through libb200ssm (CUDA only); bf16 out under autocast (= what the next Linear casts to)."""
    return LnGateFn.apply(y, z, norm.weight, norm.bias, norm.eps, _autocast_out_dtype())


def layer_norm_rows(y, norm: nn.LayerNorm):
    """Plain LayerNorm over the last dimension of a (possibly strided) fp32 tensor through libb200ssm."""
    return LnGateFn.apply(y, None, norm.weight, norm.bias, norm.eps, _autocast_out_dtype())


class SS2D(nn.Module):
    def __init__(self, d_model, d_state=16, d_conv=3, expand=2, dt_rank="auto", dt_min=0.001, dt_max=0.1,
                 dt_init="random", dt_scale=1.0, dt_init_floor=1e-4, dropout=0.0, conv_bias=True, bias=False,
                 device=None, dtype=None, **kwargs):
        fk = {"device": device, "dtype": dtype}
        super().__init__()
        self.d_model = d_model
        self.d_state = d_state
        self.d_conv = d_conv
        self.expand = expand
        self.d_inner = int(expand * d_model)
        self.dt_rank = math.ceil(d_model / 16) if dt_rank == "auto" else dt_rank
        K, D, N, R = 4, self.d_inner, d_state, self.dt_rank

        self.in_proj = nn.Linear(d_model, 2 * D, bias=bias, **fk)
        self.conv2d = nn.Conv2d(D, D, kernel_size=d_conv, padding=(d_conv - 1) // 2, groups=D, bias=conv_bias, **fk)
        self.act = nn.SiLU()

        # per-direction projections, stacked (MedMamba.py:296-317)
        bound = 1.0 / math.sqrt(D)
        self.x_proj_weight = nn.Parameter(torch.empty(K, R + 2 * N, D, **fk).uniform_(-bound, bound))
        std = R ** -0.5 * dt_scale
        w = torch.empty(K, D, R, **fk)
        if dt_init == "constant":
            w.fill_(std)
        elif dt_init == "random":
            w.uniform_(-std, std)
        else:
            raise NotImplementedError(dt_init)
        self.dt_projs_weight = nn.Parameter(w)
        # bias such that softplus(bias) is log-uniform in [dt_min, dt_max] (MedMamba.py:343-351)
        dt = torch.exp(torch.rand(K, D, **fk) * (math.log(dt_max) - math.log(dt_min)) + math.log(dt_min))
        dt = dt.clamp(min=dt_init_floor)
        self.dt_projs_bias = nn.Parameter(dt + torch.log(-torch.expm1(-dt)))
        self.dt_projs_bias._no_reinit = True

        # S4D-real A = -(1..N) per channel and direction; D = 1 (MedMamba.py:357-384)
        A = torch.arange(1, N + 1, dtype=torch.float32, device=device).repeat(K * D, 1)
        self.A_logs = nn.Parameter(torch.log(A))
        self.A_logs._no_weight_decay = True
        self.Ds = nn.Parameter(torch.ones(K * D, device=device))
        self.Ds._no_weight_decay = True

        self.out_norm = nn.LayerNorm(D)
        self.out_proj = nn.Linear(D, d_model, bias=bias, **fk)
        self.dropout = nn.Dropout(dropout) if dropout > 0.0 else None
        # the fused core keeps 16 states per row in registers; wider state spaces (unused by the reference's models) take the
        # operator-API data flow, where selective_scan_fn runs them as 16-state slices
        self.forward_core = self.forward_core_fused if d_state <= 16 else self.forward_core_api

    # ---- the hot path --------------------------------------------------------------------------
    @staticmethod
    def _to_internal(w):
        """Re-order a per-direction tensor (4, ...) from the reference order k = layout + 2*reverse
        to the internal order 2*layout + reverse (cross.DIR_PERM) without an index tensor, so the
        step stays CUDA-graph capturable."""
        return w.view(2, 2, *w.shape[1:]).transpose(0, 1).reshape(w.shape)

    def _dir_params(self):
        """Per-direction parameters in the internal direction order."""
        K, D, N = 4, self.d_inner, self.d_state
        Wx = self._to_internal(self.x_proj_weight.float())                         # (4, R+2N, D)
        Wdt = self._to_internal(self.dt_projs_weight.float())                      # (4, D, R)
        bias = self._to_internal(self.dt_projs_bias.float()).reshape(-1)           # (4D)
        As = self._to_internal(-torch.exp(self.A_logs.float()).view(K, D, N)).reshape(K * D, N)
        Ds = self._to_internal(self.Ds.float().view(K, D)).reshape(-1)
        return Wx, Wdt, bias, As, Ds

    def forward_core_fused(self, x: torch.Tensor):
        """x (B, D, H, W) -> merged y (B, H, W, D) fp32 == y1+y2+y3+y4 of the reference's
        forward_corev0 (MedMamba.py:386-424) already transposed to channels-last (:476-477)."""
        B, D, H, W = x.shape
        L = H * W
        R, N = self.dt_rank, self.d_state
        tf32 = torch.is_autocast_enabled()   # the reference computes these projections in bf16 under autocast
        with torch.autocast("cuda", enabled=False):
            Wx, Wdt, bias, As, Ds = self._dir_params()
            # one projection matrix per direction: rows of B, rows of C, and the rank-R dt projection folded through
            # x_proj's dt rows (delta = Wdt (Wx_dt x) = (Wdt Wx_dt) x), so B, C and delta come out of ONE GEMM
            W_all = torch.cat([Wx[:, R:], torch.matmul(Wdt, Wx[:, :R])], dim=1)              # (4, 2N + D, D)
            y = ss2d_core(x, W_all, As, Ds, bias, N, tf32)                                    # (B, L, D)
        return y.view(B, H, W, D)

    def forward_core_api(self, x: torch.Tensor):
        """The reference's data flow verbatim (four materialised directions, operator-API call,
        flips and transposes), kept for parity tests of `selective_scan_fn` inside the module."""
        B, D, H, W = x.shape
        L = H * W
        K = 4
        x_hwwh = torch.stack([x.view(B, -1, L), x.transpose(2, 3).contiguous().view(B, -1, L)], dim=1)
        xs = torch.cat([x_hwwh, x_hwwh.flip(-1)], dim=1)
        x_dbl = torch.einsum("bkdl,kcd->bkcl", xs, self.x_proj_weight)
        dts, Bs, Cs = torch.split(x_dbl, [self.dt_rank, self.d_state, self.d_state], dim=2)
        dts = torch.einsum("bkrl,kdr->bkdl", dts, self.dt_projs_weight)
        out_y = selective_scan_fn(
            xs.float().view(B, -1, L), dts.contiguous().float().view(B, -1, L),
            -torch.exp(self.A_logs.float()), Bs.float(), Cs.float(), self.Ds.float(), z=None,
            delta_bias=self.dt_projs_bias.float().view(-1), delta_softplus=True).view(B, K, -1, L)
        inv_y = out_y[:, 2:4].flip(-1)
        wh_y = out_y[:, 1].view(B, -1, W, H).transpose(2, 3).contiguous().view(B, -1, L)
        invwh_y = inv_y[:, 1].view(B, -1, W, H).transpose(2, 3).contiguous().view(B, -1, L)
        y = out_y[:, 0] + inv_y[:, 0] + wh_y + invwh_y
        return y.transpose(1, 2).contiguous().view(B, H, W, -1)

    def forward(self, x: torch.Tensor, **kwargs):
        B, H, W, C = x.shape
        xz = self.in_proj(x)
        x, z = split_halves(xz)
        _lib.require_cuda(x)                                        # no CPU path: oracle/cpu_path.py holds the eager CPU tree
        if (self.d_conv == 3 and W <= 64 and x.dtype in (torch.float32, torch.bfloat16)
                and self.forward_core == self.forward_core_fused):
            x = DwConvSiluFn.apply(x, self.conv2d.weight, self.conv2d.bias)   # conv3x3 + SiLU, channels-last in -> fp32 planes out
        else:   # shapes outside the kernel's envelope / the API-path parity tests: the reference's two library ops
            x = x.permute(0, 3, 1, 2).contiguous()
            x = self.act(self.conv2d(x))
        y = self.forward_core(x)                                    # (B, H, W, D) fp32
        assert y.dtype == torch.float32
        if self.d_inner <= 1024 and z.dtype in (torch.float32, torch.bfloat16):
            y = ln_gate(y, z, self.out_norm)                        # out_norm + silu(z) gate, one pass (csrc/lngate.cu)
        else:   # wider than the row kernel holds in registers: the reference's two library ops
            y = self.out_norm(y)
            y = y * F.silu(z)
        out = self.out_proj(y)
        if self.dropout is not None:
            out = self.dropout(out)
        return out
