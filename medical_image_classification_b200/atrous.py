"""EfficientVMamba-style atrous ("skip") scan for the FusionMamba blocks -- host-side mirror of
CrossMamba/FusionMamba/models/cross.py:34-262 (`EfficientMerge`, `SelectiveScan`, `EfficientScan`,
`cross_selective_scan_new`) on libb200ssm (SURVEY.md section 8(f) rank 4).

The four "directions" of this scan are the four sub-lattices of the image (row parity x column parity), two flattened
row-major and two column-major; each is a quarter-length sequence for the ordinary selective scan.  The reference builds them
with strided slices + transposes + four copies (and the inverse with four strided assignments); here each way is one kernel
(csrc/cross.cu::atrous_scan_kernel / atrous_merge_kernel), and since the two maps are each other's adjoint the backward of one
is the forward of the other.  step_size 2 only (the reference's default and only use; with larger steps the reference's merge
leaves the other residues uninitialised)."""
from __future__ import annotations

import math

import torch


from ._lib import no_autocast as _no_autocast
from . import _lib
from .selective_scan_interface import selective_scan_fn


def _check_step(step_size):
    if step_size != 2:
        raise RuntimeError(f"atrous scan: step_size {step_size} is not supported by the B200 kernels (the reference uses 2)")


class EfficientScan(torch.autograd.Function):
    """x (B, C, H, W) -> xs (B, 4, C, ceil(H/2) * ceil(W/2)) -- reference models/cross.py:139-190."""

    @staticmethod
    @_no_autocast
    def forward(ctx, x, step_size=2):
        _check_step(step_size)
        _lib.require_cuda(x)
        x = x.contiguous()
        B, C, H, W = x.shape
        L2 = math.ceil(H / 2) * math.ceil(W / 2)
        xs = torch.empty((B, 4, C, L2), dtype=x.dtype, device=x.device)
        _lib.launch("b200_atrous_scan", x.device, x.data_ptr(), xs.data_ptr(), B, C, H, W, _lib.dtype_code(x.dtype))
        ctx.shape = (B, C, H, W)
        return xs

    @staticmethod
    @_no_autocast
    def backward(ctx, grad_xs):
        B, C, H, W = ctx.shape
        grad_xs = grad_xs.contiguous()
        gx = torch.empty((B, C, H, W), dtype=grad_xs.dtype, device=grad_xs.device)
        _lib.launch("b200_atrous_merge", grad_xs.device, grad_xs.data_ptr(), gx.data_ptr(), B, C, H, W, _lib.dtype_code(grad_xs.dtype))
        return gx, None


class EfficientMerge(torch.autograd.Function):
    """ys (B, 4, C, ceil(H/2) * ceil(W/2)) -> y (B, C, H * W) -- reference models/cross.py:34-92."""

    @staticmethod
    @_no_autocast
    def forward(ctx, ys, ori_h, ori_w, step_size=2):
        _check_step(step_size)
        _lib.require_cuda(ys)
        ys = ys.contiguous()
        B, K, C, L2 = ys.shape
        H, W = int(ori_h), int(ori_w)
        if K != 4 or L2 != math.ceil(H / 2) * math.ceil(W / 2):
            raise RuntimeError(f"EfficientMerge: ys {tuple(ys.shape)} does not match a {H} x {W} image")
        y = torch.empty((B, C, H, W), dtype=ys.dtype, device=ys.device)
        _lib.launch("b200_atrous_merge", ys.device, ys.data_ptr(), y.data_ptr(), B, C, H, W, _lib.dtype_code(ys.dtype))
        ctx.shape = (B, C, H, W)
        return y.view(B, C, H * W)

    @staticmethod
    @_no_autocast
    def backward(ctx, grad_y):
        B, C, H, W = ctx.shape
        grad_y = grad_y.contiguous()
        L2 = math.ceil(H / 2) * math.ceil(W / 2)
        gys = torch.empty((B, 4, C, L2), dtype=grad_y.dtype, device=grad_y.device)
        _lib.launch("b200_atrous_scan", grad_y.device, grad_y.data_ptr(), gys.data_ptr(), B, C, H, W, _lib.dtype_code(grad_y.dtype))
        return gys, None, None, None


class SelectiveScan:
    """`SelectiveScan.apply(u, delta, A, B, C, D, delta_bias, delta_softplus, nrows)` of models/cross.py:94-137: the plain
    operator in fp32 (`custom_fwd(cast_inputs=torch.float32)`); `nrows` was a tiling knob of the reference's kernel build."""

    @staticmethod
    def apply(u, delta, A, B, C, D=None, delta_bias=None, delta_softplus=False, nrows=1):
        f = lambda t: None if t is None else t.float()
        with torch.autocast("cuda", enabled=False):
            return selective_scan_fn(f(u), f(delta), f(A), f(B), f(C), f(D), None, f(delta_bias), delta_softplus)


def cross_selective_scan_new(x, x_proj_weight, x_proj_bias, dt_projs_weight, dt_projs_bias, A_logs, Ds, out_norm=None, nrows=-1,
                             delta_softplus=True, to_dtype=True, step_size=2):
    """Mirror of models/cross.py:193-262: atrous scan -> x_proj / dt_proj -> four quarter-length selective scans -> atrous merge
    -> out_norm.  x (B, D, H, W) -> (B, H, W, D)."""
    B, D, H, W = x.shape
    N = A_logs.shape[1]
    K, _, R = dt_projs_weight.shape
    xs = EfficientScan.apply(x, step_size)
    L = xs.shape[-1]
    x_dbl = torch.einsum("b k d l, k c d -> b k c l", xs, x_proj_weight)
    if x_proj_bias is not None:
        x_dbl = x_dbl + x_proj_bias.view(1, K, -1, 1)
    dts, Bs, Cs = torch.split(x_dbl, [R, N, N], dim=2)
    dts = torch.einsum("b k r l, k d r -> b k d l", dts, dt_projs_weight)
    ys = SelectiveScan.apply(xs.reshape(B, -1, L), dts.reshape(B, -1, L), -torch.exp(A_logs.float()), Bs, Cs, Ds.float(),
                             dt_projs_bias.reshape(-1), delta_softplus, nrows).view(B, K, -1, L)
    y = EfficientMerge.apply(ys, H, W, step_size)                     # (B, D, H*W)
    y = y.transpose(1, 2).contiguous()
    if out_norm is not None:
        y = out_norm(y)
    y = y.view(B, H, W, -1)
    return y.to(x.dtype) if to_dtype else y
