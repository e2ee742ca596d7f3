"""SS2D cross-scan / selective scan / cross-merge as autograd Functions over libb200ssm.

Reference semantics (MedMamba.py:386-424, 476-477): four orderings of every channel plane --
k=0 row-major, k=1 column-major, k=2/3 their time reversals -- are scanned independently and the
four outputs are un-permuted and summed into (B, H, W, D).

B200 layout: directions are kept in the order  hw, hw-reversed, wh, wh-reversed  (`DIR_PERM` maps
this internal index to the reference's k), because then
  * the two reversed directions need no data at all (the kernel scans backwards, rev_mask=0b1010),
  * directions (0,1) and (2,3) read the same image (u_group_div=2) and receive the same upstream
    gradient (dout_group_div=2),
so cross-scan is one pack kernel (x -> [x, x^T]) and cross-merge is one kernel.
"""
from __future__ import annotations

import torch


from ._lib import no_autocast as _no_autocast
from . import _lib
from .selective_scan_interface import launch_bwd, launch_fwd

DIR_PERM = (0, 2, 1, 3)   # internal direction -> reference direction k (self-inverse)
REV_MASK = 0b1010         # internal directions 1 and 3 run backwards in time


class CrossScanPackFn(torch.autograd.Function):
    """x (B, D, H, W) -> x2 (B, 2, D, L): x2[:,0] row-major image, x2[:,1] column-major image."""

    @staticmethod
    @_no_autocast
    def forward(ctx, x):
        _lib.require_cuda(x)
        x = x.contiguous()
        B, D, H, W = x.shape
        x2 = torch.empty((B, 2, D, H * W), dtype=x.dtype, device=x.device)
        _lib.launch("b200_cross_scan_pack", x.device, x.data_ptr(), x2.data_ptr(), B, D, H, W, _lib.dtype_code(x.dtype))
        ctx.hw = (H, W)
        return x2

    @staticmethod
    @_no_autocast
    def backward(ctx, dx2):
        H, W = ctx.hw
        dx2 = dx2.contiguous()
        B, _, D, _ = dx2.shape
        dx = torch.empty((B, D, H, W), dtype=dx2.dtype, device=dx2.device)
        _lib.launch("b200_cross_scan_pack_bwd", dx2.device, dx2.data_ptr(), dx.data_ptr(), B, D, H, W, _lib.dtype_code(dx2.dtype))
        return dx


class CrossMergeFn(torch.autograd.Function):
    """ys (B, 4, D, L) at memory positions (internal direction order) -> y (B, L, D)."""

    @staticmethod
    @_no_autocast
    def forward(ctx, ys, H, W):
        _lib.require_cuda(ys)
        ys = ys.contiguous()
        B, K, D, L = ys.shape
        assert K == 4 and L == H * W
        y = torch.empty((B, L, D), dtype=ys.dtype, device=ys.device)
        _lib.launch("b200_cross_merge", ys.device, ys.data_ptr(), y.data_ptr(), B, D, H, W, _lib.dtype_code(ys.dtype))
        ctx.hw = (H, W)
        return y

    @staticmethod
    @_no_autocast
    def backward(ctx, dy):
        H, W = ctx.hw
        dy = dy.contiguous()
        B, L, D = dy.shape
        d2 = torch.empty((B, 2, D, L), dtype=dy.dtype, device=dy.device)
        _lib.launch("b200_cross_merge_bwd", dy.device, dy.data_ptr(), d2.data_ptr(), B, D, H, W, _lib.dtype_code(dy.dtype))
        dys = d2.unsqueeze(2).expand(B, 2, 2, D, L).reshape(B, 4, D, L)
        return dys, None, None


class _Tf32:
    """torch.backends.cuda.matmul.allow_tf32 for the duration of a with-block."""

    def __init__(self, on):
        self.on = bool(on)

    def __enter__(self):
        self.prev = torch.backends.cuda.matmul.allow_tf32
        if self.on:
            torch.backends.cuda.matmul.allow_tf32 = True

    def __exit__(self, *exc):
        torch.backends.cuda.matmul.allow_tf32 = self.prev


def _weight_grad_splitk(g_big, x2m):
    """dW (2, 2M, D) = g_big (2, 2M, B*L) @ x2m (2, D, B*L)^T.  The output is a handful of tiles while K = B*L is ~200 K, so
    K is split across the batch dimension of a strided bmm (views only, no copies) and the partials are summed."""
    _, M2, BL = g_big.shape
    D = x2m.shape[1]
    tiles = 2 * ((M2 + 127) // 128) * ((D + 63) // 64)
    S = 1
    while tiles * S < 592 and BL % (2 * S) == 0 and BL // (2 * S) >= 448:
        S *= 2
    if S == 1:
        return torch.bmm(g_big, x2m.transpose(1, 2))
    Kp = BL // S
    parts = []
    for i in range(2):
        a = g_big[i].view(M2, S, Kp).permute(1, 0, 2)                  # (S, 2M, K')
        b = x2m[i].view(D, S, Kp).permute(1, 2, 0)                     # (S, K', D)
        parts.append(torch.bmm(a, b).sum(0))
    return torch.stack(parts)


class SS2DCoreFn(torch.autograd.Function):
    """The whole SS2D core -- cross-scan, x_proj / dt_proj, four-direction selective scan, cross-merge (reference
    MedMamba.py:386-424, 476-477) -- as ONE autograd node, so that every intermediate lives in a layout of our choosing:

      x (B, D, H, W) fp32 --pack--> x2 (2, D, B, L)                          [row-major planes | column-major planes]
      big (2, 2M, B*L) = W_all (2, 2M, D) @ x2 (2, D, B*L)                   ONE batched GEMM with B*L columns
         W_all[k] (M = 2N + D rows) = [x_proj rows of B ; of C ; dt_proj_weight @ x_proj rows of dt]   (internal direction
         order; the rank-R dt projection is folded into the same GEMM, so `delta` comes out of it directly)
      scan reads B, C, delta as strided views of `big`, u as a view of x2   (b200_sscan_* take arbitrary leading strides)
      y (B, L, D) = cross-merge of the four direction outputs.

    Backward: the scan kernel writes ddelta and accumulates dB, dC straight into `g_big` (the layout of `big`), so
    dW_all = g_big @ x2^T and gx2 = W_all^T @ g_big are two GEMMs over K resp. N = B*L with no per-sample partials, no
    slice / cat / add kernels; dx = b200_cross_scan_unpack4(du, gx2) finishes the adjoint of the cross-scan in one pass.
    tf32: run the three GEMMs in TF32 (used under autocast, where the reference runs these einsums in bf16)."""

    @staticmethod
    @_no_autocast
    def forward(ctx, x, W_all, A, Ds, delta_bias, N, tf32):
        _lib.require_cuda(x, W_all, A, Ds, delta_bias)
        x = x.float().contiguous()
        B, D, H, W = x.shape
        L = H * W
        M = W_all.shape[1]
        assert W_all.shape == (4, M, D) and M == 2 * N + D
        dev = x.device
        # Rows are laid out with a pitch Lp = L rounded up to 4 elements, so that every row of x2 / big starts on a 16-byte
        # boundary and the TMA-staged scan kernels (csrc/sscan2.cu) apply at L = 49 too (stage 3: 7 x 7).  The pad columns of x2
        # are zero, hence delta = B = C = u = 0 there: a pad step leaves the (zero) state and every gradient untouched whichever
        # direction meets it first, so the scan simply runs over Lp steps.
        Lp = (L + 3) // 4 * 4
        x2 = torch.empty((2, D, B, Lp), dtype=torch.float32, device=dev) if Lp == L else torch.zeros((2, D, B, Lp), dtype=torch.float32, device=dev)
        strides = (Lp, D * B * Lp, B * Lp)                            # (batch, layout, row) element strides of x2
        _lib.launch("b200_cross_scan_pack_strided", dev, x.data_ptr(), x2.data_ptr(), *strides, B, D, H, W)
        Wm = W_all.detach().float().reshape(2, 2 * M, D).contiguous()
        with _Tf32(tf32):
            big = torch.bmm(Wm, x2.view(2, D, B * Lp))                 # (2, 2M, B*Lp)
        big4 = big.view(4, M, B, Lp).permute(2, 0, 1, 3)               # (B, 4, M, Lp) view
        A32, D32, b32 = _lib.f32c(A), _lib.f32c(Ds), _lib.f32c(delta_bias)
        need_grad = any(ctx.needs_input_grad)
        ys, _, ckpt = launch_fwd(x2.permute(2, 0, 1, 3), big4[:, :, 2 * N:], A32, big4[:, :, :N], big4[:, :, N:2 * N], D32, None, b32,
                                 True, REV_MASK, 2, want_ckpt=need_grad, algo_len=L)
        if Lp != L:
            ys = ys[:, :, :L].contiguous()
        y = torch.empty((B, L, D), dtype=torch.float32, device=dev)
        _lib.launch("b200_cross_merge", dev, ys.data_ptr(), y.data_ptr(), B, D, H, W, _lib.dtype_code(ys.dtype))
        if need_grad:
            ctx.save_for_backward(x2, big, Wm, A32, D32, b32, ckpt)
        ctx.meta = (B, D, H, W, M, N, bool(tf32))
        ctx.dtypes = (W_all.dtype, A.dtype, Ds.dtype, delta_bias.dtype)
        return y

    @staticmethod
    @_no_autocast
    def backward(ctx, dy):
        x2, big, Wm, A32, D32, b32, ckpt = ctx.saved_tensors
        B, D, H, W, M, N, tf32 = ctx.meta
        L = H * W
        Lp = x2.shape[-1]
        dev = dy.device
        dy = dy.contiguous().float()
        d2 = torch.empty((B, 2 * D, L), dtype=torch.float32, device=dev)
        _lib.launch("b200_cross_merge_bwd", dev, dy.data_ptr(), d2.data_ptr(), B, D, H, W, _lib.dtype_code(dy.dtype))
        if Lp != L:
            d2 = torch.nn.functional.pad(d2, (0, Lp - L))              # zero upstream gradient at the pad steps
        big4 = big.view(4, M, B, Lp).permute(2, 0, 1, 3)
        g_big = torch.empty_like(big)
        g4 = g_big.view(4, M, B, Lp).permute(2, 0, 1, 3)               # (B, 4, M, Lp) view, like big4
        gflat = g_big.view(4, M * B * Lp)
        for k in range(4):                                             # dB, dC are accumulated with atomics (ddelta is written):
            gflat[k, :2 * N * B * Lp].zero_()                          # four contiguous fills instead of one strided one
        du, _, dA, _, _, dD, dbias, _ = launch_bwd(x2.permute(2, 0, 1, 3), big4[:, :, 2 * N:], A32, big4[:, :, :N], big4[:, :, N:2 * N],
                                                   D32, None, b32, True, ckpt, d2, REV_MASK, 2, 2, True, True,
                                                   ddelta=g4[:, :, 2 * N:], dB=g4[:, :, :N], dC=g4[:, :, N:2 * N], algo_len=L)
        if Lp != L:
            du = du[:, :, :L].contiguous()
        x2m = x2.view(2, D, B * Lp)
        with _Tf32(tf32):
            dW = _weight_grad_splitk(g_big, x2m)                       # (2, 2M, D)
            gx2 = torch.bmm(Wm.transpose(1, 2), g_big)                 # (2, D, B*Lp)
        dx = torch.empty((B, D, H, W), dtype=torch.float32, device=dev)
        _lib.launch("b200_cross_scan_unpack4", dev, du.data_ptr(), gx2.data_ptr(), Lp, D * B * Lp, B * Lp, dx.data_ptr(), B, D, H, W)
        wdt, adt, ddt, bdt = ctx.dtypes
        return dx, dW.view(4, M, D).to(wdt), dA.to(adt), dD.to(ddt), dbias.to(bdt), None, None


def ss2d_core(x, W_all, A, Ds, delta_bias, N, tf32=False):
    return SS2DCoreFn.apply(x, W_all, A, Ds, delta_bias, N, tf32)


class CrossScan4SplitFn(torch.autograd.Function):
    """cross_scan4 of the channel slices `sizes` of x (B, C, H, W) (SSD/MedSSD.py:328-336: split into x, B, C, dt, then the
    four-direction scan of each) as ONE node: the backward writes the four adjoints straight into the channel slices of one
    (B, C, H, W) gradient instead of four tensors that autograd would then concatenate (1.4 ms of `cat` per MedSSD step)."""

    @staticmethod
    @_no_autocast
    def forward(ctx, x, *sizes):
        _lib.require_cuda(x)
        x = x.float()
        B, C, H, W = x.shape
        assert sum(sizes) == C
        if not (x.stride(3) == 1 and x.stride(2) == W and x.stride(1) == H * W):
            x = x.contiguous()
        outs, c0 = [], 0
        for n in sizes:
            o = torch.empty((B, 4, n, H * W), dtype=torch.float32, device=x.device)
            _lib.launch("b200_cross_scan4", x.device, x[:, c0:c0 + n].data_ptr(), x.stride(0), o.data_ptr(), B, n, H, W)
            outs.append(o)
            c0 += n
        ctx.meta = (B, C, H, W, tuple(sizes))
        return tuple(outs)

    @staticmethod
    @_no_autocast
    def backward(ctx, *douts):
        B, C, H, W, sizes = ctx.meta
        dev = next(g for g in douts if g is not None).device
        dx = torch.empty((B, C, H, W), dtype=torch.float32, device=dev)
        c0 = 0
        for n, g in zip(sizes, douts):
            part = dx[:, c0:c0 + n]
            if g is None:
                part.zero_()
            else:
                g = g.float().contiguous()
                _lib.launch("b200_cross_scan4_bwd", dev, g.data_ptr(), part.data_ptr(), dx.stride(0), B, n, H, W)
            c0 += n
        return (dx,) + (None,) * len(sizes)


def cross_scan4_split(x, sizes):
    return CrossScan4SplitFn.apply(x, *sizes)


class SsdMerge4Fn(torch.autograd.Function):
    """SSD twin of the cross-merge: y (B, L, 4, d) fp32 -> (B, L, d), the four directions un-permuted and summed
    (SSD/MedSSD.py:380-391)."""

    @staticmethod
    @_no_autocast
    def forward(ctx, y, H, W):
        _lib.require_cuda(y)
        y = y.float().contiguous()
        B, L, K, d = y.shape
        assert K == 4 and L == H * W
        out = torch.empty((B, L, d), dtype=torch.float32, device=y.device)
        _lib.launch("b200_ssd_merge4", y.device, y.data_ptr(), out.data_ptr(), B, d, H, W)
        ctx.meta = (B, L, d, H, W)
        return out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout):
        B, L, d, H, W = ctx.meta
        dout = dout.float().contiguous()
        dy = torch.empty((B, L, 4, d), dtype=torch.float32, device=dout.device)
        _lib.launch("b200_ssd_merge4_bwd", dout.device, dout.data_ptr(), dy.data_ptr(), B, d, H, W)
        return dy, None, None


def cross_scan4(x):
    """SSD twin of the cross-scan: x (B, C, H, W) fp32 (a channel slice of a wider NCHW tensor is read in place) ->
    x4 (B, 4, C, L) in the reference's direction order (hw, wh, hw reversed, wh reversed; SSD/MedSSD.py:332-336)."""
    return cross_scan4_split(x, (x.shape[1],))[0]


def ssd_merge4(y, H, W):
    return SsdMerge4Fn.apply(y, H, W)


def cross_scan_pack(x):
    return CrossScanPackFn.apply(x)


def cross_merge(ys, H, W):
    return CrossMergeFn.apply(ys, H, W)
