"""MedMamba (VSSM) classifier built on the B200 SS2D block -- module tree and parameter names follow
the reference `MedMamba.py` (PatchEmbed2D :146-169, PatchMerging2D :172-212, channel_shuffle
:486-499, SS_Conv_SSM :502-538, VSSLayer :541-604, VSSM :671-767) so that a reference state_dict
loads with strict=True.  MedMamba-T = VSSM(depths=[2,2,4,2], dims=[96,192,384,768]) (defaults).

This file is host-side glue around the hot path (ss2d.SS2D); convolutions, linears and norms stay
on cuDNN/cuBLAS exactly as in the reference.
"""
from __future__ import annotations

from functools import partial

import torch

import torch.nn as nn

from . import _lib
from ._lib import no_autocast as _no_autocast
from .ss2d import SS2D, LnGateFn, layer_norm_rows, split_halves
from .ss2d_ssd import SS2D_with_SSD


class DropPath(nn.Module):
    """Stochastic depth per sample (the reference takes it from timm)."""

    def __init__(self, drop_prob: float = 0.0):
        super().__init__()
        self.drop_prob = float(drop_prob)

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        mask = x.new_empty((x.shape[0],) + (1,) * (x.dim() - 1)).bernoulli_(keep)
        return x * mask.div_(keep)

    def extra_repr(self):
        return f"drop_prob={self.drop_prob}"


def _layer_norm(x, norm):
    """nn.LayerNorm over the last dimension through libb200ssm's row kernel (csrc/lngate.cu), whose backward
    replaces PyTorch's gamma/beta reduction (3.9 % of the step at 200 K rows x 96 channels).  Output dtype follows
    autocast like F.layer_norm's consumer would see it (fp32 without autocast)."""
    if isinstance(norm, nn.LayerNorm) and norm.elementwise_affine and x.shape[-1] <= 1024 and x.dtype in (torch.float32, torch.bfloat16):
        x = x.contiguous()   # rows contiguous (no-op when already so); fp32 or bf16 rows are read as they are
        return LnGateFn.apply(x, None, norm.weight, norm.bias, norm.eps, torch.float32)
    return norm(x)


class PatchEmbed2D(nn.Module):
    def __init__(self, patch_size=4, in_chans=3, embed_dim=96, norm_layer=None, **kwargs):
        super().__init__()
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.norm = norm_layer(embed_dim) if norm_layer is not None else None

    def forward(self, x):
        # channels-last convolution: its output IS the (B, H, W, C) tensor the blocks consume, the permute below is a view and the
        # LayerNorm kernel reads it in place (no NCHW -> NHWC copy forward, none backward; A/B 20.17-20.75 -> 20.12-20.13 ms per step)
        x = x.contiguous(memory_format=torch.channels_last)
        x = self.proj(x).permute(0, 2, 3, 1)
        if self.norm is None:
            return x
        return _layer_norm(x, self.norm)


class PatchMergeGatherFn(torch.autograd.Function):
    """The 2x2 gather of PatchMerging2D (`x0..x3 = x[:, i::2, j::2, :]`, `torch.cat`, MedMamba.py:186-204) in one pass; the backward is
    the inverse permutation (csrc/glue.cu::patch_merge_kernel)."""

    @staticmethod
    def forward(ctx, x):
        _lib.require_cuda(x)
        x = x.contiguous()
        B, H, W, C = x.shape
        out = torch.empty((B, H // 2, W // 2, 4 * C), dtype=x.dtype, device=x.device)
        _lib.launch("b200_patch_merge", x.device, x.data_ptr(), out.data_ptr(), B, H, W, C * x.element_size(), 0)
        ctx.shape = (B, H, W, C)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, H, W, C = ctx.shape
        dout = dout.contiguous()
        dx = torch.empty((B, H, W, C), dtype=dout.dtype, device=dout.device)
        _lib.launch("b200_patch_merge", dout.device, dout.data_ptr(), dx.data_ptr(), B, H, W, C * dout.element_size(), 1)
        return dx


class PatchMerging2D(nn.Module):
    """2x2 patch merge: (B, H, W, C) -> (B, H/2, W/2, 2C)."""

    def __init__(self, dim, norm_layer=nn.LayerNorm):
        super().__init__()
        self.dim = dim
        self.reduction = nn.Linear(4 * dim, 2 * dim, bias=False)
        self.norm = norm_layer(4 * dim)

    def forward(self, x):
        B, H, W, C = x.shape
        h2, w2 = H // 2, W // 2
        if (C * x.element_size()) % 16 == 0 and h2 > 0 and w2 > 0:
            x = PatchMergeGatherFn.apply(x)                # one gather pass (csrc/glue.cu)
        else:
            parts = [x[:, i::2, j::2, :][:, :h2, :w2, :] for (i, j) in ((0, 0), (1, 0), (0, 1), (1, 1))]
            x = torch.cat(parts, dim=-1)
        return self.reduction(_layer_norm(x, self.norm))


def channel_shuffle(x, groups: int):
    B, H, W, C = x.shape
    return x.view(B, H, W, groups, C // groups).transpose(3, 4).reshape(B, H, W, C)


class ShuffleCatAddFn(torch.autograd.Function):
    """out (B, H, W, 2c) = channel_shuffle(cat(left^T, x), 2) + input with left the conv branch's (B, c, H, W)
    output -- NCHW planes or torch.channels_last -- and x (B, H, W, c) channels-last (csrc/glue.cu) -- reference
    MedMamba.py:486-499, 533-538.  out has torch's promoted dtype: fp32 for an fp32 residual stream, bf16 when the
    stream and both branches are bf16 (stages 1-3 of an autocast model)."""

    @staticmethod
    @_no_autocast
    def forward(ctx, left, x, inp):
        _lib.require_cuda(left, x, inp)
        B, c, H, W = left.shape
        cl = left.is_contiguous(memory_format=torch.channels_last) and not left.is_contiguous()
        if not cl:
            left = left.contiguous()
        if inp.dtype == torch.bfloat16 and left.dtype != torch.bfloat16:
            inp = inp.float()                                  # torch would promote the sum to fp32
        x, inp = x.to(left.dtype).contiguous(), inp.contiguous()
        out = torch.empty((B, H, W, 2 * c), dtype=inp.dtype, device=inp.device)
        _lib.launch("b200_shuffle_cat_add_fwd", inp.device, left.data_ptr(), int(cl), x.data_ptr(), _lib.dtype_code(left.dtype),
                    inp.data_ptr(), out.data_ptr(), _lib.dtype_code(inp.dtype), B, c, H * W)
        ctx.meta = (B, c, H, W, left.dtype, cl, inp.dtype)
        return out

    @staticmethod
    @_no_autocast
    def backward(ctx, dout):
        B, c, H, W, ldt, cl, iodt = ctx.meta
        dout = dout.to(iodt).contiguous()
        dleft = torch.empty((B, c, H, W), dtype=ldt, device=dout.device, memory_format=torch.channels_last if cl else torch.contiguous_format)
        dx = torch.empty((B, H, W, c), dtype=ldt, device=dout.device)
        _lib.launch("b200_shuffle_cat_add_bwd", dout.device, dout.data_ptr(), _lib.dtype_code(iodt), dleft.data_ptr(), int(cl), dx.data_ptr(),
                    _lib.dtype_code(ldt), B, c, H * W)
        return dleft, dx, dout


_BRANCH_STREAMS = {}


def branch_stream(device):
    """The side stream (one per device) on which the blocks' convolution branch runs while the SS2D branch runs on the
    caller's stream."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    st = _BRANCH_STREAMS.get(key)
    if st is None:
        st = _BRANCH_STREAMS[key] = torch.cuda.Stream(device=device)
    return st


class SS_Conv_SSM(nn.Module):
    """Two-branch block: half the channels through conv3x3-conv3x3-conv1x1, half through
    LayerNorm -> SS2D; concat, channel shuffle, residual."""

    def __init__(self, hidden_dim=0, drop_path=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                 attn_drop_rate=0.0, d_state=16, **kwargs):
        super().__init__()
        c = hidden_dim // 2
        self.ln_1 = norm_layer(c)
        self.self_attention = SS2D(d_model=c, dropout=attn_drop_rate, d_state=d_state, **kwargs)
        self.drop_path = DropPath(drop_path)
        self.conv33conv33conv11 = nn.Sequential(
            nn.BatchNorm2d(c),
            nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1),
            nn.BatchNorm2d(c),
            nn.ReLU(),
            nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1),
            nn.BatchNorm2d(c),
            nn.ReLU(),
            nn.Conv2d(c, c, kernel_size=1, stride=1),
            nn.ReLU(),
        )

    # The two branches of a block are independent until the concatenation (MedMamba.py:533-538).  On CUDA the convolution branch
    # (cuDNN convolutions, BatchNorm, ReLU: bandwidth-bound library kernels) is issued on a side stream and the SS2D branch on the
    # caller's: the scan kernels leave issue slots, DRAM bandwidth and -- at the end of their single wave -- whole SMs idle, which
    # the other branch's kernels fill.  Autograd replays each op on its forward stream, so the backward overlaps the same way, and
    # the fork / join is captured like any other dependency when the step is recorded in a CUDA graph.  Measured (bench.py, N = 1):
    # 23.80 -> 20.89 ms per MedMamba-T step, 98.8 -> 96.9 ms per MedSSD step.  Stream priorities (SS2D branch on a high-priority
    # stream) made no difference (21.17-21.22 ms on one box).
    overlap_branches = True

    def _conv_branch(self, left):
        # the conv branch consumes channels-last data: on CUDA keep it in torch.channels_last (cuDNN / BatchNorm run NHWC
        # natively: no NCHW<->NHWC converter kernels; measured 33.2 -> 29.2 ms per MedMamba-T step)
        left = left.permute(0, 3, 1, 2)
        left = left.contiguous(memory_format=torch.channels_last)
        return self.conv33conv33conv11(left)

    def forward(self, input):
        _lib.require_cuda(input)                           # no CPU path: oracle/cpu_path.py holds the eager CPU tree
        left, right = split_halves(input)
        side = None
        if self.overlap_branches:
            cur = torch.cuda.current_stream(input.device)
            side = branch_stream(input.device)
            side.wait_stream(cur)                          # fork: `left` is ready on the caller's stream
            with torch.cuda.stream(side):
                left = self._conv_branch(left)
        if right.dtype in (torch.float32, torch.bfloat16) and isinstance(self.ln_1, nn.LayerNorm) and right.shape[-1] <= 1024:
            normed = layer_norm_rows(right, self.ln_1)     # pre-norm, the right half read in place (csrc/lngate.cu)
        else:
            normed = self.ln_1(right)
        x = self.drop_path(self.self_attention(normed))
        if side is not None:
            cur.wait_stream(side)                          # join
            left.record_stream(cur)                        # allocated on the side stream, consumed (and later freed) on this one
        else:
            left = self._conv_branch(left)
        if (input.dtype in (torch.float32, torch.bfloat16) and left.dtype in (torch.float32, torch.bfloat16)
                and x.dtype in (torch.float32, torch.bfloat16) and left.shape[0] <= 65535):
            return ShuffleCatAddFn.apply(left, x, input)   # cat + channel shuffle + residual in one pass (csrc/glue.cu)
        left = left.permute(0, 2, 3, 1)
        out = channel_shuffle(torch.cat((left, x.to(left.dtype)), dim=-1), groups=2)
        return out + input


class SS_Conv_SSD(SS_Conv_SSM):
    """The same two-branch block with the SSD mixer (reference SSD/MedSSD.py:421-457)."""

    def __init__(self, hidden_dim=0, drop_path=0.0, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                 attn_drop_rate=0.0, d_state=64, **kwargs):
        nn.Module.__init__(self)
        c = hidden_dim // 2
        self.ln_1 = norm_layer(c)
        self.self_attention = SS2D_with_SSD(d_model=c, dropout=attn_drop_rate, d_state=d_state, **kwargs)
        self.drop_path = DropPath(drop_path)
        self.conv33conv33conv11 = nn.Sequential(
            nn.BatchNorm2d(c),
            nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1),
            nn.BatchNorm2d(c),
            nn.ReLU(),
            nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1),
            nn.BatchNorm2d(c),
            nn.ReLU(),
            nn.Conv2d(c, c, kernel_size=1, stride=1),
            nn.ReLU(),
        )


class VSSLayer(nn.Module):
    def __init__(self, dim, depth, attn_drop=0.0, drop_path=0.0, norm_layer=nn.LayerNorm, downsample=None,
                 use_checkpoint=False, d_state=16, block=SS_Conv_SSM, **kwargs):
        super().__init__()
        self.dim = dim
        self.use_checkpoint = use_checkpoint
        self.blocks = nn.ModuleList([
            block(hidden_dim=dim, drop_path=drop_path[i] if isinstance(drop_path, (list, tuple)) else drop_path,
                        norm_layer=norm_layer, attn_drop_rate=attn_drop, d_state=d_state)
            for i in range(depth)])
        self.downsample = downsample(dim=dim, norm_layer=norm_layer) if downsample is not None else None

    def forward(self, x):
        for blk in self.blocks:
            x = torch.utils.checkpoint.checkpoint(blk, x, use_reentrant=False) if self.use_checkpoint else blk(x)
        return self.downsample(x) if self.downsample is not None else x


class VSSM(nn.Module):
    def __init__(self, patch_size=4, in_chans=3, num_classes=1000, depths=(2, 2, 4, 2), dims=(96, 192, 384, 768),
                 d_state=16, drop_rate=0.0, attn_drop_rate=0.0, drop_path_rate=0.1, norm_layer=nn.LayerNorm,
                 patch_norm=True, use_checkpoint=False, block=SS_Conv_SSM, **kwargs):
        super().__init__()
        depths, n = list(depths), len(depths)
        dims = [int(dims * 2 ** i) for i in range(n)] if isinstance(dims, int) else list(dims)
        self.num_classes, self.num_layers = num_classes, n
        self.embed_dim, self.num_features, self.dims = dims[0], dims[-1], dims
        self.patch_embed = PatchEmbed2D(patch_size=patch_size, in_chans=in_chans, embed_dim=dims[0],
                                        norm_layer=norm_layer if patch_norm else None)
        self.pos_drop = nn.Dropout(p=drop_rate)
        dpr = torch.linspace(0, drop_path_rate, sum(depths)).tolist()
        self.layers = nn.ModuleList()
        for i in range(n):
            self.layers.append(VSSLayer(
                dim=dims[i], depth=depths[i], d_state=d_state, attn_drop=attn_drop_rate,
                drop_path=dpr[sum(depths[:i]):sum(depths[:i + 1])], norm_layer=norm_layer,
                downsample=PatchMerging2D if i < n - 1 else None, use_checkpoint=use_checkpoint, block=block))
        self.avgpool = nn.AdaptiveAvgPool2d(1)
        self.head = nn.Linear(self.num_features, num_classes) if num_classes > 0 else nn.Identity()
        self.apply(self._init_weights)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")

    @staticmethod
    def _init_weights(m):
        if isinstance(m, nn.Linear):
            nn.init.trunc_normal_(m.weight, std=0.02, a=-2.0, b=2.0)
            if m.bias is not None:
                nn.init.zeros_(m.bias)
        elif isinstance(m, nn.LayerNorm):
            nn.init.ones_(m.weight)
            nn.init.zeros_(m.bias)

    def forward_backbone(self, x):
        x = self.pos_drop(self.patch_embed(x))
        for layer in self.layers:
            x = layer(x)
        return x

    def forward(self, x):
        x = self.forward_backbone(x)
        x = self.avgpool(x.permute(0, 3, 1, 2)).flatten(1)
        return self.head(x)


class VSSM_KAN(VSSM):
    """MedSSD_kan: the SSD backbone with the KAN classification head `kans` in place of `head`
    (reference MedSSD_kan/MedSSD_kan.py:1097-1204; d_state 16 -> N' = 64)."""

    def __init__(self, num_classes=1000, dims=(128, 256, 512, 1024), d_state=16, block=None, **kw):
        from .kan_head import KansModule
        super().__init__(num_classes=0, dims=dims, d_state=d_state, block=block or SS_Conv_SSD, **kw)
        del self.head
        self.num_classes = num_classes
        self.kans = KansModule(in_channels=self.num_features, out_channels=num_classes)

    def forward(self, x, update_grid=False):
        x = self.forward_backbone(x)
        x = self.avgpool(x.permute(0, 3, 1, 2)).flatten(1)
        return self.kans(x.float())


def medmamba_t(num_classes=6, **kw):
    """MedMamba-T, the configuration BASELINE.json names (depths 2-2-4-2, dims 96-768)."""
    return VSSM(num_classes=num_classes, depths=[2, 2, 4, 2], dims=[96, 192, 384, 768], **kw)


def medssd_kan(num_classes=6, dims=(128, 256, 512, 1024), d_state=16, depths=(2, 2, 4, 2), **kw):
    """MedSSD_kan (BASELINE.json configs[3]): MedSSD backbone, d_state 16, KAN head."""
    return VSSM_KAN(num_classes=num_classes, depths=list(depths), dims=list(dims), d_state=d_state, **kw)


def medssd(num_classes=6, dims=(128, 256, 512, 1024), d_state=128, depths=(2, 2, 4, 2), **kw):
    """MedSSD: the SSD/MedSSD.py VSSM defaults (depths 2-2-4-2, dims 128-1024, d_state 128), BASELINE.json configs[2].
    MedSSD_kan / CNN_Mamba backbones are the same graph with d_state=16."""
    return VSSM(num_classes=num_classes, depths=list(depths), dims=list(dims), d_state=d_state, block=SS_Conv_SSD, **kw)
