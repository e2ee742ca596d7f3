"""SS2D_with_SSD block (Mamba-2 SSD four-direction 2-D scan) -- B200 mirror of the reference module
`SS2D_with_SSD` (reference SSD/MedSSD.py:160-402; AST-identical copies in CNN_Mamba.py,
MedSSD_kan/*.py, medmamba_kan/*.py): same constructor arguments, same parameter names and shapes
(`in_proj.weight, conv2d.{weight,bias}, dt_bias (4, nheads), A_logs (4*nheads), Ds (4*nheads),
norm.weight, out_proj.weight`), so reference checkpoints load with strict=True, and the same
`forward((B,H,W,C)) -> (B,H,W,C)`.

The scan itself is `mamba_chunk_scan_combined` from .ssd_combined (libb200ssm, csrc/ssd.cu), called
with exactly the tensors the reference builds (SSD/MedSSD.py:332-375): (b, l, .) views of
channel-major storage, ngroups groups of 4*d_state states (one in the reference).  The gated RMSNorm
(`mamba_ssm...layernorm_gated.RMSNorm`, SSD/MedSSD.py:268-269,393-394) is .ssd_combined.RMSNormGated, with
group_size = d_ssm / ngroups and either order of norm and gate.
Tensor / sequence parallel branches of the reference constructor (process_group is always None
there, SURVEY.md 2.4) are not mirrored.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .cross import cross_scan4_split, ssd_merge4
from .ss2d import DwConvSiluFn, _autocast_out_dtype
from .ssd_combined import RMSNormGated, mamba_chunk_scan_combined


class SS2D_with_SSD(nn.Module):
    def __init__(self, d_model, d_state=128, d_conv=3, expand=2, headdim=64, d_ssm=None, ngroups=1,
                 A_init_range=(1, 16), D_has_hdim=False, rmsnorm=True, norm_before_gate=False, dt_rank="auto",
                 dt_min=0.001, dt_max=0.1, dt_init="random", dt_scale=1.0, dt_init_floor=1e-4,
                 dt_limit=(0.0, float("inf")), dropout=0.0, conv_bias=True, bias=False, chunk_size=256,
                 use_mem_eff_path=True, layer_idx=None, process_group=None, sequence_parallel=True,
                 device=None, dtype=None, **kwargs):
        fk = {"device": device, "dtype": dtype}
        super().__init__()
        if process_group is not None:
            raise NotImplementedError("SS2D_with_SSD: tensor parallelism is dead code in the reference (process_group=None)")
        self.d_model, self.d_state, self.d_conv, self.expand = d_model, d_state, d_conv, expand
        self.d_inner = int(expand * d_model)
        self.headdim = headdim
        self.d_ssm = self.d_inner if d_ssm is None else d_ssm
        self.ngroups = ngroups
        assert self.d_ssm % headdim == 0
        self.nheads = self.d_ssm // headdim
        self.D_has_hdim, self.rmsnorm, self.norm_before_gate = D_has_hdim, rmsnorm, norm_before_gate
        self.dt_limit, self.chunk_size = dt_limit, chunk_size
        self.dt_rank = math.ceil(d_model / 16) if dt_rank == "auto" else dt_rank

        # order: [z, x, B, C, dt]  (SSD/MedSSD.py:224-225)
        d_in_proj = 2 * self.d_inner + 2 * ngroups * d_state + self.nheads
        self.in_proj = nn.Linear(d_model, d_in_proj, bias=bias, **fk)
        conv_dim = self.d_ssm + 2 * ngroups * d_state + self.nheads
        self.conv2d = nn.Conv2d(conv_dim, conv_dim, groups=conv_dim, bias=conv_bias, kernel_size=d_conv,
                                padding=(d_conv - 1) // 2, **fk)
        self.act = nn.SiLU()

        dt = torch.exp(torch.rand(self.nheads, **fk) * (math.log(dt_max) - math.log(dt_min)) + math.log(dt_min))
        dt = torch.clamp(dt, min=dt_init_floor)
        inv_dt = dt + torch.log(-torch.expm1(-dt))
        self.dt_bias = nn.Parameter(torch.stack([inv_dt] * 4, dim=0))                 # (4, nheads)
        self.dt_bias._no_weight_decay = True
        A = torch.empty(self.nheads, dtype=torch.float32, device=device).uniform_(*A_init_range)
        self.A_logs = nn.Parameter(torch.log(A).to(dtype=dtype).repeat(4))            # (4*nheads)
        self.A_logs._no_weight_decay = True
        self.Ds = nn.Parameter(torch.ones(4 * (self.d_ssm if D_has_hdim else self.nheads), device=device))
        self.Ds._no_weight_decay = True
        if rmsnorm:
            self.norm = RMSNormGated(self.d_ssm, eps=1e-5, norm_before_gate=norm_before_gate,
                                     group_size=self.d_ssm // ngroups, **fk)
        self.out_proj = nn.Linear(self.d_inner, d_model, bias=bias, **fk)
        self.dropout = nn.Dropout(dropout) if dropout > 0.0 else None

    def forward(self, u: torch.Tensor, seqlen=None, seq_idx=None, cu_seqlens=None):
        B, H, W, C = u.shape
        L, K = H * W, 4
        zxbcdt = self.in_proj(u)
        d_mlp = (zxbcdt.shape[-1] - 2 * self.d_ssm - 2 * self.ngroups * self.d_state - self.nheads) // 2
        z0, x0, z, xBCdt = torch.split(
            zxbcdt, [d_mlp, d_mlp, self.d_ssm, self.d_ssm + 2 * self.ngroups * self.d_state + self.nheads], dim=-1)
        _lib.require_cuda(xBCdt)                                                        # no CPU path
        if self.d_conv == 3 and W <= 64 and xBCdt.dtype in (torch.float32, torch.bfloat16):
            xBCdt = DwConvSiluFn.apply(xBCdt, self.conv2d.weight, self.conv2d.bias)    # conv3x3 + SiLU, channels-last slice in place -> fp32 planes (B, c, H, W)
        else:   # outside the kernel's envelope: the reference's library ops
            xBCdt = self.act(self.conv2d(xBCdt.permute(0, 3, 1, 2).contiguous()))       # (B, c, H, W)

        # cross-scan of x, B, C and dt (SSD/MedSSD.py:332-336)
        gn = self.ngroups * self.d_state
        # one pass per component (csrc/cross.cu::cross_scan4_kernel), channel slices read in place
        xs, Bs, Cs, dts = cross_scan4_split(xBCdt, (self.d_ssm, gn, gn, self.nheads))   # one node: its backward fills one gradient tensor
        # (b, l, k*d) views with L stride 1 -- never made contiguous (SSD/MedSSD.py:344-347)
        xs = xs.float().reshape(B, -1, L).permute(0, 2, 1).unflatten(2, (-1, self.headdim))     # (B, L, 4*nheads, P)
        Bs = Bs.float().reshape(B, -1, L).permute(0, 2, 1).unflatten(2, (self.ngroups, -1))     # (B, L, G, 4*N)
        Cs = Cs.float().reshape(B, -1, L).permute(0, 2, 1).unflatten(2, (self.ngroups, -1))
        dts = dts.float().reshape(B, -1, L).permute(0, 2, 1)                                   # (B, L, 4*nheads)
        As = -torch.exp(self.A_logs.float())
        Ds = self.Ds.view(-1, self.headdim) if self.D_has_hdim else self.Ds
        kw = {} if tuple(self.dt_limit) == (0.0, float("inf")) else dict(dt_limit=self.dt_limit)
        y = mamba_chunk_scan_combined(xs, dts, As, Bs, Cs, chunk_size=self.chunk_size, D=Ds, z=None,
                                      dt_bias=self.dt_bias.view(-1), dt_softplus=True, seq_idx=seq_idx,
                                      cu_seqlens=cu_seqlens, **kw)                              # (B, L, 4*nheads, P)
        y = y.reshape(B, L, K, -1)
        assert y.dtype == torch.float32

        # cross-merge in the (B, L, K, d) layout (SSD/MedSSD.py:380-391)
        out = ssd_merge4(y, H, W).view(B, H, W, -1)                                             # one gather pass (csrc/cross.cu)

        if self.rmsnorm:
            out = self.norm(out, z, out_dtype=_autocast_out_dtype())   # z read in place from zxbcdt; bf16 out under bf16 autocast
        if d_mlp > 0:
            out = torch.cat([F.silu(z0) * x0, out], dim=-1)
        out = self.out_proj(out.to(self.out_proj.weight.dtype) if not torch.is_autocast_enabled() else out)
        if self.dropout is not None:
            out = self.dropout(out)
        return out
