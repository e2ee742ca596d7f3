"""Every dispatch path of the Mamba-1 selective scan against the fp64 oracle, with the path that served each call asserted.

b200_sscan_fwd / b200_sscan_bwd pick a kernel per call (csrc/sscan.cu, host side): sscan2.cu ("v2", TMA-staged, fp32,
L % 4 == 0, tensor-map-describable layouts, backward without z) or sscan.cu ("v1": 16-byte cp.async staging, element-wise
staging for L % 4 != 0 / unaligned views, the opt-in TMA row staging, 16-bit I/O).  b200_sscan_last_variant() reports
1 (sscan.cu), 2 (sscan2.cu) or 3 (sscan.cu with TMA staging).  `expected_fwd` / `expected_bwd` below restate the
eligibility rules (v2::try_fwd / try_bwd / make_*_maps, v1 make_fwd_maps / make_row_map / can_vectorize), so a change of the
dispatch rules fails here instead of silently moving a case to another kernel.

The calls are made at the C ABI (params filled by selective_scan_interface._fill_fwd), so every output lands in a
caller-owned buffer: out / du / ddelta / dz in a buffer prefilled with a NaN payload, with a row pitch > L and gaps between
rows, groups and batches; dB / dC zero inside their view and NaN outside.  After each call everything outside the views must be
bit-for-bit unchanged (TMA stores and reduce-adds clip to the tensor map's dimensions).  Inputs with a pitch carry NaN in the
padding too, so reading outside a view poisons the result.

The environment switches are read once per process, so each configuration runs the whole case list once in a child process
(this file's __main__), which writes one .npz; the parent computes the oracle once per case and checks every configuration:

    config   env                                     fwd / bwd variant
    default  -                                       2 / 2 where eligible, otherwise 1
    v1       B200_SSCAN_V1=1                         1 / 1
    v1tma    B200_SSCAN_V1=1 B200_SSCAN_TMA=1        3 / 3 where v1's TMA maps apply, otherwise 1
    bwdv1    B200_SSCAN_BWD_V1=1                     2 / 1 (v2 checkpoints consumed by the v1 backward)

Oracle: oracle.sscan_fwd / sscan_bwd (fp64), per group; a reversed group is the plain scan of its time-flipped rows with
outputs and gradients flipped back (its last_state is the state after position 0); u_group_div / dout_group_div repeat the
shared u / dout rows.  du is compared per channel, as the kernel writes it (callers sum it over the groups sharing a row).

Tolerances (as tests/test_sscan_parity.py): norm-wise relative error max|a-b| / max|b| <= 1e-5 on out and last_state, 2e-5
on every gradient, and the reference's element-wise bounds (test_selective_scan.py:398-404) on top; 16-bit I/O gets the
reference's element-wise bounds only.

Cases (batch 2 unless noted; rows = channels per group; "pad": every input with a NaN-padded pitch; "ugroup": u as the
x2.permute(2, 0, 1, 3) view; "proj": delta / B / C as slices of one projection buffer (state stride > L); "gbig": ddelta / dB /
dC as views of one wider gradient buffer; "wide": delta + bias uniform in [-30, 30]; "fn": selective_scan_fn's 16-state slices):

    name                L    rows  N   G  rev     ugd dgd  flags                 layout     grads
    L4                  4    16    16  1  0       1   1    sp D bias last        contig     own
    L8_r1_N1            8    1     1   1  0       1   1    -                     pad        own
    L12_rev             12   3     2   2  0101    1   1    sp D bias             pad        own
    L16_rev             16   8     5   2  1010    1   1    sp D last             contig     own
    L20_overhang        20   15    8   4  1111    1   1    sp bias last          pad        own
    L28_ugd             28   17    15  2  1010    2   1    sp D bias             ugroup     own
    L36_ss2d_like       36   24    16  4  1010    2   2    sp D bias             ugroup     gbig
    L44_dgd             44   33    5   2  0101    1   2    D bias                proj       own
    L64_z               64   16    16  2  0       1   1    sp D bias z last      contig     own
    L100_z_nosp         100  24    8   2  1010    1   1    D z                   pad        own
    L132_rev            132  17    2   4  1111    2   2    sp bias last          proj       gbig
    L200_tma_case       200  24    16  4  1010    1   1    sp D bias             contig     own
    L260_long           260  33    16  2  0101    1   1    sp D bias last        pad        gbig
    L64_z_nosp_rev      64   8     16  2  1111    1   1    bias z                contig     own
    L36_z_dgd           36   15    1   2  1010    2   2    sp D z last           ugroup     own
    L16_z_N15           16   3     15  1  0       1   1    sp z                  proj       own
    L20_z_wide          20   16    16  2  0101    1   1    sp D bias z wide      contig     own
    L100_wide           100  17    16  2  1010    1   1    sp D bias wide last   contig     own
    L8_r24_N2           8    24    2   4  0101    2   1    sp bias               pad        gbig
    L12_r33_N8          12   33    8   1  1       1   1    D                     contig     own
    L4_rev_N15          4    15    15  2  1111    1   2    sp D bias last        contig     own
    L28_nosp            28   1     8   4  1010    1   1    -                     proj       own
    L44_r16_N1          44   16    1   2  1111    2   2    sp D bias last        ugroup     gbig
    L64_r3_N2           64   3     2   1  0       1   1    sp D bias last        proj       gbig
    L200_r15_N5         200  15    5   2  0101    2   1    sp bias               ugroup     own
    L132_r8             132  8     16  2  0       1   1    sp D bias z           pad        own
    L260_r24_nosp       260  24    15  4  1010    1   2    D                     contig     own
    L36_out_misaligned  36   16    16  4  1010    1   1    sp D bias             contig     own   out at +4 bytes: v1 fwd -> v2 bwd
    L1                  1    16    16  1  0       1   1    sp D bias last        contig     own
    L2_rev              2    3     5   2  1111    1   1    sp D bias             contig     own
    L3_z                3    8     16  2  1010    2   2    sp D bias z last      ugroup     own
    L5_r1               5    1     2   1  1       1   1    sp bias               pad        own
    L9_r17              9    17    8   2  0101    1   1    D                     contig     own
    L17_rev             17   24    15  4  1111    2   2    sp D bias last        ugroup     gbig
    L49_z               49   33    16  2  1010    1   1    sp D bias z           contig     own
    L49_proj_odd        49   16    16  4  1010    1   1    sp D bias             proj(R=3)  own
    L17_wide            17   16    16  2  0101    1   1    sp D bias z wide last contig     own
    L9_nosp_z           9    15    1   1  0       1   1    z                     pad        own
    fp16/bf16_L49       49   16    16  2  1010    2   1    sp D bias z           ugroup     own   (two cases)
    fp16/bf16_L17       17   24    5   4  0101    2   2    sp bias z last        contig     own   (two cases)
    fn_N17 / fn_N40     64   8     17/40 1 0       1   1    sp D bias z last      selective_scan_fn (16-state slices)
    ss2d_7x7            49   96    16  4  1010    2   2    sp D bias             SS2DCoreFn (x2 / big / g_big, Lp = 52)
"""
import ctypes
import os
import subprocess
import sys
import tempfile
from collections import Counter

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

CONFIGS = {
    "default": {},
    "v1": {"B200_SSCAN_V1": "1"},
    "v1tma": {"B200_SSCAN_V1": "1", "B200_SSCAN_TMA": "1"},
    "bwdv1": {"B200_SSCAN_BWD_V1": "1"},
}
SWITCHES = ("B200_SSCAN_V1", "B200_SSCAN_BWD_V1", "B200_SSCAN_TMA")
CKPT_EVERY = 8
SENT32 = 0x7FC0DEAD   # NaN payload of the fp32 sentinel
SENT16 = 0x7FDB       # a NaN in both fp16 and bf16


class Case:
    def __init__(self, name, L, rows, N, G=1, rev=0, ugd=1, dgd=1, flags="sp D bias", layout="contig", grads="own",
                 batch=2, dtype="f32", out_off=0, api="abi"):
        self.name, self.L, self.rows, self.N, self.G = name, L, rows, N, G
        self.rev, self.ugd, self.dgd, self.layout, self.grads = rev, ugd, dgd, layout, grads
        f = flags.split()
        self.softplus, self.has_D, self.has_bias = "sp" in f, "D" in f, "bias" in f
        self.has_z, self.last, self.wide = "z" in f, "last" in f, "wide" in f
        self.batch, self.dtype, self.out_off, self.api = batch, dtype, out_off, api
        self.dim = rows * G
        self.L_true = 49 if layout == "ss2d" else L     # SS2DCoreFn pads rows to a 16-byte pitch: the scan runs over Lp steps
        self.L = 52 if layout == "ss2d" else L

    def __repr__(self):
        return (f"{self.name}(L={self.L}, rows={self.rows}, N={self.N}, G={self.G}, rev={self.rev:#06b}, ugd={self.ugd}, "
                f"dgd={self.dgd}, softplus={self.softplus}, D={self.has_D}, bias={self.has_bias}, z={self.has_z}, "
                f"last={self.last}, wide={self.wide}, layout={self.layout}, grads={self.grads}, dtype={self.dtype}, "
                f"out_off={self.out_off}, api={self.api})")


CASES = [
    # v2-eligible sequence lengths (fp32, L % 4 == 0)
    Case("L4", 4, 16, 16, 1, flags="sp D bias last"),
    Case("L8_r1_N1", 8, 1, 1, 1, flags="", layout="pad"),
    Case("L12_rev", 12, 3, 2, 2, rev=0b0101, layout="pad"),
    Case("L16_rev", 16, 8, 5, 2, rev=0b1010, flags="sp D last"),
    Case("L20_overhang", 20, 15, 8, 4, rev=0b1111, flags="sp bias last", layout="pad"),
    Case("L28_ugd", 28, 17, 15, 2, rev=0b1010, ugd=2, layout="ugroup"),
    Case("L36_ss2d_like", 36, 24, 16, 4, rev=0b1010, ugd=2, dgd=2, layout="ugroup", grads="gbig"),
    Case("L44_dgd", 44, 33, 5, 2, rev=0b0101, dgd=2, flags="D bias", layout="proj"),
    Case("L64_z", 64, 16, 16, 2, flags="sp D bias z last"),
    Case("L100_z_nosp", 100, 24, 8, 2, rev=0b1010, flags="D z", layout="pad"),
    Case("L132_rev", 132, 17, 2, 4, rev=0b1111, ugd=2, dgd=2, flags="sp bias last", layout="proj", grads="gbig"),
    Case("L200_tma_case", 200, 24, 16, 4, rev=0b1010),
    Case("L260_long", 260, 33, 16, 2, rev=0b0101, flags="sp D bias last", layout="pad", grads="gbig"),
    Case("L64_z_nosp_rev", 64, 8, 16, 2, rev=0b1111, flags="bias z"),
    Case("L36_z_dgd", 36, 15, 1, 2, rev=0b1010, ugd=2, dgd=2, flags="sp D z last", layout="ugroup"),
    Case("L16_z_N15", 16, 3, 15, 1, flags="sp z", layout="proj"),
    Case("L20_z_wide", 20, 16, 16, 2, rev=0b0101, flags="sp D bias z wide"),
    Case("L100_wide", 100, 17, 16, 2, rev=0b1010, flags="sp D bias wide last"),
    Case("L8_r24_N2", 8, 24, 2, 4, rev=0b0101, ugd=2, flags="sp bias", layout="pad", grads="gbig"),
    Case("L12_r33_N8", 12, 33, 8, 1, rev=0b1, flags="D"),
    Case("L4_rev_N15", 4, 15, 15, 2, rev=0b1111, dgd=2, flags="sp D bias last"),
    Case("L28_nosp", 28, 1, 8, 4, rev=0b1010, flags="", layout="proj"),
    Case("L44_r16_N1", 44, 16, 1, 2, rev=0b1111, ugd=2, dgd=2, flags="sp D bias last", layout="ugroup", grads="gbig"),
    Case("L64_r3_N2", 64, 3, 2, 1, flags="sp D bias last", layout="proj", grads="gbig"),
    Case("L200_r15_N5", 200, 15, 5, 2, rev=0b0101, ugd=2, flags="sp bias", layout="ugroup"),
    Case("L132_r8", 132, 8, 16, 2, flags="sp D bias z", layout="pad"),
    Case("L260_r24_nosp", 260, 24, 15, 4, rev=0b1010, dgd=2, flags="D"),
    # out 4 bytes off a 16-byte boundary: v1 forward, every backward tensor aligned: v2 backward (v1 -> v2 checkpoint handoff)
    Case("L36_out_misaligned", 36, 16, 16, 4, rev=0b1010, out_off=1),
    # v1 only: L % 4 != 0
    Case("L1", 1, 16, 16, 1, flags="sp D bias last"),
    Case("L2_rev", 2, 3, 5, 2, rev=0b1111),
    Case("L3_z", 3, 8, 16, 2, rev=0b1010, ugd=2, dgd=2, flags="sp D bias z last", layout="ugroup"),
    Case("L5_r1", 5, 1, 2, 1, rev=0b1, flags="sp bias", layout="pad"),
    Case("L9_r17", 9, 17, 8, 2, rev=0b0101, flags="D"),
    Case("L17_rev", 17, 24, 15, 4, rev=0b1111, ugd=2, dgd=2, flags="sp D bias last", layout="ugroup", grads="gbig"),
    Case("L49_z", 49, 33, 16, 2, rev=0b1010, flags="sp D bias z"),
    Case("L49_proj_odd", 49, 16, 16, 4, rev=0b1010, layout="proj_odd"),
    Case("L17_wide", 17, 16, 16, 2, rev=0b0101, flags="sp D bias z wide last"),
    Case("L9_nosp_z", 9, 15, 1, 1, flags="z", layout="pad"),
    # 16-bit I/O (sscan.cu only)
    Case("bf16_L49", 49, 16, 16, 2, rev=0b1010, ugd=2, flags="sp D bias z", layout="ugroup", dtype="bf16"),
    Case("fp16_L49", 49, 16, 16, 2, rev=0b1010, ugd=2, flags="sp D bias z", layout="ugroup", dtype="fp16"),
    Case("bf16_L17", 17, 24, 5, 4, rev=0b0101, ugd=2, dgd=2, flags="sp bias z last", dtype="bf16"),
    Case("fp16_L17", 17, 24, 5, 4, rev=0b0101, ugd=2, dgd=2, flags="sp bias z last", dtype="fp16"),
    # dstate > 16 through selective_scan_fn's 16-state slices at L % 4 == 0
    Case("fn_N17", 64, 8, 17, 1, flags="sp D bias z last", api="fn"),
    Case("fn_N40", 64, 8, 40, 1, flags="sp D bias z last", api="fn"),
    # SS2DCoreFn's launch at the stage-3 plane: 7 x 7, rows padded to Lp = 52, dim 4 * 96
    Case("ss2d_7x7", 52, 96, 16, 4, rev=0b1010, ugd=2, dgd=2, layout="ss2d", batch=2),
]
CASE_BY_NAME = {c.name: c for c in CASES}
assert len(CASE_BY_NAME) == len(CASES)


# ---------------------------------------------------------------------------------------------------------------------
# seeded inputs (numpy, logical layout) -- identical in the parent and in every child
# ---------------------------------------------------------------------------------------------------------------------
def make_inputs(c, seed):
    r = np.random.RandomState(seed)
    f = lambda *s: r.randn(*s).astype(np.float32)
    b, dim, L, N, G = c.batch, c.dim, c.L, c.N, c.G
    x = dict(u=f(b, dim // c.ugd, L), A=(-0.5 * r.rand(dim, N) - 0.05).astype(np.float32),
             B=f(b, G, N, L), C=f(b, G, N, L), dout=f(b, dim // c.dgd, L))
    if c.wide:   # delta + bias spans [-30, 30]: crosses the softplus threshold at 20, decays of ~1 and ~0
        x["delta"] = r.uniform(-25, 25, (b, dim, L)).astype(np.float32)
        x["bias"] = r.uniform(-5, 5, dim).astype(np.float32)
    else:
        x["delta"] = (0.5 * r.rand(b, dim, L)).astype(np.float32)
        x["bias"] = (0.5 * r.rand(dim)).astype(np.float32)
    x["D"] = f(dim)
    if c.has_z:   # gates down to about -100 (silu(z) ~ 0, sigmoid underflows)
        z = 2.0 * f(b, dim, L)
        low = r.rand(b, dim, L) < 0.1
        z[low] = r.uniform(-100, -20, int(low.sum()))
        x["z"] = z.astype(np.float32)
    if not c.has_D:
        x["D"] = None
    if not c.has_bias:
        x["bias"] = None
    if c.L_true != c.L:   # SS2DCoreFn's pad steps: zero u / delta / B / C and zero upstream gradient
        for k in ("u", "delta", "B", "C", "dout"):
            x[k][..., c.L_true:] = 0.0
    if c.dtype != "f32":   # quantise the 16-bit inputs so both sides see the same numbers
        import torch
        dt = torch.bfloat16 if c.dtype == "bf16" else torch.float16
        for k in ("u", "delta", "B", "C", "z", "dout"):
            if x.get(k) is not None:
                x[k] = torch.tensor(x[k]).to(dt).float().numpy()
    return x


def case_seed(c):
    return 1000 + CASES.index(c)


# ---------------------------------------------------------------------------------------------------------------------
# the dispatch rules, restated (csrc/sscan2.cu try_fwd / try_bwd / make_*_maps, csrc/tma.cuh tma_make_map_f32,
# csrc/sscan.cu make_fwd_maps / make_row_map / bc_vec_ok / can_vectorize)
# ---------------------------------------------------------------------------------------------------------------------
def _fix(s, n):   # sscan2.cu fix_stride: a size-1 dimension's stride is free
    return 4 if n == 1 and (s <= 0 or s % 4) else s


def _map_ok(ptr, *strides):   # tma_make_map_f32 (element strides)
    return ptr % 16 == 0 and all(s > 0 and s % 4 == 0 and s * 4 < (1 << 40) for s in strides)


def _row_map_ok(ptr, L, *strides):   # sscan.cu make_row_map (no fix_stride there)
    return L % 4 == 0 and _map_ok(ptr, *strides)


def _v2_fwd_ok(p, env):
    if env.get("B200_SSCAN_V1") == "1" or p.io_dtype != 0 or p.dstate > 16 or p.seqlen % 4:
        return False
    if p.out % 16 or p.out_row_stride % 4 or p.out_batch_stride % 4:
        return False
    if p.z and (p.z % 16 or p.z_row_stride % 4 or p.z_batch_stride % 4):
        return False
    G, Bt, N = p.n_groups, p.batch, p.dstate
    rpg = p.dim // G
    if G % p.u_group_div:
        return False
    Gu = G // p.u_group_div
    return (_map_ok(p.u, _fix(p.u_row_stride, rpg), _fix(p.u_group_stride, Gu), _fix(p.u_batch_stride, Bt))
            and _map_ok(p.delta, _fix(p.delta_row_stride, rpg), _fix(p.delta_group_stride, G), _fix(p.delta_batch_stride, Bt))
            and _map_ok(p.B, _fix(p.B_state_stride, N), _fix(p.B_group_stride, G), _fix(p.B_batch_stride, Bt))
            and _map_ok(p.C, _fix(p.C_state_stride, N), _fix(p.C_group_stride, G), _fix(p.C_batch_stride, Bt)))


def _v2_bwd_ok(q, env):
    p = q.f
    if env.get("B200_SSCAN_V1") == "1" or env.get("B200_SSCAN_BWD_V1") == "1":
        return False
    if p.io_dtype != 0 or p.dstate > 16 or p.seqlen % 4 or p.z:
        return False
    G, Bt, N = p.n_groups, p.batch, p.dstate
    rpg = p.dim // G
    if G % p.u_group_div or G % q.dout_group_div:
        return False
    Gu, Gd = G // p.u_group_div, G // q.dout_group_div
    rows = lambda ptr, g, rs, gs, bs: _map_ok(ptr, _fix(rs, rpg), _fix(gs, g), _fix(bs, Bt))
    states = lambda ptr, ss, gs, bs: _map_ok(ptr, _fix(ss, N), _fix(gs, G), _fix(bs, Bt))
    return (rows(p.u, Gu, p.u_row_stride, p.u_group_stride, p.u_batch_stride)
            and rows(p.delta, G, p.delta_row_stride, p.delta_group_stride, p.delta_batch_stride)
            and rows(q.dout, Gd, q.dout_row_stride, q.dout_group_stride, q.dout_batch_stride)
            and rows(q.du, G, q.du_row_stride, rpg * q.du_row_stride, q.du_batch_stride)
            and rows(q.ddelta, G, q.ddelta_row_stride, q.ddelta_group_stride, q.ddelta_batch_stride)
            and states(p.B, p.B_state_stride, p.B_group_stride, p.B_batch_stride)
            and states(p.C, p.C_state_stride, p.C_group_stride, p.C_batch_stride)
            and states(q.dB, q.dB_state_stride, q.dB_group_stride, q.dB_batch_stride)
            and states(q.dC, q.dC_state_stride, q.dC_group_stride, q.dC_batch_stride))


def _v1_tma_fwd_ok(p, env):
    if env.get("B200_SSCAN_TMA") != "1" or p.io_dtype != 0 or p.n_groups % p.u_group_div:
        return False
    bc = lambda ptr, *s: ptr % 16 == 0 and all(x % 4 == 0 for x in s)
    if not (bc(p.B, p.B_state_stride, p.B_batch_stride, p.B_group_stride) and bc(p.C, p.C_state_stride, p.C_batch_stride, p.C_group_stride)):
        return False
    return (_row_map_ok(p.u, p.seqlen, p.u_row_stride, p.u_group_stride, p.u_batch_stride)
            and _row_map_ok(p.delta, p.seqlen, p.delta_row_stride, p.delta_group_stride, p.delta_batch_stride))


def _v1_tma_bwd_ok(q, env):
    return (_v1_tma_fwd_ok(q.f, env) and q.f.n_groups % q.dout_group_div == 0
            and _row_map_ok(q.dout, q.f.seqlen, q.dout_row_stride, q.dout_group_stride, q.dout_batch_stride))


def _v1_vec(p, *tensors):   # can_vectorize for every staged tensor: 16-byte (fp32) / 8-byte (16-bit) cp.async staging
    align = 16 if p.io_dtype == 0 else 8
    return p.seqlen % 4 == 0 and all(ptr % align == 0 and all(s % 4 == 0 for s in st) for ptr, st in tensors)


def expected_fwd(p, env):
    """(variant, staging) the forward must take: staging is 'tma', 'vec' or 'elem' for sscan.cu, '' for sscan2.cu."""
    if _v2_fwd_ok(p, env):
        return 2, ""
    if _v1_tma_fwd_ok(p, env):
        return 3, "tma"
    vec = _v1_vec(p, (p.u, (p.u_row_stride, p.u_batch_stride, p.u_group_stride)),
                  (p.delta, (p.delta_row_stride, p.delta_batch_stride, p.delta_group_stride)),
                  (p.B, (p.B_state_stride, p.B_batch_stride, p.B_group_stride)), (p.C, (p.C_state_stride, p.C_batch_stride, p.C_group_stride)))
    return 1, "vec" if vec else "elem"


def expected_bwd(q, env):
    if _v2_bwd_ok(q, env):
        return 2, ""
    if _v1_tma_bwd_ok(q, env):
        return 3, "tma"
    p = q.f
    vec = _v1_vec(p, (p.u, (p.u_row_stride, p.u_batch_stride, p.u_group_stride)),
                  (p.delta, (p.delta_row_stride, p.delta_batch_stride, p.delta_group_stride)),
                  (q.dout, (q.dout_row_stride, q.dout_batch_stride, q.dout_group_stride)),
                  (p.B, (p.B_state_stride, p.B_batch_stride, p.B_group_stride)), (p.C, (p.C_state_stride, p.C_batch_stride, p.C_group_stride)))
    return 1, "vec" if vec else "elem"


def kernel_name(direction, variant, staging, c):
    """The kernel instantiation a call ran, for the coverage census."""
    sp, z = int(c.softplus), int(c.has_z)
    if variant == 2:
        return f"sscan_fwd2_kernel<z={z},softplus={sp}>" if direction == "fwd" else f"sscan_bwd2_kernel<softplus={sp}>"
    T = {"f32": "float", "bf16": "bf16", "fp16": "half"}[c.dtype]
    return f"sscan_{direction}_kernel<{T},z={z},tma={int(variant == 3)}>/{staging}"


# ---------------------------------------------------------------------------------------------------------------------
# child: run every case under this process's environment, write one .npz
# ---------------------------------------------------------------------------------------------------------------------
class Arena:
    """A flat buffer prefilled with a NaN payload; views cut from it are recorded so everything else can be checked afterwards."""

    def __init__(self, numel, dtype, dev):
        import torch
        self.torch = torch
        self.buf = torch.empty(numel, dtype=dtype, device=dev)
        self.ibits = torch.int32 if dtype == torch.float32 else torch.int16
        self.sent = SENT32 if dtype == torch.float32 else SENT16
        self.buf.view(self.ibits).fill_(self.sent)
        self.mask = torch.zeros(numel, dtype=torch.bool, device=dev)

    def view(self, shape, strides, offset, zero=False):
        v = self.buf.as_strided(shape, strides, offset)
        self.mask.as_strided(shape, strides, offset).fill_(True)
        if zero:
            v.zero_()
        return v

    def changed_outside(self):
        return int(((self.buf.view(self.ibits) != self.sent) & ~self.mask).sum().item())


def _pitch(L):
    return (L + 8, 8) if L % 4 == 0 else (L + 3, 5)   # (row pitch, gap): multiples of 4 keep 16-byte alignment


def _rows_out(c, rows, dtype, dev, off=0):
    """(batch, rows, L) output in a NaN arena: pitch > L, a gap after every batch, `off` elements from the arena's start."""
    P, gap = _pitch(c.L)
    bs = rows * P + gap
    a = Arena(off + c.batch * bs + gap, dtype, dev)
    return a, a.view((c.batch, rows, c.L), (bs, P, 1), off)


def _padded_in(arr, dtype, dev, pitch=None):
    """A (..., L) input copied into a NaN-padded buffer of row pitch `pitch` (default: L + 4 or L + 1)."""
    import torch
    L = arr.shape[-1]
    P = pitch or (L + 4 if L % 4 == 0 else L + 1)
    buf = torch.full(arr.shape[:-1] + (P,), float("nan"), dtype=dtype, device=dev)
    buf[..., :L] = torch.tensor(arr).to(dtype)
    return buf[..., :L]


def _build_inputs(c, x, dtype, dev):
    """u (3-D or a 4-D (batch, Gu, rows, L) view), delta, B, C (4-D), z, dout in the case's layout."""
    import torch
    T = lambda a: torch.tensor(a, device=dev).to(dtype).contiguous()
    b, L, N, G, rpg = c.batch, c.L, c.N, c.G, c.rows
    Gu = G // c.ugd
    z = T(x["z"]) if c.has_z else None
    if c.layout == "contig":
        return T(x["u"]), T(x["delta"]), T(x["B"]), T(x["C"]), z, T(x["dout"])
    if c.layout == "pad":
        return (_padded_in(x["u"], dtype, dev), _padded_in(x["delta"], dtype, dev), _padded_in(x["B"], dtype, dev),
                _padded_in(x["C"], dtype, dev), None if z is None else _padded_in(x["z"], dtype, dev), _padded_in(x["dout"], dtype, dev))
    if c.layout == "ugroup":   # x2 (Gu, rows, batch, P) -> permute(2, 0, 1, 3): u with a group stride
        P = L + 4 if L % 4 == 0 else L + 1
        x2 = torch.full((Gu, rpg, b, P), float("nan"), dtype=dtype, device=dev)
        x2[..., :L] = torch.tensor(x["u"]).view(b, Gu, rpg, L).permute(1, 2, 0, 3).to(dtype)
        u = x2.permute(2, 0, 1, 3)[..., :L]
        return u, _padded_in(x["delta"], dtype, dev), _padded_in(x["B"], dtype, dev), _padded_in(x["C"], dtype, dev), z, T(x["dout"])
    if c.layout in ("proj", "proj_odd"):   # one projection buffer (batch, G, R + 2N + rows, P): B, C, delta are slices of it
        R, P = (4, L + 4 if L % 4 == 0 else L + 1) if c.layout == "proj" else (3, L)
        proj = torch.full((b, G, R + 2 * N + rpg, P), float("nan"), dtype=dtype, device=dev)
        proj[:, :, R:R + N, :L] = torch.tensor(x["B"]).to(dtype)
        proj[:, :, R + N:R + 2 * N, :L] = torch.tensor(x["C"]).to(dtype)
        proj[:, :, R + 2 * N:, :L] = torch.tensor(x["delta"]).view(b, G, rpg, L).to(dtype)
        return (T(x["u"]), proj[:, :, R + 2 * N:, :L], proj[:, :, R:R + N, :L], proj[:, :, R + N:R + 2 * N, :L], z,
                _padded_in(x["dout"], dtype, dev))
    raise AssertionError(c.layout)


def _run_abi(c, x, env, lib, dev):
    import torch
    from medical_image_classification_b200 import _lib
    from medical_image_classification_b200.selective_scan_interface import _fill_fwd, _row_strides
    dtype = {"f32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[c.dtype]
    b, L, N, G, rpg, dim = c.batch, c.L, c.N, c.G, c.rows, c.dim
    T32 = lambda a: None if a is None else torch.tensor(a, device=dev).float().contiguous()
    A32, D32, bias32 = T32(x["A"]), T32(x["D"]), T32(x["bias"])
    arenas = {}
    if c.layout == "ss2d":   # the exact SS2DCoreFn launch (cross.py): x2 (2, D, B, Lp), big (2, 2M, B*Lp), g_big like big
        M = 2 * N + rpg
        x2 = torch.zeros((2, rpg, b, L), dtype=dtype, device=dev)
        x2[...] = torch.tensor(x["u"]).view(b, 2, rpg, L).permute(1, 2, 0, 3).to(dtype)
        big = torch.empty((2, 2 * M, b * L), dtype=dtype, device=dev)
        big4 = big.view(4, M, b, L).permute(2, 0, 1, 3)
        big4[:, :, :N] = torch.tensor(x["B"]).to(dtype)
        big4[:, :, N:2 * N] = torch.tensor(x["C"]).to(dtype)
        big4[:, :, 2 * N:] = torch.tensor(x["delta"]).view(b, 4, rpg, L).to(dtype)
        u, delta, Bm, Cm, z = x2.permute(2, 0, 1, 3), big4[:, :, 2 * N:], big4[:, :, :N], big4[:, :, N:2 * N], None
        dout = torch.tensor(x["dout"], device=dev).to(dtype).contiguous()
    else:
        u, delta, Bm, Cm, z, dout = _build_inputs(c, x, dtype, dev)

    # ---- forward ----
    arenas["out"], out = _rows_out(c, dim, dtype, dev, off=c.out_off)
    last = torch.full((b, dim, N), float("nan"), device=dev) if c.last else None
    ckpt = torch.empty(lib.b200_sscan_ckpt_bytes(b, dim, L, N, G, CKPT_EVERY) // 4, dtype=torch.float32, device=dev)
    p = _lib.SScanFwdParams()
    _fill_fwd(p, u, delta, A32, Bm, Cm, D32, z, bias32, c.softplus, c.rev, c.ugd)
    p.ckpt_every = CKPT_EVERY
    p.out_batch_stride, p.out_row_stride = out.stride(0), out.stride(1)
    p.out, p.last_state, p.ckpt = out.data_ptr(), _lib.ptr(last), ckpt.data_ptr()
    exp_f = expected_fwd(p, env)
    _lib.check(lib.b200_sscan_fwd(ctypes.byref(p), _lib.stream_ptr(dev)), "b200_sscan_fwd")
    var_f = lib.b200_sscan_last_variant()

    # ---- backward ----
    if c.grads == "gbig" or c.layout == "ss2d":   # ddelta / dB / dC as views of one wider buffer (batch, G, M', P)
        if c.layout == "ss2d":   # g_big exactly as SS2DCoreFn.backward lays it out: M' = 2N + rows, pitch Lp
            Mg, P, rB, rC, rD = 2 * N + rpg, L, 0, N, 2 * N
            g_big = Arena(2 * 2 * Mg * b * L, dtype, dev)
            st = (P, Mg * b * P, b * P, 1)   # (batch, group, row, l) strides of g_big.view(4, M, B, Lp).permute(2, 0, 1, 3)
        else:                    # gap rows between the three blocks, row pitch > L
            Mg, (P, _) = 2 * N + rpg + 3, _pitch(L)
            rB, rC, rD = 0, N + 1, 2 * N + 3
            g_big = Arena(b * G * Mg * P + 8, dtype, dev)
            st = (G * Mg * P, Mg * P, P, 1)
        dB = g_big.view((b, G, N, L), st, rB * st[2], zero=True)
        dC = g_big.view((b, G, N, L), st, rC * st[2], zero=True)
        ddelta = g_big.view((b, G, rpg, L), st, rD * st[2])
        arenas["g_big"] = g_big
        if dtype != torch.float32:
            raise AssertionError("dB / dC are fp32 accumulators: the g_big form needs fp32 I/O")
    else:
        P, gap = _pitch(L)
        gs = rpg * P + gap
        bs = G * gs + gap
        arenas["ddelta"] = Arena(b * bs + gap, dtype, dev)
        ddelta = arenas["ddelta"].view((b, G, rpg, L), (bs, gs, P, 1), 0)
        sgs, sbs = N * P + gap, G * (N * P + gap) + gap
        arenas["dB"], arenas["dC"] = Arena(b * sbs + gap, torch.float32, dev), Arena(b * sbs + gap, torch.float32, dev)
        dB = arenas["dB"].view((b, G, N, L), (sbs, sgs, P, 1), 0, zero=True)
        dC = arenas["dC"].view((b, G, N, L), (sbs, sgs, P, 1), 0, zero=True)
    if c.layout == "ss2d":
        du = torch.empty((b, dim, L), dtype=dtype, device=dev)   # launch_bwd's own du
    else:
        arenas["du"], du = _rows_out(c, dim, dtype, dev)
    dz = None
    if c.has_z:
        arenas["dz"], dz = _rows_out(c, dim, dtype, dev)
    dA = torch.zeros((dim, N), dtype=torch.float32, device=dev)
    dD = torch.zeros(dim, dtype=torch.float32, device=dev) if c.has_D else None
    dbias = torch.zeros(dim, dtype=torch.float32, device=dev) if c.has_bias else None
    q = _lib.SScanBwdParams()
    _fill_fwd(q.f, u, delta, A32, Bm, Cm, D32, z, bias32, c.softplus, c.rev, c.ugd)
    q.f.ckpt_every = CKPT_EVERY
    q.f.ckpt = ckpt.data_ptr()
    q.dout_batch_stride, q.dout_row_stride = dout.stride(0), dout.stride(1)
    q.dout_group_stride, q.dout_group_div = rpg * dout.stride(1), c.dgd
    q.du_batch_stride, q.du_row_stride = du.stride(0), du.stride(1)
    q.ddelta_batch_stride, q.ddelta_group_stride, q.ddelta_row_stride = _row_strides(ddelta, rpg)
    q.dB_batch_stride, q.dB_group_stride, q.dB_state_stride = dB.stride(0), dB.stride(1), dB.stride(2)
    q.dC_batch_stride, q.dC_group_stride, q.dC_state_stride = dC.stride(0), dC.stride(1), dC.stride(2)
    if dz is not None:
        q.dz_batch_stride, q.dz_row_stride = dz.stride(0), dz.stride(1)
    q.dout, q.du, q.ddelta, q.dz = dout.data_ptr(), du.data_ptr(), ddelta.data_ptr(), _lib.ptr(dz)
    q.dA, q.dB, q.dC, q.dD, q.ddelta_bias = dA.data_ptr(), dB.data_ptr(), dC.data_ptr(), _lib.ptr(dD), _lib.ptr(dbias)
    exp_b = expected_bwd(q, env)
    _lib.check(lib.b200_sscan_bwd(ctypes.byref(q), _lib.stream_ptr(dev)), "b200_sscan_bwd")
    var_b = lib.b200_sscan_last_variant()
    torch.cuda.synchronize()

    npy = lambda t: None if t is None else t.detach().float().cpu().numpy()
    res = dict(out=npy(out), last_state=npy(last), du=npy(du), ddelta=npy(ddelta).reshape(b, dim, L), dA=npy(dA),
               dB=npy(dB), dC=npy(dC), dD=npy(dD), ddelta_bias=npy(dbias), dz=npy(dz))
    for k, a in arenas.items():
        res[f"outside_{k}"] = np.array(a.changed_outside())
    res.update(var_f=np.array(var_f), var_b=np.array(var_b), exp_f=np.array([exp_f[0]]), exp_b=np.array([exp_b[0]]),
               stage_f=np.array(exp_f[1]), stage_b=np.array(exp_b[1]))
    return res


def _run_fn(c, x, env, lib, dev):
    """selective_scan_fn with dstate > 16: ceil(N / 16) calls on 16-state slices.  The backward runs on this thread
    (autograd multithreading off) so b200_sscan_last_variant() sees it."""
    import torch
    from medical_image_classification_b200 import _lib
    from medical_image_classification_b200.selective_scan_interface import _fill_fwd, selective_scan_fn
    T = lambda a: None if a is None else torch.tensor(a, device=dev).requires_grad_(True)
    u, delta, A, Bm, Cm, D, z, bias = (T(x[k]) for k in ("u", "delta", "A", "B", "C", "D", "z", "bias"))
    with torch.autograd.set_multithreading_enabled(False):
        out, last = selective_scan_fn(u, delta, A, Bm, Cm, D, z=z, delta_bias=bias, delta_softplus=c.softplus, return_last_state=True)
        var_f = lib.b200_sscan_last_variant()
        out.backward(torch.tensor(x["dout"], device=dev))
        var_b = lib.b200_sscan_last_variant()
    torch.cuda.synchronize()
    # every slice's call, restated with the tensors SelectiveScanFn hands to the C ABI (fresh, contiguous outputs)
    exp_f, exp_b = set(), set()
    b, dim, L = c.batch, c.dim, c.L
    for n0 in range(0, c.N, 16):
        n = min(16, c.N - n0)
        Bs, Cs = Bm.detach().narrow(2, n0, n), Cm.detach().narrow(2, n0, n)
        p = _lib.SScanFwdParams()
        A32 = A.detach()[:, n0:n0 + n].contiguous()
        _fill_fwd(p, u.detach(), delta.detach(), A32, Bs, Cs, None, None, bias.detach(), c.softplus, 0, 1)
        p.out, p.out_row_stride, p.out_batch_stride = 256, L, dim * L
        exp_f.add(expected_fwd(p, env))
        q = _lib.SScanBwdParams()
        q.f = p
        q.dout, q.dout_batch_stride, q.dout_row_stride, q.dout_group_stride, q.dout_group_div = 256, dim * L, L, dim * L, 1
        q.du, q.du_batch_stride, q.du_row_stride = 256, dim * L, L
        q.ddelta, q.ddelta_batch_stride, q.ddelta_group_stride, q.ddelta_row_stride = 256, dim * L, dim * L, L
        q.dB, q.dB_batch_stride, q.dB_group_stride, q.dB_state_stride = 256, n * L, n * L, L
        q.dC, q.dC_batch_stride, q.dC_group_stride, q.dC_state_stride = 256, n * L, n * L, L
        exp_b.add(expected_bwd(q, env))
    assert len({v for v, _ in exp_f}) == 1 and len({v for v, _ in exp_b}) == 1, (exp_f, exp_b)
    (ef, sf), (eb, sb) = sorted(exp_f)[0], sorted(exp_b)[0]
    npy = lambda t: None if t is None else t.detach().float().cpu().numpy()
    return dict(out=npy(out), last_state=npy(last), du=npy(u.grad), ddelta=npy(delta.grad), dA=npy(A.grad), dB=npy(Bm.grad),
                dC=npy(Cm.grad), dD=npy(D.grad), ddelta_bias=npy(bias.grad), dz=npy(z.grad),
                var_f=np.array(var_f), var_b=np.array(var_b), exp_f=np.array([ef]), exp_b=np.array([eb]),
                stage_f=np.array(sf), stage_b=np.array(sb))


def child_main(config, path):
    import torch
    from medical_image_classification_b200 import _lib
    env = {k: os.environ[k] for k in SWITCHES if k in os.environ}
    assert env == CONFIGS[config], (env, CONFIGS[config])
    lib = _lib.load()
    dev = torch.device("cuda:0")
    flat = {}
    for c in CASES:
        x = make_inputs(c, case_seed(c))
        res = (_run_fn if c.api == "fn" else _run_abi)(c, x, env, lib, dev)
        for k, v in res.items():
            if v is not None:
                flat[f"{c.name}/{k}"] = v
    np.savez(path, **flat)


# ---------------------------------------------------------------------------------------------------------------------
# parent: one child per configuration, the oracle once per case
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def runs():
    """config -> {case name -> {key: array}}; a child that fails is reported by every test of its configuration."""
    results = {}
    with tempfile.TemporaryDirectory() as tmp:
        for config, extra in CONFIGS.items():
            env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
            env.update(extra)
            path = os.path.join(tmp, f"{config}.npz")
            r = subprocess.run([sys.executable, os.path.abspath(__file__), config, path], env=env, cwd=ROOT,
                               capture_output=True, text=True, timeout=900)
            if r.returncode != 0:
                results[config] = RuntimeError(f"child for config {config!r} failed (rc={r.returncode}):\n"
                                               f"{r.stdout[-3000:]}\n{r.stderr[-6000:]}")
                continue
            per = {}
            with np.load(path) as z:
                for key in z.files:
                    name, k = key.split("/", 1)
                    per.setdefault(name, {})[k] = z[key]
            results[config] = per
    return results


_ORACLE = {}


def oracle_case(c):
    """fp64 oracle of one case: per group, reversed groups as time flips, shared u / dout rows repeated."""
    if c.name in _ORACLE:
        return _ORACLE[c.name]
    import oracle
    x = make_inputs(c, case_seed(c))
    Lt = c.L_true
    cut = lambda a: None if a is None else np.ascontiguousarray(a[..., :Lt])
    rpg, G = c.rows, c.G
    b, dim, N = c.batch, c.dim, c.N
    if c.api == "fn":
        kw = dict(D=x["D"], z=x.get("z"), delta_bias=x["bias"], delta_softplus=c.softplus, precision="f64")
        out, last = oracle.sscan_fwd(x["u"], x["delta"], x["A"], x["B"], x["C"], **kw)
        gr = oracle.sscan_bwd(x["u"], x["delta"], x["A"], x["B"], x["C"], dout=x["dout"], **kw)
        ref = dict(out=out, last_state=last, **gr)
        _ORACLE[c.name] = ref
        return ref
    ref = dict(out=np.zeros((b, dim, Lt)), last_state=np.zeros((b, dim, N)), du=np.zeros((b, dim, Lt)), ddelta=np.zeros((b, dim, Lt)),
               dA=np.zeros((dim, N)), dB=np.zeros((b, G, N, Lt)), dC=np.zeros((b, G, N, Lt)),
               dD=np.zeros(dim) if c.has_D else None, ddelta_bias=np.zeros(dim) if c.has_bias else None,
               dz=np.zeros((b, dim, Lt)) if c.has_z else None)
    for g in range(G):
        rows = slice(g * rpg, (g + 1) * rpg)
        urows = slice((g // c.ugd) * rpg, (g // c.ugd + 1) * rpg)
        grows = slice((g // c.dgd) * rpg, (g // c.dgd + 1) * rpg)
        rev = (c.rev >> g) & 1
        fl = (lambda a: None if a is None else np.ascontiguousarray(a[..., ::-1])) if rev else (lambda a: a)
        sub = lambda a, s: None if a is None else a[:, s]
        args = [fl(cut(x["u"][:, urows])), fl(cut(x["delta"][:, rows])), x["A"][rows], fl(cut(x["B"][:, g:g + 1])), fl(cut(x["C"][:, g:g + 1]))]
        kw = dict(D=None if x["D"] is None else x["D"][rows], z=fl(cut(sub(x.get("z"), rows))),
                  delta_bias=None if x["bias"] is None else x["bias"][rows], delta_softplus=c.softplus, precision="f64")
        out, last = oracle.sscan_fwd(*args, **kw)
        gr = oracle.sscan_bwd(*args, dout=fl(cut(x["dout"][:, grows])), **kw)
        ref["out"][:, rows] = fl(out)
        ref["last_state"][:, rows] = last
        for k in ("du", "ddelta", "dz"):
            if ref[k] is not None:
                ref[k][:, rows] = fl(gr[k])
        ref["dB"][:, g:g + 1], ref["dC"][:, g:g + 1] = fl(gr["dB"]), fl(gr["dC"])
        ref["dA"][rows] = gr["dA"]
        for k in ("dD", "ddelta_bias"):
            if ref[k] is not None:
                ref[k][rows] = gr[k]
    _ORACLE[c.name] = ref
    return ref


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# element-wise bounds of the reference test (test_selective_scan.py:398-404): (rtol, atol) of out; x2 du / dz, x5 / x10 ddelta,
# x1 / x4 dB and dC
ELEMENTWISE = {"f32": (6e-4, 2e-3), "bf16": (3e-2, 5e-2), "fp16": (3e-3, 5e-3)}
SCALE = {"out": (1, 1), "last_state": (1, 1), "du": (2, 2), "dz": (2, 2), "ddelta": (5, 10), "dB": (1, 4), "dC": (1, 4)}
GRADS = ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dz")


def check_case(c, r, ref):
    """Compare one case's kernel results with the oracle; returns the list of failures (empty when it passes)."""
    fails = []
    Lt = c.L_true
    cut = lambda k, a: a[..., :Lt] if k in ("out", "du", "ddelta", "dB", "dC", "dz") else a
    if c.L_true != c.L:   # SS2DCoreFn's pad steps: zero inputs, zero upstream gradient -> exactly zero gradients
        for k in ("du", "ddelta", "dB", "dC"):
            pad = np.abs(r[k][..., Lt:]).max()
            if pad != 0:
                fails.append(f"{k} at the pad steps is {pad:.3g}, expected 0")
    keys = ["out"] + (["last_state"] if c.last else []) + [k for k in GRADS if ref.get(k) is not None]
    for k in keys:
        if k not in r:
            fails.append(f"{k} missing from the kernel results")
            continue
        a, b = cut(k, r[k]), ref[k]
        if a.shape != b.shape:
            fails.append(f"{k}: shape {a.shape} vs oracle {b.shape}")
            continue
        if not np.isfinite(a).all():
            fails.append(f"{k}: {int((~np.isfinite(a)).sum())} non-finite values")
            continue
        if c.dtype == "f32":
            bound = 1e-5 if k in ("out", "last_state") else 2e-5
            e = relerr(a, b)
            if e >= bound:
                fails.append(f"{k}: norm-wise relative error {e:.3g} >= {bound:g}")
        rtol, atol = ELEMENTWISE[c.dtype]
        if k in SCALE:
            sr, sa = SCALE[k]
            if not np.allclose(a, b, rtol=sr * rtol, atol=sa * atol):
                bad = ~np.isclose(a, b, rtol=sr * rtol, atol=sa * atol)
                fails.append(f"{k}: {int(bad.sum())} elements outside rtol {sr * rtol:g} / atol {sa * atol:g} "
                             f"(max |diff| {np.abs(a - b).max():.3g})")
        elif c.dtype != "f32":   # dA, dD, ddelta_bias of 16-bit I/O (as tests/test_sscan_parity.py::test_low_precision_io)
            if not np.allclose(a, b, rtol=1e-3, atol=5e-3 * max(1.0, float(np.abs(b).max()))):
                fails.append(f"{k}: max |diff| {np.abs(a - b).max():.3g} beyond rtol 1e-3 / atol 5e-3 max|ref|")
    return fails


@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("name", [c.name for c in CASES])
def test_path_matches_oracle(runs, config, name):
    c = CASE_BY_NAME[name]
    per = runs[config]
    if isinstance(per, Exception):
        raise per
    r = per[name]
    var_f, var_b, exp_f, exp_b = int(r["var_f"]), int(r["var_b"]), int(r["exp_f"][0]), int(r["exp_b"][0])
    assert (var_f, var_b) == (exp_f, exp_b), (
        f"[{config}] {c!r}: ran variant fwd {var_f} / bwd {var_b}, the dispatch rules give fwd {exp_f} / bwd {exp_b}")
    outside = {k[len("outside_"):]: int(v) for k, v in r.items() if k.startswith("outside_") and int(v)}
    assert not outside, f"[{config}] {c!r} (fwd {var_f} / bwd {var_b}): elements changed outside the output views: {outside}"
    fails = check_case(c, r, oracle_case(c))
    assert not fails, f"[{config}] {c!r} (fwd {var_f} / bwd {var_b}):\n  " + "\n  ".join(fails)


REQUIRED = (
    [f"sscan_fwd2_kernel<z={z},softplus={s}>" for z in (0, 1) for s in (0, 1)]
    + [f"sscan_bwd2_kernel<softplus={s}>" for s in (0, 1)]
    + [f"sscan_{d}_kernel<float,z={z},tma=1>/tma" for d in ("fwd", "bwd") for z in (0, 1)]
    + [f"sscan_{d}_kernel<float,z={z},tma=0>/{st}" for d in ("fwd", "bwd") for z in (0, 1) for st in ("vec", "elem")]
    + [f"sscan_{d}_kernel<{T},z=1,tma=0>/elem" for d in ("fwd", "bwd") for T in ("bf16", "half")]
)


def test_kernel_census(runs, capsys):
    """Per configuration, how many cases ran on each variant; every kernel instantiation listed in REQUIRED ran at least once."""
    seen = Counter()
    lines = []
    for config, per in runs.items():
        if isinstance(per, Exception):
            raise per
        vf, vb = Counter(), Counter()
        for name, r in per.items():
            c = CASE_BY_NAME[name]
            vf[int(r["var_f"])] += 1
            vb[int(r["var_b"])] += 1
            seen[kernel_name("fwd", int(r["var_f"]), str(r["stage_f"]), c)] += 1
            seen[kernel_name("bwd", int(r["var_b"]), str(r["stage_b"]), c)] += 1
        lines.append(f"  {config:8s} fwd {dict(sorted(vf.items()))}  bwd {dict(sorted(vb.items()))}")
    with capsys.disabled():
        print("\nselective-scan variants per configuration (1 = sscan.cu, 2 = sscan2.cu, 3 = sscan.cu TMA staging):")
        print("\n".join(lines))
        print("kernel instantiations (calls over all configurations):")
        for k in sorted(seen):
            print(f"  {seen[k]:4d}  {k}")
    missing = [k for k in REQUIRED if k not in seen]
    assert not missing, f"kernel instantiations no case reached: {missing}"


if __name__ == "__main__":
    child_main(sys.argv[1], sys.argv[2])
