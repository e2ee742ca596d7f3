"""Gated RMSNorm with groups (csrc/rmsnorm.cu: b200_rmsnorm_fwd / _bwd / _grid) against an fp64 restatement of mamba_ssm's
layernorm_gated.rms_norm_ref (mamba_ssm 2.2.2), through the C ABI with guarded buffers, through RMSNormGated / rmsnorm_fn, and
inside SS2D_with_SSD with ngroups = 2, norm_before_gate = True and D_has_hdim = True against a CPU eager restatement."""
import copy
import ctypes

import pytest
import torch
import torch.nn.functional as F

from medical_image_classification_b200 import _lib

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


def rms_norm_ref(x, weight, bias, z=None, eps=1e-6, group_size=None, norm_before_gate=True):
    """mamba_ssm.ops.triton.layernorm_gated.rms_norm_ref, in the dtype of its arguments (no cast back)."""
    if z is not None and not norm_before_gate:
        x = x * F.silu(z)
    gs = x.shape[-1] if group_size is None else group_size
    xg = x.unflatten(-1, (-1, gs))
    rstd = 1 / torch.sqrt(xg.square().mean(dim=-1, keepdim=True) + eps)
    out = (xg * rstd).flatten(-2) * weight
    if bias is not None:
        out = out + bias
    if z is not None and norm_before_gate:
        out = out * F.silu(z)
    return out


def nrel(a, b):
    """Norm-wise relative error."""
    a, b = a.detach().double().to(b.device), b.detach().double()
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def _oracle(x, z, w, b, dy, eps, gs, nbg):
    """out and gradients of rms_norm_ref in fp64, from the values the kernels read."""
    leaf = lambda t: None if t is None else t.detach().double().requires_grad_()
    xd, zd, wd, bd = leaf(x), leaf(z), leaf(w), leaf(b)
    out = rms_norm_ref(xd, wd, bd, zd, eps, gs, nbg)
    out.backward(dy.double())
    grad = lambda t: None if t is None else t.grad
    return out.detach(), grad(xd), grad(zd), grad(wd), grad(bd)


class Guarded:
    """A (rows, dim) contiguous buffer of `dtype` inside a NaN-filled allocation with `pad` elements on each side; check() requires
    the padding to be bit-for-bit what it was."""

    def __init__(self, rows, dim, dtype, pad=8):
        self.n, self.pad = rows * dim, pad
        self.buf = torch.full((self.n + 2 * pad,), float("nan"), dtype=dtype, device="cuda")
        self.view = self.buf[pad:pad + self.n].view(rows, dim)
        self.before = self.buf.clone()

    def check(self, what):
        ib = {4: torch.int32, 2: torch.int16}[self.buf.element_size()]
        a, b = self.buf.view(ib), self.before.view(ib)
        p = self.pad
        assert torch.equal(a[:p], b[:p]) and torch.equal(a[p + self.n:], b[p + self.n:]), f"{what}: write outside the view"
        assert bool(torch.isfinite(self.view).all()), f"{what}: view not fully written"


def strided(rows, dim, dtype, pitch=None, offset=0, gen=None):
    """(rows, dim) random values of `dtype`, as columns [offset, offset + dim) of a (rows, pitch) tensor when pitch is given."""
    if pitch is None:
        return torch.randn(rows, dim, generator=gen, device="cuda").to(dtype)
    wide = torch.randn(rows, pitch, generator=gen, device="cuda").to(dtype)
    return wide[:, offset:offset + dim]


def run_abi(x, z, w, b, dy, gs, nbg, out_dtype, eps=1e-5, pad=8):
    """One forward and one backward through the C ABI, every output in a NaN-guarded allocation.
    Returns out, rstd, dx, dz, dw, db."""
    rows, dim = x.shape
    ng = dim // gs
    lib = _lib.load()
    dev = x.device
    out, rstd = Guarded(rows, dim, out_dtype, pad), Guarded(rows, ng, F32, pad)
    code = lambda t: _lib.dtype_code(t.dtype) if t is not None else 0
    stride = lambda t: t.stride(0) if t is not None else 0
    _lib.launch("b200_rmsnorm_fwd", dev, x.data_ptr(), code(x), stride(x), _lib.ptr(z), code(z), stride(z), w.data_ptr(), _lib.ptr(b),
                out.view.data_ptr(), _lib.dtype_code(out_dtype), rstd.view.data_ptr(), rows, dim, gs, int(nbg), float(eps))
    grid = lib.b200_rmsnorm_grid(rows, dim, gs)
    assert grid >= 1
    dx = Guarded(rows, dim, x.dtype, pad)
    dz = Guarded(rows, dim, z.dtype, pad) if z is not None else None
    dw = Guarded(grid, dim, F32, pad)
    db = Guarded(grid, dim, F32, pad) if b is not None else None
    _lib.launch("b200_rmsnorm_bwd", dev, dy.data_ptr(), code(dy), stride(dy), x.data_ptr(), code(x), stride(x), _lib.ptr(z), code(z), stride(z),
                w.data_ptr(), _lib.ptr(b), rstd.view.data_ptr(), dx.view.data_ptr(), dz.view.data_ptr() if dz else None, dw.view.data_ptr(),
                db.view.data_ptr() if db else None, rows, dim, gs, int(nbg))
    torch.cuda.synchronize()
    for name, gbuf in (("out", out), ("rstd", rstd), ("dx", dx), ("dz", dz), ("dw", dw), ("db", db)):
        if gbuf is not None:
            gbuf.check(name)
    return (out.view, rstd.view, dx.view, dz.view if dz else None, dw.view.sum(0), db.view.sum(0) if db else None)


def _check(x, z, w, b, dy, gs, nbg, out_dtype, eps=1e-5, pad=8):
    got = run_abi(x, z, w, b, dy, gs, nbg, out_dtype, eps, pad)
    out, rstd, dx, dz, dw, db = got
    ro, rdx, rdz, rdw, rdb = _oracle(x, z, w, b, dy, eps, gs, nbg)
    exact = x.dtype == F32 and (z is None or z.dtype == F32) and out_dtype == F32 and dy.dtype == F32
    pairs = [("out", out, ro), ("dx", dx, rdx), ("dw", dw, rdw)] + ([("dz", dz, rdz)] if z is not None else []) \
        + ([("db", db, rdb)] if b is not None else [])
    for name, a, r in pairs:
        if exact:
            assert nrel(a, r) <= 1e-5, (name, nrel(a, r))
        else:
            assert torch.allclose(a.double(), r, rtol=3e-2, atol=5e-2), (name, float((a.double() - r).abs().max()))
    return got


def _params(dim, gen, bias):
    w = (0.5 + torch.rand(dim, generator=gen, device="cuda")).contiguous()
    b = (0.1 * torch.randn(dim, generator=gen, device="cuda")) if bias else None
    return w, b


# ---- the C ABI over the shape / mode matrix, fp32 --------------------------------------------------------------------------------
SHAPES = [(96, 96), (96, 48), (96, 12), (96, 3), (128, 128), (128, 64), (128, 16), (1024, 1024), (1024, 512), (1024, 128),
          (135, 135), (135, 45), (135, 5), (6144, 6144), (6144, 3072), (6144, 768)]


@pytest.mark.gpu
@pytest.mark.parametrize("dim,gs", SHAPES)
def test_fp32_modes_match_reference(dim, gs):
    """norm_before_gate in {0, 1} x z present / absent x bias present / absent, fp32 everywhere, contiguous and strided z / dy."""
    gen = torch.Generator(device="cuda").manual_seed(dim * 7 + gs)
    rows = 37
    for nbg in (0, 1):
        for has_z in (True, False):
            for bias in (False, True):
                x = strided(rows, dim, F32, gen=gen)
                z = strided(rows, dim, F32, pitch=dim + 3, offset=1, gen=gen) if has_z else None
                dy = strided(rows, dim, F32, pitch=dim + 5, offset=2, gen=gen) if bias else strided(rows, dim, F32, gen=gen)
                w, b = _params(dim, gen, bias)
                _check(x, z, w, b, dy, gs, nbg, F32)


# ---- mixed 16-bit dtypes, unaligned pitches ---------------------------------------------------------------------------------------
DTYPE_SETS = [  # x, z, out, dy
    (F32, BF16, BF16, BF16), (F32, BF16, F32, F32), (BF16, BF16, BF16, BF16), (F16, F16, F16, F16), (F16, BF16, F32, F16),
    (BF16, F16, F16, F32), (F32, F16, BF16, BF16), (BF16, F32, F32, BF16)]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", DTYPE_SETS, ids=["-".join(str(t)[6:] for t in s) for s in DTYPE_SETS])
@pytest.mark.parametrize("dim,gs", [(128, 128), (96, 48), (135, 45), (1024, 256), (6144, 3072)])
def test_mixed_dtypes_and_pitches(dt, dim, gs):
    """z and dy as column slices of a wider tensor: pitch 514 (4-byte rows for 16-bit data) and an odd element offset (2-byte
    rows), output buffers unaligned too; oracle on the values the kernel read, bars of the reference's bf16 tests."""
    tx, tz, to, tdy = dt
    gen = torch.Generator(device="cuda").manual_seed(dim + gs)
    rows = 53
    pitch = max(514, dim + 8)
    for nbg in (0, 1):
        for offset, pad in ((0, 8), (1, 1)):
            x = strided(rows, dim, tx, gen=gen)
            z = strided(rows, dim, tz, pitch=pitch, offset=offset, gen=gen)
            dy = strided(rows, dim, tdy, pitch=pitch, offset=offset, gen=gen)
            w, b = _params(dim, gen, nbg == 1)
            _check(x, z, w, b, dy, gs, nbg, to, pad=pad)
        x = strided(rows, dim, tx, pitch=pitch, offset=1, gen=gen)          # no gate: x strided
        w, b = _params(dim, gen, True)
        _check(x, None, w, b, strided(rows, dim, tdy, gen=gen), gs, nbg, to)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,dim", [(1, 128), (200704, 128), (50176, 256), (12544, 512), (3136, 1024)])
def test_medssd_shapes(rows, dim):
    """MedSSD's four stage shapes at batch 64 (and one row) as SS2D_with_SSD runs them under bf16 autocast: fp32 x from the
    cross-merge, bf16 z read in place from in_proj's output (row pitch 2 d_inner + 2 G N + nheads = 514 at stage 0),
    bf16 out and dy; then the same in fp32."""
    gen = torch.Generator(device="cuda").manual_seed(rows)
    pitch = 2 * dim + 2 * 128 + dim // 64                      # d_state 128, one group, headdim 64
    x = strided(rows, dim, F32, gen=gen)
    z = strided(rows, dim, BF16, pitch=pitch, gen=gen)
    dy = strided(rows, dim, BF16, gen=gen)
    w, _ = _params(dim, gen, False)
    _check(x, z, w, None, dy, dim, 0, BF16)
    _check(x, z.float(), w, None, dy.float(), dim, 0, F32)


@pytest.mark.gpu
def test_default_path_matches_rmsnorm_gated():
    """One group, norm after the gate, fp32 contiguous: the new entry points agree with b200_rmsnorm_gated_fwd / _bwd to a
    couple of ulp (the two kernels sum the row in different orders); dw also differs by the order of its row reduction."""
    gen = torch.Generator(device="cuda").manual_seed(5)
    rows, dim = 4099, 768
    x, z, dy = (strided(rows, dim, F32, gen=gen) for _ in range(3))
    w, _ = _params(dim, gen, False)
    out, rstd, dx, dz, dw, _ = run_abi(x, z, w, None, dy, dim, 0, F32)
    y0, r0 = torch.empty_like(x), torch.empty(rows, device="cuda")
    dx0, dz0 = torch.empty_like(x), torch.empty_like(x)
    nblk = min(rows, 592)
    dwp0 = torch.empty(nblk, dim, device="cuda")
    _lib.launch("b200_rmsnorm_gated_fwd", x.device, x.data_ptr(), z.data_ptr(), w.data_ptr(), y0.data_ptr(), r0.data_ptr(), rows, dim,
                1e-5)
    _lib.launch("b200_rmsnorm_gated_bwd", x.device, x.data_ptr(), z.data_ptr(), w.data_ptr(), r0.data_ptr(), dy.data_ptr(), dx0.data_ptr(),
                dz0.data_ptr(), dwp0.data_ptr(), nblk, rows, dim)
    ulp2 = 2 * 2.0 ** -23
    assert nrel(out, y0) <= ulp2 and nrel(rstd[:, 0], r0) <= ulp2
    assert nrel(dx, dx0) <= ulp2 and nrel(dz, dz0) <= ulp2
    assert nrel(dw, dwp0.sum(0)) <= 1e-6


# ---- modules --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("gs,nbg,gated", [(None, False, True), (32, False, True), (64, True, True), (16, True, False), (None, True, False)])
def test_rmsnorm_gated_module(gs, nbg, gated):
    from medical_image_classification_b200.ssd_combined import RMSNormGated
    torch.manual_seed(1)
    m = RMSNormGated(128, group_size=gs, norm_before_gate=nbg).cuda()
    with torch.no_grad():
        m.weight.uniform_(0.5, 1.5)
    x = torch.randn(2, 5, 7, 128, device="cuda", requires_grad=True)
    z = torch.randn(2, 5, 7, 128, device="cuda", requires_grad=True) if gated else None
    y = m(x, z)
    assert y.dtype == x.dtype and y.shape == x.shape
    g = torch.randn_like(y)
    y.backward(g)
    ro, rdx, rdz, rdw, _ = _oracle(x, z, m.weight, None, g, 1e-5, gs, nbg)
    assert nrel(y, ro) <= 1e-5 and nrel(x.grad, rdx) <= 1e-5 and nrel(m.weight.grad, rdw) <= 1e-5
    if gated:
        assert nrel(z.grad, rdz) <= 1e-5


@pytest.mark.gpu
def test_rmsnorm_fn_bf16_with_bias():
    """rmsnorm_fn with mamba_ssm's defaults (eps 1e-6, norm_before_gate=True): output and gradients in the primals' dtypes."""
    from medical_image_classification_b200.ssd_combined import rmsnorm_fn
    torch.manual_seed(2)
    x = torch.randn(300, 256, device="cuda", dtype=BF16, requires_grad=True)
    zxb = torch.randn(300, 600, device="cuda", dtype=BF16)
    z = zxb[:, 3:259].requires_grad_()
    w = (0.5 + torch.rand(256, device="cuda")).requires_grad_()
    b = (0.1 * torch.randn(256, device="cuda")).requires_grad_()
    y = rmsnorm_fn(x, w, b, z=z, group_size=64)
    assert y.dtype == BF16
    g = torch.randn_like(y)
    y.backward(g)
    assert x.grad.dtype == BF16 and z.grad.dtype == BF16 and w.grad.dtype == F32
    ro, rdx, rdz, rdw, rdb = _oracle(x, z, w, b, g, 1e-6, 64, True)
    for a, r in ((y, ro), (x.grad, rdx), (z.grad, rdz), (w.grad, rdw), (b.grad, rdb)):
        assert torch.allclose(a.double(), r, rtol=3e-2, atol=5e-2)


# ---- SS2D_with_SSD with the generalised norm against a CPU eager restatement ------------------------------------------------------
def _cpu_ss2d_ssd_forward(self, u, seqlen=None, seq_idx=None, cu_seqlens=None):
    """oracle/cpu_path.CpuSS2DWithSSD's data flow (reference SSD/MedSSD.py:310-402) with D of shape (H, P) when D_has_hdim and
    the norm of mamba_ssm's rms_norm_ref (group_size = d_ssm / ngroups, either order of norm and gate)."""
    from oracle.cpu_path import OracleSsdFn
    B, H, W, C = u.shape
    L, K = H * W, 4
    zxbcdt = self.in_proj(u)
    d_mlp = (zxbcdt.shape[-1] - 2 * self.d_ssm - 2 * self.ngroups * self.d_state - self.nheads) // 2
    z0, x0, z, xBCdt = torch.split(
        zxbcdt, [d_mlp, d_mlp, self.d_ssm, self.d_ssm + 2 * self.ngroups * self.d_state + self.nheads], dim=-1)
    xBCdt = self.act(self.conv2d(xBCdt.permute(0, 3, 1, 2).contiguous()))
    gn = self.ngroups * self.d_state
    hwwh = torch.stack([xBCdt.reshape(B, -1, L), xBCdt.transpose(2, 3).reshape(B, -1, L)], dim=1)
    xBCdts = torch.cat([hwwh, hwwh.flip(-1)], dim=1)
    xs, Bs, Cs, dts = torch.split(xBCdts, [self.d_ssm, gn, gn, self.nheads], dim=2)
    xs = xs.float().reshape(B, -1, L).permute(0, 2, 1).unflatten(2, (-1, self.headdim))
    Bs = Bs.float().reshape(B, -1, L).permute(0, 2, 1).unflatten(2, (self.ngroups, -1))
    Cs = Cs.float().reshape(B, -1, L).permute(0, 2, 1).unflatten(2, (self.ngroups, -1))
    dts = dts.float().reshape(B, -1, L).permute(0, 2, 1)
    As = -torch.exp(self.A_logs.float())
    Ds = self.Ds.float().view(-1, self.headdim) if self.D_has_hdim else self.Ds.float()
    y = OracleSsdFn.apply(xs.contiguous(), dts.contiguous(), As, Bs.contiguous(), Cs.contiguous(), Ds,
                          self.dt_bias.view(-1).float(), True)
    y = y.reshape(B, L, K, -1)
    inv_y = y[:, :, 2:4].flip(1)
    wh_y = y[:, :, 1].view(B, W, H, -1).transpose(1, 2).reshape(B, L, -1)
    invwh_y = inv_y[:, :, 1].view(B, W, H, -1).transpose(1, 2).reshape(B, L, -1)
    out = (y[:, :, 0] + inv_y[:, :, 0] + wh_y + invwh_y).view(B, H, W, -1)
    out = rms_norm_ref(out, self.norm.weight, None, z, self.norm.eps, self.d_ssm // self.ngroups, self.norm_before_gate)
    if d_mlp > 0:
        out = torch.cat([F.silu(z0) * x0, out], dim=-1)
    out = self.out_proj(out)
    return self.dropout(out) if self.dropout is not None else out


def _cpu_twin(model):
    from medical_image_classification_b200.models import SS_Conv_SSD
    from medical_image_classification_b200.ss2d_ssd import SS2D_with_SSD
    from oracle.cpu_path import CpuSSConvSSD

    class CpuSS2DWithSSDGeneral(SS2D_with_SSD):
        forward = _cpu_ss2d_ssd_forward

    twin = copy.deepcopy(model)
    for mod in twin.modules():
        if type(mod) is SS2D_with_SSD:
            mod.__class__ = CpuSS2DWithSSDGeneral
        elif type(mod) is SS_Conv_SSD:
            mod.__class__ = CpuSSConvSSD
    return twin


def _max_rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(ngroups=2), dict(norm_before_gate=True), dict(D_has_hdim=True),
                                dict(ngroups=2, norm_before_gate=True, D_has_hdim=True)],
                         ids=["ngroups2", "norm_before_gate", "D_has_hdim", "all"])
def test_ss2d_with_ssd_generalised_norm(kw):
    from medical_image_classification_b200.ss2d_ssd import SS2D_with_SSD
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(3)
    m = SS2D_with_SSD(d_model=32, d_state=8, headdim=16, chunk_size=32, **kw)
    with torch.no_grad():
        m.norm.weight.uniform_(0.5, 1.5)
        m.Ds.uniform_(0.5, 1.5)
    cpu = _cpu_twin(m)
    x = torch.randn(2, 7, 5, 32)
    g = torch.randn(2, 7, 5, 32)
    xc = x.clone().requires_grad_()
    ref = cpu(xc)
    ref.backward(g)
    m = m.cuda()
    xg = x.cuda().requires_grad_()
    out = m(xg)
    out.backward(g.cuda())
    assert _max_rel(out, ref) < 2e-5
    assert _max_rel(xg.grad, xc.grad) < 5e-5
    cp = dict(cpu.named_parameters())
    for k, p in m.named_parameters():
        assert _max_rel(p.grad, cp[k].grad) < 2e-4, k


@pytest.mark.gpu
def test_two_ss_conv_ssd_blocks_ngroups2_bf16_autocast():
    """Two SS_Conv_SSD blocks whose mixers are SS2D_with_SSD(ngroups=2), under bf16 autocast against their fp32 CPU twin, with
    the bars of the MedSSD bf16 autocast test: output within 5e-2 of its largest magnitude, global gradient cosine >= 0.99."""
    from medical_image_classification_b200.models import SS_Conv_SSD
    torch.manual_seed(4)
    net = torch.nn.Sequential(*(SS_Conv_SSD(hidden_dim=64, d_state=8, ngroups=2, chunk_size=64) for _ in range(2)))
    for blk in net:
        assert blk.self_attention.ngroups == 2 and blk.self_attention.norm.group_size == 32
    cpu = _cpu_twin(net)
    x = torch.randn(2, 8, 8, 64)
    xc = x.clone().requires_grad_()
    ref = cpu(xc)
    g = torch.randn_like(ref)
    ref.backward(g)
    net = net.cuda()
    xg = x.cuda().requires_grad_()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = net(xg)
    out.float().backward(g.cuda())
    assert _max_rel(out, ref) < 5e-2
    cp = dict(cpu.named_parameters())
    num = den_a = den_b = 0.0
    for k, p in net.named_parameters():
        a, b = p.grad.double().cpu().ravel(), cp[k].grad.double().ravel()
        num += float(a @ b); den_a += float(a @ a); den_b += float(b @ b)
    assert num / (den_a * den_b) ** 0.5 >= 0.99


# ---- CPU: argument checks, compat ----------------------------------------------------------------------------------------------
def test_error_returns_without_launching():
    lib = _lib.load()
    fake = ctypes.c_void_p(256)
    before = lib.b200_kernel_launches()
    fwd = lambda x, rows, dim, gs: lib.b200_rmsnorm_fwd(x, 0, dim, None, 0, 0, fake, None, fake, 0, fake, rows, dim, gs, 0, 1e-5, None)
    assert fwd(fake, 4, 96, 40) < 0 and b"does not divide" in lib.b200_last_error()
    assert fwd(fake, 4, 96, 0) < 0
    assert fwd(fake, 4, 8200, 8200) < 0 and b"dim" in lib.b200_last_error()
    assert fwd(None, 4, 96, 96) < 0 and b"NULL" in lib.b200_last_error()
    assert lib.b200_rmsnorm_fwd(fake, 5, 96, None, 0, 0, fake, None, fake, 0, fake, 4, 96, 96, 0, 1e-5, None) < 0   # bad dtype
    assert lib.b200_rmsnorm_bwd(fake, 0, 96, fake, 0, 96, fake, 0, 96, fake, None, fake, fake, None, fake, None, 4, 96, 96, 0, None) < 0
    assert b"dz" in lib.b200_last_error()
    assert lib.b200_rmsnorm_bwd(fake, 0, 96, fake, 0, 96, None, 0, 0, fake, None, fake, fake, None, None, None, 4, 96, 96, 0, None) < 0
    assert lib.b200_rmsnorm_grid(4, 96, 7) < 0 and lib.b200_rmsnorm_grid(4, 0, 1) < 0
    assert lib.b200_rmsnorm_grid(4, 96, 32) >= 1
    assert lib.b200_kernel_launches() == before


def test_module_argument_checks():
    from medical_image_classification_b200.ssd_combined import RMSNormGated
    with pytest.raises(ValueError, match="does not divide"):
        RMSNormGated(96, group_size=40)
    m = RMSNormGated(96, group_size=32, norm_before_gate=True)
    assert m.bias is None and tuple(m.weight.shape) == (96,) and m.norm_before_gate and m.group_size == 32


def test_compat_resolves_rmsnorm_fn():
    import importlib
    import os
    import sys
    compat = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "compat")
    sys.path.insert(0, compat)
    try:
        lg = importlib.import_module("mamba_ssm.ops.triton.layernorm_gated")
    finally:
        sys.path.remove(compat)
    from medical_image_classification_b200 import ssd_combined
    assert lg.rmsnorm_fn is ssd_combined.rmsnorm_fn and lg.RMSNorm is ssd_combined.RMSNormGated
    import inspect
    params = inspect.signature(lg.rmsnorm_fn).parameters
    assert list(params) == ["x", "weight", "bias", "z", "eps", "group_size", "norm_before_gate"]
    assert params["eps"].default == 1e-6 and params["group_size"].default is None and params["norm_before_gate"].default is True
