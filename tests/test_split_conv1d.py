"""The fused Mamba-2 mixer mamba_split_conv1d_scan_combined and the causal depth-wise conv1d under it (causal_conv1d_fn).

mixer_ref64 restates the operator in float64 from its parts -- F.conv1d + activation, ssd_ref64 (tests/test_ssd_state_ref.py),
rms_norm_ref (tests/test_rmsnorm.py), SwiGLU and F.linear -- and torch.autograd differentiates it.  The CPU tests pin it against
transformers' Mamba2Mixer.torch_forward and its packed-sequence handling against running each sequence alone; the GPU tests check
the kernels against it.

Bars (norm-wise relative error), as in the rest of the suite: 2e-5 for element tensors and 2e-4 for sums over the sequence at the
default precision, 5e-3 / 5e-2 in single-pass TF32; with bf16 zxbcdt, the output at rtol 3e-2 / atol 5e-2 against the
restatement on the bf16-rounded inputs and the gradients norm-wise at 3e-2.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_rmsnorm import nrel, rms_norm_ref
from test_ssd_state_ref import ssd_ref64

INF = float("inf")
ELEM = ("out", "fin", "zxbcdt", "initial_states")


# ---- the float64 restatement ------------------------------------------------------------------------------------------------
def conv_ref(xBC, w, b, seq_idx, silu):
    """act(causal depth-wise conv) of xBC (batch, L, C); with seq_idx a tap counts only when its id equals the output's."""
    W, L = w.shape[1], xBC.shape[1]
    if seq_idx is None:
        o = F.conv1d(xBC.transpose(1, 2), w.unsqueeze(1), b, padding=W - 1, groups=w.shape[0])[..., :L].transpose(1, 2)
    else:
        xp = F.pad(xBC, (0, 0, W - 1, 0))
        sp = F.pad(seq_idx, (W - 1, 0), value=int(seq_idx.min()) - 1)
        o = sum(xp[:, k:k + L] * w[:, k] * (sp[:, k:k + L] == seq_idx).unsqueeze(-1) for k in range(W))
        if b is not None:
            o = o + b
    return F.silu(o) if silu else o


def segments(ids, L):
    """[(start, end, id)] of the runs of one row's ids (one run with id 0 when ids is None)."""
    if ids is None:
        return [(0, L, 0)]
    ids = [int(v) for v in ids]
    out, s = [], 0
    for t in range(1, L + 1):
        if t == L or ids[t] != ids[s]:
            out.append((s, t, ids[s]))
            s = t
    return out


def mixer_ref64(zxbcdt, conv_w, conv_b, dt_bias, A, D, initial_states=None, seq_idx=None, dt_limit=(0.0, INF), activation="silu",
                rmsnorm_weight=None, rmsnorm_eps=1e-6, outproj_weight=None, outproj_bias=None, headdim=None, ngroups=1,
                norm_before_gate=True):
    """(out, final_states, y) of mamba_split_conv1d_scan_combined, y the SSD output before the gate.  The SSD runs on each
    sequence of a packed row alone; initial_states reach a row's first sequence when its id is 0."""
    H = D.shape[0]
    P = D.shape[1] if D.dim() == 2 else headdim
    dim, G = H * P, ngroups
    N = (conv_w.shape[0] - dim) // G // 2
    batch, L, width = zxbcdt.shape
    d_nonssm = (width - 2 * dim - 2 * G * N - H) // 2
    z0, x0, z, xBC, dt = zxbcdt.split([d_nonssm, d_nonssm, dim, dim + 2 * G * N, H], dim=-1)
    xbc = conv_ref(xBC, conv_w, conv_b, seq_idx, activation is not None)
    x, B, C = xbc.split([dim, G * N, G * N], -1)
    x, B, C = x.unflatten(-1, (H, P)), B.unflatten(-1, (G, N)), C.unflatten(-1, (G, N))
    ys, fins = [], []
    for b in range(batch):
        parts = []
        for s, e, sid in segments(None if seq_idx is None else seq_idx[b], L):
            ini = initial_states[b:b + 1] if initial_states is not None and s == 0 and sid == 0 else None
            sl = (slice(b, b + 1), slice(s, e))
            o, f = ssd_ref64(x[sl], dt[sl], A, B[sl], C[sl], None, dt_bias, True, dt_limit, ini)
            parts.append(o)
        ys.append(torch.cat(parts, 1))
        fins.append(f)
    y = torch.cat(ys, 0) + x * (D[:, None] if D.dim() == 1 else D)
    y = y.flatten(2)
    if rmsnorm_weight is None:
        out = y * F.silu(z)
    else:
        out = rms_norm_ref(y, rmsnorm_weight, None, z, rmsnorm_eps, dim // G, norm_before_gate)
    if d_nonssm:
        out = torch.cat([F.silu(z0) * x0, out], -1)
    if outproj_weight is not None:
        out = F.linear(out, outproj_weight, outproj_bias)
    return out, torch.cat(fins, 0), y


# ---- inputs ----------------------------------------------------------------------------------------------------------------
def make(batch, L, H, P, G, N, width=4, d_nonssm=0, bias=True, D_hp=False, rms=True, outproj=None, init=False, seed=0):
    """float64 CPU leaves of one call (None where absent) and the static arguments."""
    gen = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=gen, dtype=torch.float64)
    dim, conv_dim = H * P, H * P + 2 * G * N
    zx = r(batch, L, 2 * d_nonssm + dim + conv_dim + H)
    zx[..., -H:] = zx[..., -H:] * 0.5 - 0.5          # dt before softplus
    t = dict(zxbcdt=zx, conv_w=r(conv_dim, width) * 0.5, conv_b=r(conv_dim) * 0.2 if bias else None,
             dt_bias=torch.rand(H, generator=gen, dtype=torch.float64) * 0.5, A=-0.5 - torch.rand(H, generator=gen, dtype=torch.float64),
             D=r(H, P) if D_hp else r(H), rms_w=1 + 0.2 * r(dim) if rms else None,
             outproj_w=r(24, d_nonssm + dim) / (d_nonssm + dim) ** 0.5 if outproj else None,
             outproj_b=r(24) if outproj == "wb" else None, initial_states=r(batch, H, P, N) if init else None)
    return t, dict(headdim=P, ngroups=G)


def call_args(t, dev, dtype=torch.float64, zx_dtype=None):
    """Leaves on dev: zxbcdt in zx_dtype (default dtype), parameters in dtype."""
    out = {}
    for k, v in t.items():
        if v is None:
            out[k] = None
            continue
        out[k] = v.to(dev, zx_dtype if (k == "zxbcdt" and zx_dtype is not None) else dtype).requires_grad_()
    return out


def run(fn, a, kw, gout=None, gfin=None, **extra):
    """Forward and backward of fn (the operator or mixer_ref64) on leaves a; returns {name: tensor} of outputs and gradients."""
    res = fn(a["zxbcdt"], a["conv_w"], a["conv_b"], a["dt_bias"], a["A"], a["D"], initial_states=a["initial_states"],
             rmsnorm_weight=a["rms_w"], outproj_weight=a["outproj_w"], outproj_bias=a["outproj_b"], **kw, **extra)
    out, fin = (res[0], res[1]) if isinstance(res, tuple) else (res, None)
    loss = (out.double() * gout.to(out.device)).sum()
    if gfin is not None:
        loss = loss + (fin.double() * gfin.to(fin.device)).sum()
    leaves = {k: v for k, v in a.items() if v is not None}
    grads = torch.autograd.grad(loss, list(leaves.values()), allow_unused=True)
    r = {"out": out.detach(), "fin": None if fin is None else fin.detach()}
    r.update({"d" + k: g for k, g in zip(leaves, grads)})
    return r


def op():
    from medical_image_classification_b200.ssd_combined import mamba_split_conv1d_scan_combined
    return mamba_split_conv1d_scan_combined


def ref_call(*args, return_final_states=False, **kw):
    out, fin, _ = mixer_ref64(*args, **kw)
    return (out, fin) if return_final_states else out


def compare(got, want, elem_bar, sum_bar, skip=()):
    errs = {}
    for k, w in want.items():
        if w is None or k in skip or got.get(k) is None:
            continue
        errs[k] = nrel(got[k], w)
    bad = {k: v for k, v in errs.items() if v > (elem_bar if k.lstrip("d") in ELEM else sum_bar)}
    assert not bad, errs
    return errs


def check_case(t, static, chunk, dev="cuda", seq_idx=None, dt_limit=(0.0, INF), activation="silu", nbg=True, with_fin=False,
               elem_bar=2e-5, sum_bar=2e-4, zx_dtype=None, skip=()):
    kw = dict(static, dt_limit=dt_limit, activation=activation, norm_before_gate=nbg, return_final_states=with_fin)
    gen = torch.Generator().manual_seed(99)
    a64 = call_args(t, dev)
    ref0 = mixer_ref64(a64["zxbcdt"], a64["conv_w"], a64["conv_b"], a64["dt_bias"], a64["A"], a64["D"], a64["initial_states"],
                       None if seq_idx is None else seq_idx.to(dev), dt_limit, activation, a64["rms_w"], 1e-6, a64["outproj_w"],
                       a64["outproj_b"], static["headdim"], static["ngroups"], nbg)
    gout = torch.randn(ref0[0].shape, generator=gen, dtype=torch.float64)
    gfin = torch.randn(ref0[1].shape, generator=gen, dtype=torch.float64) if with_fin else None
    sq = None if seq_idx is None else seq_idx.to(dev)
    a = call_args(t, dev, torch.float32, zx_dtype)
    got = run(op(), a, dict(kw, chunk_size=chunk, seq_idx=sq), gout, gfin)
    if zx_dtype is not None:        # the restatement on what the kernels read
        t = dict(t, zxbcdt=t["zxbcdt"].to(zx_dtype).double())
        a64 = call_args(t, dev)
    want = run(ref_call, a64, dict(kw, seq_idx=sq), gout, gfin)
    return compare(got, want, elem_bar, sum_bar, skip), got, want


# ---- CPU: the restatement against transformers and against per-sequence runs ---------------------------------------------------
def test_restatement_matches_transformers_mixer():
    from test_oracle_ssd import _hf_mixer
    L, heads, headdim, dstate, chunk = 45, 4, 8, 12, 16
    mixer = _hf_mixer(L, heads, headdim, 1, dstate, chunk, seed=3)
    with torch.no_grad():
        mixer.norm.weight.copy_(1 + 0.3 * torch.randn(heads * headdim, dtype=torch.float64))
    torch.manual_seed(4)
    hidden = torch.randn(2, L, heads * headdim // 2, dtype=torch.float64)
    cap = {}
    hook = mixer.norm.register_forward_pre_hook(lambda mod, args: cap.update(y=args[0]))     # returns None: args unchanged
    out_hf = mixer.torch_forward(hidden)
    hook.remove()
    zx = mixer.in_proj(hidden)
    kw = dict(conv_b=mixer.conv1d.bias, A=-torch.exp(mixer.A_log), rmsnorm_weight=mixer.norm.weight,
              rmsnorm_eps=mixer.norm.variance_epsilon, outproj_weight=mixer.out_proj.weight, outproj_bias=mixer.out_proj.bias,
              headdim=headdim, ngroups=1, norm_before_gate=False)
    out, _, y = mixer_ref64(zx, mixer.conv1d.weight.squeeze(1), kw["conv_b"], mixer.dt_bias, kw["A"], mixer.D,
                            rmsnorm_weight=kw["rmsnorm_weight"], rmsnorm_eps=kw["rmsnorm_eps"], outproj_weight=kw["outproj_weight"],
                            outproj_bias=kw["outproj_bias"], headdim=headdim, ngroups=1, norm_before_gate=False)
    # torch_forward casts x, B, C and A to float32 before its SSD and forms the C.B contraction in float32 (the rest in
    # float64): the SSD outputs agree to float32 rounding (3e-8 here)
    assert nrel(y, cap["y"]) < 1e-7
    # its gated norm computes in float32 even in a float64 mixer: the output and every parameter gradient agree to 1e-6
    assert nrel(out, out_hf) < 1e-6
    g = torch.randn_like(out)
    params = [p for p in mixer.parameters() if p.requires_grad]
    g_hf = torch.autograd.grad((out_hf * g).sum(), params)
    g_ref = torch.autograd.grad((out * g).sum(), params, allow_unused=True)
    names = [n for n, p in mixer.named_parameters() if p.requires_grad]
    for n, a, b in zip(names, g_ref, g_hf):
        assert a is not None, n
        assert nrel(a, b) < 1e-6, n


@pytest.mark.parametrize("width", [2, 4])
def test_restatement_segments_equal_separate_runs(width):
    """A packed row equals its sequences run one by one: the conv taps and the SSD restart at each boundary, initial_states reach
    the row's leading id-0 sequence, final_states come from its last one; the gradients agree too."""
    t, static = make(2, 23, 2, 4, 1, 3, width=width, d_nonssm=2, outproj="wb", init=True, seed=width)
    rows = [[(0, 1, 0), (1, 3, 1), (3, 23, 2)], [(0, 10, 3), (10, 11, 4), (11, 23, 5)]]
    seq_idx = torch.tensor([[sid for s, e, sid in row for _ in range(s, e)] for row in rows])
    a = call_args(t, "cpu")
    kw = dict(rmsnorm_weight=a["rms_w"], outproj_weight=a["outproj_w"], outproj_bias=a["outproj_b"], **static)
    full, fin, _ = mixer_ref64(a["zxbcdt"], a["conv_w"], a["conv_b"], a["dt_bias"], a["A"], a["D"], a["initial_states"], seq_idx, **kw)
    outs, fins = [], []
    for b, row in enumerate(rows):
        parts = []
        for s, e, sid in row:
            ini = a["initial_states"][b:b + 1] if s == 0 and sid == 0 else None
            o, f, _ = mixer_ref64(a["zxbcdt"][b:b + 1, s:e], a["conv_w"], a["conv_b"], a["dt_bias"], a["A"], a["D"], ini, **kw)
            parts.append(o)
        outs.append(torch.cat(parts, 1))
        fins.append(f)
    sep, sep_fin = torch.cat(outs, 0), torch.cat(fins, 0)
    assert nrel(full, sep) < 1e-13 and nrel(fin, sep_fin) < 1e-13
    g = torch.randn_like(full)
    leaves = [a[k] for k in ("zxbcdt", "conv_w", "conv_b", "dt_bias", "A", "D", "initial_states", "rms_w", "outproj_w")]
    ga = torch.autograd.grad((full * g).sum() + fin.sum(), leaves, allow_unused=True)
    gb = torch.autograd.grad((sep * g).sum() + sep_fin.sum(), leaves, allow_unused=True)
    for x, y in zip(ga, gb):
        assert (x is None and y is None) or nrel(x, y) < 1e-12


def test_conv_ref_with_one_sequence_is_conv1d():
    t, _ = make(2, 9, 2, 4, 1, 3, width=3, seed=1)
    xBC = t["zxbcdt"][..., 8:8 + 14]
    a = conv_ref(xBC, t["conv_w"][:14], t["conv_b"][:14], None, True)
    b = conv_ref(xBC, t["conv_w"][:14], t["conv_b"][:14], torch.full((2, 9), 7), True)
    assert nrel(a, b) < 1e-15


# ---- GPU: the operator against the restatement ------------------------------------------------------------------------------
# (width, activation, bias, d_nonssm, ngroups, norm: None / "nbg" / "nag", outproj: None / "w" / "wb", D (H, P), dt_limit, chunk, L)
CASES = [
    (4, "silu", True, 0, 1, "nag", None, False, (0.0, INF), 256, 200),
    (2, None, False, 0, 1, None, None, False, (0.0, INF), 64, 130),
    (3, "silu", True, 16, 2, "nbg", "w", True, (0.01, 0.5), 64, 100),
    (4, "silu", False, 8, 2, "nag", "wb", False, (0.0, INF), 256, 300),
    (2, "swish", True, 0, 2, None, "wb", True, (0.0, INF), 64, 65),
    (3, None, True, 8, 1, "nbg", None, False, (0.0, 0.3), 256, 77),
    (4, "silu", True, 0, 1, "nbg", "wb", False, (0.0, INF), 64, 3),
    (3, "silu", True, 0, 2, "nag", "w", True, (0.0, INF), 64, 2),
    (2, "silu", True, 16, 1, "nag", None, False, (0.0, INF), 64, 64),
    (4, None, False, 0, 2, None, "w", False, (0.05, INF), 256, 257),
]


def _case(c, batch=2, H=4, P=16, N=16, init=False, seed=0):
    width, act, bias, dn, G, norm, proj, dhp, limit, chunk, L = c
    t, static = make(batch, L, H, P, G, N, width=width, d_nonssm=dn, bias=bias, D_hp=dhp, rms=norm is not None, outproj=proj,
                     init=init, seed=seed)
    return t, static, dict(chunk=chunk, dt_limit=limit, activation=act, nbg=norm != "nag")


@pytest.mark.gpu
@pytest.mark.parametrize("ci", range(len(CASES)))
def test_matrix(ci):
    t, static, kw = _case(CASES[ci], seed=ci)
    errs, _, _ = check_case(t, static, **kw)
    print(CASES[ci], errs)


@pytest.mark.gpu
def test_single_pass_tf32():
    from medical_image_classification_b200 import ssd_combined
    t, static, kw = _case(CASES[3], seed=21)
    ssd_combined.set_precision(1)
    try:
        errs, _, _ = check_case(t, static, elem_bar=5e-3, sum_bar=5e-2, **kw)
    finally:
        ssd_combined.set_precision(None)
    print(errs)


@pytest.mark.gpu
@pytest.mark.parametrize("ci", [0, 2])
def test_bf16_zxbcdt(ci):
    """bf16 zxbcdt: out at rtol 3e-2 / atol 5e-2 element-wise.  Its gradient comes back bf16 and passes through the bf16 y and dy
    between the stages, which the restatement does not round, so it is compared norm-wise at 3e-2 (measured 5e-3), as are the
    parameter gradients; ddt, dA and ddt_bias are left out, as in the SSD's bf16 tests: the SSD backward derives d(cumsum) from its
    bf16 forward output."""
    t, static, kw = _case(CASES[ci], seed=30 + ci)
    _, got, want = check_case(t, static, zx_dtype=torch.bfloat16, elem_bar=INF, sum_bar=INF, **kw)
    H = t["A"].shape[0]
    f = lambda v: v.detach().double().cpu()
    assert torch.allclose(f(got["out"]), f(want["out"]), rtol=3e-2, atol=5e-2)
    assert nrel(f(got["dzxbcdt"])[..., :-H], f(want["dzxbcdt"])[..., :-H]) < 3e-2
    for k in ("dconv_w", "dconv_b", "drms_w", "doutproj_w", "dD"):
        if want.get(k) is not None:
            assert nrel(got[k], want[k]) < 3e-2, k


def _seq_ids(L, bounds):
    ids, sid = [], 0
    for t in range(L):
        if t in bounds:
            sid += 1
        ids.append(sid)
    return ids


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["init", "fin", "both"])
def test_state_arguments(mode):
    """initial_states with a gradient and a loss on the returned final_states.  With a final_states loss, dA and ddt_bias carry
    the chunked backward's last-chunk term, which largely cancels (tests/test_ssd_state_grads.py): they get the single-pass bar."""
    t, static, kw = _case(CASES[2], init=mode != "fin", seed=40)
    with_fin = mode != "init"
    errs, _, _ = check_case(t, static, with_fin=with_fin, skip=("dA", "ddt_bias") if with_fin else (), **kw)
    if with_fin:
        _, got, want = check_case(t, static, with_fin=True, elem_bar=INF, sum_bar=INF, **kw)
        for k in ("dA", "ddt_bias"):
            assert nrel(got[k], want[k]) < 5e-2, (k, nrel(got[k], want[k]))
    print(mode, errs)


# segmentations of L = 100: single tokens, a boundary one / two steps before another (inside the conv window), chunk-crossing runs
SEGMENTATIONS = [[1, 2, 3], [50], [7, 8, 10, 64, 65], [33, 35, 36, 97, 99]]


@pytest.mark.gpu
@pytest.mark.parametrize("si", range(len(SEGMENTATIONS)))
@pytest.mark.parametrize("lead0", [True, False])
def test_seq_idx(si, lead0):
    t, static, kw = _case(CASES[2], init=True, seed=50 + si)
    L = CASES[2][-1]
    ids = _seq_ids(L, SEGMENTATIONS[si])
    rows = [ids, [v + (0 if lead0 else 1) for v in _seq_ids(L, SEGMENTATIONS[(si + 1) % len(SEGMENTATIONS)])]]
    seq_idx = torch.tensor(rows, dtype=torch.int32)
    errs, _, _ = check_case(t, static, seq_idx=seq_idx, **kw)
    print(SEGMENTATIONS[si], lead0, errs)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [
    # (batch, L, H, P, G, N, width, d_nonssm): Mamba-2-130m-like (d_model 768), then MedSSD-like stages flattened to 1-D, the
    # last two with an odd row pitch of zxbcdt (every vector load one element wide)
    (2, 2048, 24, 64, 1, 128, 4, 0),
    (2, 196, 4, 64, 1, 128, 4, 0),
    (2, 49, 6, 64, 1, 64, 4, 1),
    (2, 150, 3, 64, 1, 16, 4, 0),
])
def test_shapes_at_scale(shape):
    batch, L, H, P, G, N, width, dn = shape
    t, static = make(batch, L, H, P, G, N, width=width, d_nonssm=dn, outproj="w", seed=L)
    errs, _, _ = check_case(t, static, chunk=256, nbg=False)
    print(shape, "pitch", t["zxbcdt"].shape[-1], errs)


# ---- causal_conv1d_fn --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("channel_last", [True, False])
@pytest.mark.parametrize("width,act,bias,seq", [(2, None, True, False), (3, "silu", False, True), (4, "silu", True, False),
                                                (4, None, True, True)])
def test_causal_conv1d_fn(dtype, channel_last, width, act, bias, seq):
    from medical_image_classification_b200.conv1d import causal_conv1d_fn
    gen = torch.Generator().manual_seed(width + 10 * int(seq))
    batch, C, L = 3, 70, 131
    x64 = torch.randn(batch, C, L, generator=gen, dtype=torch.float64).to(dtype).double()
    w64 = torch.randn(C, width, generator=gen, dtype=torch.float64) * 0.5
    b64 = torch.randn(C, generator=gen, dtype=torch.float64) if bias else None
    seq_idx = torch.tensor([_seq_ids(L, [1, 5, 6, 60])] * batch) if seq else None
    g = torch.randn(batch, C, L, generator=gen, dtype=torch.float64)
    # x as the kernels see it: a transposed slice of a wider channel-last buffer, or a contiguous (batch, C, L) tensor
    buf = torch.zeros(batch, L, C + 3, dtype=dtype, device="cuda")
    buf[..., 1:C + 1] = x64.transpose(1, 2).to(dtype).cuda()
    x = buf[..., 1:C + 1].transpose(1, 2) if channel_last else x64.to(dtype).cuda().contiguous()
    x.requires_grad_()
    w, b = w64.float().cuda().requires_grad_(), None if b64 is None else b64.float().cuda().requires_grad_()
    out = causal_conv1d_fn(x, w, b, seq_idx=None if seq_idx is None else seq_idx.cuda(), activation=act)
    assert out.shape == (batch, C, L) and out.dtype == dtype
    gx, gw, *gb = torch.autograd.grad(out, [x, w] + ([b] if b is not None else []), g.to(dtype).cuda())
    leaves = [x64.requires_grad_(), w64.requires_grad_()] + ([b64.requires_grad_()] if b64 is not None else [])
    ref = conv_ref(x64.transpose(1, 2), w64, b64, seq_idx, act is not None).transpose(1, 2)
    rg = torch.autograd.grad(ref, leaves, g.to(dtype).double())
    if dtype == torch.float32:
        assert nrel(out, ref) < 2e-6 and nrel(gx, rg[0]) < 2e-6
    else:
        f = lambda v: v.detach().double().cpu()
        assert torch.allclose(f(out), ref, rtol=3e-2, atol=5e-2) and torch.allclose(f(gx), rg[0], rtol=3e-2, atol=5e-2)
    assert nrel(gw, rg[1]) < 2e-5
    if b is not None:
        assert nrel(gb[0], rg[2]) < 2e-5


@pytest.mark.gpu
def test_causal_conv1d_fn_unsupported_arguments():
    from medical_image_classification_b200.conv1d import causal_conv1d_fn
    x, w = torch.randn(1, 8, 5, device="cuda"), torch.randn(8, 4, device="cuda")
    for kw in (dict(initial_states=torch.zeros(1, 8, 3, device="cuda")), dict(return_final_states=True),
               dict(final_states_out=torch.zeros(1, 8, 3, device="cuda"))):
        with pytest.raises(NotImplementedError, match="not implemented"):
            causal_conv1d_fn(x, w, **kw)
    with pytest.raises(RuntimeError, match="activation"):
        causal_conv1d_fn(x, w, activation="relu")
    with pytest.raises(RuntimeError, match="width"):
        causal_conv1d_fn(x, torch.randn(8, 5, device="cuda"))


# ---- memory, reproducibility, graphs ----------------------------------------------------------------------------------------
def _saved_bytes(fn):
    """Bytes of the distinct storages autograd saves while fn() runs."""
    seen = {}

    def pack(t):
        st = t.untyped_storage()
        seen[st.data_ptr()] = st.nbytes()
        return t

    with torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
        out = fn()
    return sum(seen.values()), out


@pytest.mark.gpu
def test_saved_memory():
    from medical_image_classification_b200 import _lib
    from medical_image_classification_b200.conv1d import causal_conv1d_fn
    from medical_image_classification_b200.ssd_combined import mamba_chunk_scan_combined, rmsnorm_fn
    batch, L, H, P, G, N, chunk = 2, 512, 8, 64, 2, 64, 256
    t, static = make(batch, L, H, P, G, N, outproj="wb", seed=5)
    a = call_args(t, "cuda", torch.float32)
    fused, _ = _saved_bytes(lambda: op()(a["zxbcdt"], a["conv_w"], a["conv_b"], a["dt_bias"], a["A"], a["D"], chunk,
                                         rmsnorm_weight=a["rms_w"], outproj_weight=a["outproj_w"], outproj_bias=a["outproj_b"],
                                         norm_before_gate=False, **static))
    dim = H * P
    params = sum(v.numel() * 4 for k, v in a.items() if v is not None and k != "zxbcdt")
    ws = _lib.load().b200_ssd_workspace_bytes(batch, L, H, P, G, N, chunk)
    bound = a["zxbcdt"].numel() * 4 + batch * L * dim * 4 + ws + 8 * batch * L * G + params

    def composed():
        z, xBC, dt = a["zxbcdt"].split([dim, dim + 2 * G * N, H], -1)
        xbc = causal_conv1d_fn(xBC.transpose(1, 2), a["conv_w"], a["conv_b"], activation="silu").transpose(1, 2)
        x, Bm, Cm = xbc.split([dim, G * N, G * N], -1)
        y = mamba_chunk_scan_combined(x.unflatten(-1, (H, P)), dt, a["A"], Bm.unflatten(-1, (G, N)), Cm.unflatten(-1, (G, N)), chunk,
                                      D=a["D"], dt_bias=a["dt_bias"], dt_softplus=True)
        o = rmsnorm_fn(y.flatten(2), a["rms_w"], None, z=z, group_size=dim // G, norm_before_gate=False)
        return F.linear(o, a["outproj_w"], a["outproj_b"])

    comp, _ = _saved_bytes(composed)
    print(f"saved bytes: fused {fused}, composed {comp}, bound {bound}")
    assert fused <= bound, (fused, bound)
    assert comp > fused


@pytest.mark.gpu
def test_conv_weight_gradients_are_reproducible():
    t, static = make(4, 700, 4, 64, 1, 64, outproj="w", seed=6)
    a = call_args(t, "cuda", torch.float32)
    out = op()(a["zxbcdt"], a["conv_w"], a["conv_b"], a["dt_bias"], a["A"], a["D"], 256, rmsnorm_weight=a["rms_w"],
               outproj_weight=a["outproj_w"], **static)
    g = torch.randn_like(out)
    r1 = torch.autograd.grad(out, [a["conv_w"], a["conv_b"]], g, retain_graph=True)
    r2 = torch.autograd.grad(out, [a["conv_w"], a["conv_b"]], g)
    assert all(torch.equal(x, y) for x, y in zip(r1, r2))


@pytest.mark.gpu
def test_graph_capture():
    t, static = make(2, 200, 4, 16, 2, 16, d_nonssm=8, outproj="wb", init=True, seed=7)
    a = call_args(t, "cuda", torch.float32)
    leaves = {k: v for k, v in a.items() if v is not None}
    seq_idx = torch.tensor([_seq_ids(200, [30, 31])] * 2, dtype=torch.int32, device="cuda")
    gout = torch.randn(2, 200, 24, device="cuda")

    def step():
        out, fin = op()(a["zxbcdt"], a["conv_w"], a["conv_b"], a["dt_bias"], a["A"], a["D"], 64, initial_states=a["initial_states"],
                        seq_idx=seq_idx, return_final_states=True, rmsnorm_weight=a["rms_w"], outproj_weight=a["outproj_w"],
                        outproj_bias=a["outproj_b"], **static)
        return (out,) + torch.autograd.grad((out * gout).sum() + fin.sum(), list(leaves.values()))

    eager = [v.detach().clone() for v in step()]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        res = step()
    g.replay()
    torch.cuda.synchronize()
    for x, y in zip(res, eager):
        assert nrel(x, y) < 1e-6


# ---- errors ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_argument_errors():
    from medical_image_classification_b200 import _lib
    t, static = make(2, 40, 4, 16, 2, 16, d_nonssm=4, outproj="wb", seed=8)
    a = {k: None if v is None else v.float().cuda() for k, v in t.items()}
    before = _lib.launches()

    def call(**kw):
        args = dict(zxbcdt=a["zxbcdt"], conv1d_weight=a["conv_w"], conv1d_bias=a["conv_b"], dt_bias=a["dt_bias"], A=a["A"], D=a["D"],
                    chunk_size=64, **static)
        args.update(kw)
        return op()(**args)

    cases = [
        (dict(zxbcdt=a["zxbcdt"][..., 1:]), "do not split"),
        (dict(zxbcdt=a["zxbcdt"][..., :100]), "do not split"),
        (dict(ngroups=3), "multiple of ngroups"),
        (dict(conv1d_weight=a["conv_w"][:, :, None]), "conv1d_weight must be"),
        (dict(conv1d_weight=torch.zeros(a["conv_w"].shape[0], 5, device="cuda")), "width 5"),
        (dict(conv1d_weight=torch.zeros(a["conv_w"].shape[0], 1, device="cuda")), "width 1"),
        (dict(activation="relu"), "activation"),
        (dict(headdim=None), "needs headdim"),
        (dict(zxbcdt=a["zxbcdt"].cpu()), "no CPU fallback"),
        (dict(seq_idx=torch.zeros(2, 39, dtype=torch.int32, device="cuda")), "seq_idx must be"),
        (dict(seq_idx=torch.zeros(2, 40, device="cuda")), "seq_idx must hold integers"),
        (dict(outproj_bias=a["outproj_b"]), "outproj_bias needs outproj_weight"),
        (dict(outproj_weight=a["outproj_w"][:, 1:]), "outproj_weight must be"),
        (dict(rmsnorm_weight=a["rms_w"][1:]), "rmsnorm_weight must be"),
        (dict(initial_states=torch.zeros(2, 4, 16, 15, device="cuda")), "initial_states must be"),
    ]
    for kw, msg in cases:
        with pytest.raises(RuntimeError, match=msg):
            call(**kw)
    assert _lib.launches() == before


@pytest.mark.gpu
def test_c_entry_point_errors():
    """Bad sizes, width, dtype codes, NULL pointers and negative strides return < 0 with a message and launch nothing."""
    from medical_image_classification_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(2, 10, 8, device="cuda")
    w = torch.zeros(8, 4, device="cuda")
    p = x.data_ptr()
    fwd = dict(x=p, xd=0, xb=80, xl=8, w=w.data_ptr(), b=None, s=None, sb=0, sl=0, o=p, od=0, ob=80, ol=8, B=2, L=10, C=8, W=4, silu=1)

    def f(**kw):
        d = dict(fwd, **kw)
        return lib.b200_causal_conv1d_fwd(*d.values(), None)

    def b(**kw):
        d = dict(g=p, gb=80, gl=8, x=p, xd=0, xb=80, xl=8, w=w.data_ptr(), bias=None, s=None, sb=0, sl=0, dx=p, dxb=80, dxl=8,
                 dwp=p, dbp=None, B=2, L=10, C=8, W=4, silu=1)
        d.update(kw)
        return lib.b200_causal_conv1d_bwd(*d.values(), None)

    before = lib.b200_kernel_launches()
    bad = [(f, dict(W=5), b"width"), (f, dict(W=1), b"width"), (f, dict(L=0), b"seqlen"), (f, dict(B=0), b"batch"),
           (f, dict(C=0), b"dim"), (f, dict(xd=7), b"dtype"), (f, dict(od=-1), b"dtype"), (f, dict(x=None), b"NULL"),
           (f, dict(xl=-8), b"negative"), (f, dict(ob=-1), b"negative"), (f, dict(sl=-1), b"negative"),
           (b, dict(W=5), b"width"), (b, dict(xd=3), b"dtype"), (b, dict(dwp=None), b"NULL"), (b, dict(gl=-8), b"negative"),
           (b, dict(dxb=-80), b"negative"), (b, dict(L=-1), b"seqlen")]
    for fn, kw, msg in bad:
        assert fn(**kw) < 0, kw
        assert msg in lib.b200_last_error(), (kw, lib.b200_last_error())
    assert lib.b200_causal_conv1d_partials(2, 10, 8, 5) < 0
    assert lib.b200_causal_conv1d_partials(2, 130, 8, 4) == 2 * 3
    assert lib.b200_kernel_launches() == before
