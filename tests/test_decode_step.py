"""Recurrent decoding: selective_state_update (csrc/state_update.cu) and causal_conv1d_update (csrc/conv1d.cu).

ssu_ref64 and conv_update_ref64 restate one step of each op in float64.  On the CPU they are pinned against the sequence
restatements (stepping them over L tokens equals ssd_ref64 / conv_ref over the L tokens) and, composed with ssd_ref64 for a
prefill, against transformers' Mamba2Mixer.torch_forward decoding through a DynamicCache.  The GPU tests check the kernels against
them, against a longer prefill, inside transformers' cuda_kernels_forward, against vLLM's Triton kernel and in a CUDA graph.

Bars (norm-wise relative error): fp32 2e-6 after one step and 2e-5 after 64; with a 16-bit state, which the restatement rounds to
that dtype after every step as the kernel does, 1e-2 (bf16) and 2e-3 (f16) after 16 steps.
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from test_rmsnorm import nrel
from test_split_conv1d import conv_ref
from test_ssd_state_ref import ssd_ref64


# ---- the float64 restatements -------------------------------------------------------------------------------------------------
def ssu_ref64(state, x, dt, A, B, C, D=None, z=None, dt_bias=None, dt_softplus=False):
    """(out, new state) of one selective_state_update step, either form, without touching `state`."""
    if state.dim() == 3:
        u1 = lambda t: None if t is None else t.unsqueeze(1)
        out, new = ssu_ref64(state.unsqueeze(1), x.unsqueeze(1), dt.unsqueeze(1), A.unsqueeze(0), B.unsqueeze(1), C.unsqueeze(1),
                             None if D is None else D.unsqueeze(0), u1(z), None if dt_bias is None else dt_bias.unsqueeze(0), dt_softplus)
        return out.squeeze(1), new.squeeze(1)
    H, G = state.shape[1], B.shape[1]
    v = dt + dt_bias if dt_bias is not None else dt
    if dt_softplus:
        v = torch.where(v > 20.0, v, torch.log1p(torch.exp(torch.clamp(v, max=20.0))))
    Bh, Ch = B.repeat_interleave(H // G, 1)[:, :, None], C.repeat_interleave(H // G, 1)[:, :, None]
    new = state * torch.exp(A * v[..., None]) + Bh * v[..., None] * x[..., None]
    out = (new * Ch).sum(-1)
    if D is not None:
        out = out + D * x
    if z is not None:
        out = out * F.silu(z)
    return out, new


def conv_update_ref64(x, conv_state, weight, bias=None, silu=False):
    """(out, new conv_state) of causal_conv1d_update over cat(conv_state, x), x (batch, dim) or (batch, dim, seqlen)."""
    x3 = x.unsqueeze(-1) if x.dim() == 2 else x
    L, S = x3.shape[-1], conv_state.shape[-1]
    v = torch.cat([conv_state, x3], -1)
    out = F.conv1d(v, weight.unsqueeze(1), bias, groups=weight.shape[0])[..., -L:]
    out = F.silu(out) if silu else out
    return (out.squeeze(-1) if x.dim() == 2 else out), v[..., -S:]


def _r(gen, *s):
    return torch.randn(*s, generator=gen, dtype=torch.float64)


# ---- CPU: the restatements against the sequence restatements and transformers ------------------------------------------------
@pytest.mark.parametrize("G,D_hp,with_z", [(1, False, False), (2, True, True), (2, False, True), (1, True, False)])
def test_ssu_ref_steps_equal_ssd_ref(G, D_hp, with_z):
    gen = torch.Generator().manual_seed(G + 2 * D_hp + 4 * with_z)
    batch, L, H, P, N = 2, 9, 4, 3, 5
    x, dt = _r(gen, batch, L, H, P), _r(gen, batch, L, H) * 0.5
    A, Bm, Cm = -0.5 - torch.rand(H, generator=gen, dtype=torch.float64), _r(gen, batch, L, G, N), _r(gen, batch, L, G, N)
    D, dt_bias, z = _r(gen, H, P) if D_hp else _r(gen, H), _r(gen, H) * 0.3, _r(gen, batch, L, H, P) if with_z else None
    S0 = _r(gen, batch, H, P, N)
    want, fin = ssd_ref64(x, dt, A, Bm, Cm, None, dt_bias, True, initial_states=S0)
    want = want + x * (D if D_hp else D[:, None])
    if with_z:
        want = want * F.silu(z)
    S, outs = S0, []
    Dx = D if D_hp else D[:, None].expand(H, P)
    for t in range(L):
        o, S = ssu_ref64(S, x[:, t], dt[:, t, :, None].expand(batch, H, P), A[:, None, None].expand(H, P, N), Bm[:, t], Cm[:, t], Dx,
                         None if z is None else z[:, t], dt_bias[:, None].expand(H, P), True)
        outs.append(o)
    assert nrel(torch.stack(outs, 1), want) < 1e-12 and nrel(S, fin) < 1e-12


@pytest.mark.parametrize("width", [2, 3, 4])
@pytest.mark.parametrize("state_extra", [0, 1, None])
def test_conv_update_ref_steps_equal_conv_ref(width, state_extra):
    """state_len width-1, width and 8; one token per step, then blocks of 3 tokens."""
    S = 8 if state_extra is None else width - 1 + state_extra
    gen = torch.Generator().manual_seed(width * 10 + S)
    batch, C, L = 2, 6, 13
    x, w, b = _r(gen, batch, C, L), _r(gen, C, width), _r(gen, C)
    want = conv_ref(x.transpose(1, 2), w, b, None, True).transpose(1, 2)
    for block in (1, 3):
        st, outs = torch.zeros(batch, C, S, dtype=torch.float64), []
        for t in range(0, L, block):
            xt = x[:, :, t] if block == 1 else x[:, :, t:t + block]
            o, st = conv_update_ref64(xt, st, w, b, True)
            outs.append(o.unsqueeze(-1) if block == 1 else o)
        assert nrel(torch.cat(outs, -1), want) < 1e-13
        tail = F.pad(x, (max(S - L, 0), 0))[..., -S:]
        assert torch.equal(st, tail)


def _hf_cfg(heads, headdim, groups, dstate, chunk):
    """The Mamba2Config test_oracle_ssd._hf_mixer builds its mixer from."""
    cfg_cls = pytest.importorskip("transformers").Mamba2Config
    return cfg_cls(num_heads=heads, head_dim=headdim, hidden_size=heads * headdim // 2, state_size=dstate, expand=2, n_groups=groups,
                   chunk_size=chunk, conv_kernel=4, num_hidden_layers=1, vocab_size=16, use_conv_bias=True, use_bias=False,
                   time_step_limit=(0.0, float("inf")))


def _mixer_decode_ref64(mixer, hidden, L0):
    """Per-token outputs of the mixer from the restatements: ssd_ref64 / conv_ref over the first L0 tokens, then one
    conv_update_ref64 + ssu_ref64 step per token; the gated norm and out_proj are the mixer's own layers."""
    H, P, N, G = mixer.num_heads, mixer.head_dim, mixer.ssm_state_size, mixer.n_groups
    dim, W = H * P, mixer.conv_kernel_size
    zx = mixer.in_proj(hidden)
    batch, L = zx.shape[:2]
    gate, xBC, dt = zx[..., -(2 * dim + 2 * G * N + H):].split([dim, dim + 2 * G * N, H], -1)
    w, b, A = mixer.conv1d.weight.squeeze(1), mixer.conv1d.bias, -torch.exp(mixer.A_log)
    xbc = conv_ref(xBC[:, :L0], w, b, None, True)
    x, Bm, Cm = xbc.split([dim, G * N, G * N], -1)
    y, S = ssd_ref64(x.unflatten(-1, (H, P)), dt[:, :L0], A, Bm.unflatten(-1, (G, N)), Cm.unflatten(-1, (G, N)), mixer.D, mixer.dt_bias)
    ys = [y.flatten(2)]
    cs = F.pad(xBC[:, :L0].transpose(1, 2), (max(W - L0, 0), 0))[..., -W:]
    for t in range(L0, L):
        o, cs = conv_update_ref64(xBC[:, t], cs, w, b, True)
        x, Bm, Cm = o.split([dim, G * N, G * N], -1)
        yt, S = ssu_ref64(S, x.unflatten(-1, (H, P)), dt[:, t, :, None].expand(batch, H, P), A[:, None, None].expand(H, P, N),
                          Bm.unflatten(-1, (G, N)), Cm.unflatten(-1, (G, N)), mixer.D[:, None].expand(H, P), None,
                          mixer.dt_bias[:, None].expand(H, P), True)
        ys.append(yt.flatten(1)[:, None])
    return mixer.out_proj(mixer.norm(torch.cat(ys, 1), gate))


def test_restatement_matches_transformers_decoding():
    """torch_forward over a prefill of L0 tokens and k decode steps through a DynamicCache against the restatements.  As in
    test_split_conv1d.test_restatement_matches_transformers_mixer, torch_forward casts parts of its SSD and its gated norm to
    float32, so the two agree to float32 rounding, not float64."""
    from test_oracle_ssd import _hf_mixer
    cache_cls = pytest.importorskip("transformers").DynamicCache
    heads, headdim, groups, dstate, chunk, L0, k = 4, 8, 2, 12, 16, 7, 3
    mixer = _hf_mixer(L0 + k, heads, headdim, groups, dstate, chunk, seed=5)
    torch.manual_seed(6)
    hidden = torch.randn(2, L0 + k, heads * headdim // 2, dtype=torch.float64)
    with torch.no_grad():
        cache = cache_cls(config=_hf_cfg(heads, headdim, groups, dstate, chunk))
        outs = [mixer.torch_forward(hidden[:, :L0], cache_params=cache)]
        outs += [mixer.torch_forward(hidden[:, t:t + 1], cache_params=cache) for t in range(L0, L0 + k)]
        hf = torch.cat(outs, 1)
        full = mixer.torch_forward(hidden)
        ref = _mixer_decode_ref64(mixer, hidden, L0)
    assert nrel(hf, full) < 1e-6
    for t in range(L0 + k):
        assert nrel(ref[:, t], hf[:, t]) < 1e-6, t


# ---- GPU: the kernels against the restatements -------------------------------------------------------------------------------
def ssu_op():
    from medical_image_classification_b200.selective_state_update import selective_state_update
    return selective_state_update


def conv_update_op():
    from medical_image_classification_b200.conv1d import causal_conv1d_update
    return causal_conv1d_update


def ssu_inputs(batch, H, P, G, N, dtype, tied, D_mode, with_z, with_bias, pitch, gen, mamba1=False):
    """One step's arguments on the GPU (x, B, C as column slices of one wider buffer when pitch is set; A, dt, dt_bias, D expanded
    when tied), and the same values in float64."""
    dev = "cuda"
    width = H * P + 2 * G * N
    buf = _r(gen, batch, (pitch or width) + 1).to(dev, dtype)
    off = 1 if pitch else 0
    x = buf[:, off:off + H * P].unflatten(-1, (H, P))
    Bm = buf[:, off + H * P:off + H * P + G * N].unflatten(-1, (G, N))
    Cm = buf[:, off + H * P + G * N:off + width].unflatten(-1, (G, N))
    if tied:
        dt = (0.5 * torch.rand(batch, H, generator=gen, dtype=torch.float64) - 0.2).to(dev, dtype)[:, :, None].expand(batch, H, P)
        A = (-0.5 - torch.rand(H, generator=gen, dtype=torch.float64)).to(dev, torch.float32)[:, None, None].expand(H, P, N)
        bias = (0.3 * torch.rand(H, generator=gen, dtype=torch.float64)).to(dev, dtype)[:, None].expand(H, P)
    else:
        dt = (0.5 * torch.rand(batch, H, P, generator=gen, dtype=torch.float64) - 0.2).to(dev, dtype)
        A = (-0.5 - torch.rand(H, P, N, generator=gen, dtype=torch.float64)).to(dev, torch.float32)
        bias = (0.3 * torch.rand(H, P, generator=gen, dtype=torch.float64)).to(dev, dtype)
    D = {None: None, "h": _r(gen, H).to(dev, dtype)[:, None].expand(H, P), "hp": _r(gen, H, P).to(dev, dtype)}[D_mode]
    z = _r(gen, batch, H, P).to(dev, dtype) if with_z else None
    a = dict(x=x, dt=dt, A=A, B=Bm, C=Cm, D=D, z=z, dt_bias=bias if with_bias else None)
    if mamba1:          # H = 1: drop the head dimension
        a = {k: None if v is None else (v[0] if k in ("A", "D", "dt_bias") else v[:, 0]) for k, v in a.items()}
    return a, {k: None if v is None else v.double() for k, v in a.items()}


# (batch, H, P, G, N, dtype, tied, D_mode, z, dt_bias, softplus, pitch); pitch None = dense; H None = Mamba-1 (dim P, dstate N)
SSU_CASES = [
    (3, 24, 64, 1, 128, torch.float32, True, "h", False, True, True, None),
    (64, 80, 64, 1, 128, torch.float32, True, "h", False, True, True, 5557),
    (1, 8, 48, 2, 64, torch.float32, False, "hp", True, False, False, 901),
    (3, 4, 64, 4, 256, torch.float32, False, None, True, True, True, None),
    (3, None, 1536, 1, 16, torch.float32, False, "hp", True, True, True, 1601),
    (64, 24, 64, 1, 128, torch.bfloat16, True, "h", False, True, True, 3333),
    (3, 8, 48, 2, 64, torch.bfloat16, False, "hp", True, True, False, None),
    (1, 4, 64, 4, 256, torch.float16, True, None, True, False, True, 2411),
    (3, None, 1536, 1, 16, torch.float16, False, "hp", False, True, True, None),
    (64, None, 1536, 1, 16, torch.bfloat16, False, None, True, True, True, 1601),
    (1, 80, 64, 1, 128, torch.float16, True, "h", True, True, True, None),
]


def _ssu_run(case, steps, seed):
    batch, H, P, G, N, dtype, tied, D_mode, with_z, with_bias, softplus, pitch = case
    mamba1 = H is None
    gen = torch.Generator().manual_seed(seed)
    shape = (batch, P, N) if mamba1 else (batch, H, P, N)
    state = _r(gen, *shape).to("cuda", dtype)
    S = state.double()
    errs = []
    for _ in range(steps):
        a, a64 = ssu_inputs(batch, 1 if mamba1 else H, P, G, N, dtype, tied, D_mode, with_z, with_bias, pitch, gen, mamba1)
        out = ssu_op()(state, **a, dt_softplus=softplus)
        want, S = ssu_ref64(S, **a64, dt_softplus=softplus)
        S = S.to(dtype).double()            # the kernel stores the state in its dtype after every step
        assert out.shape == a["x"].shape and out.dtype == dtype
        errs.append(nrel(out, want))
    return errs, nrel(state, S)


@pytest.mark.gpu
@pytest.mark.parametrize("ci", range(len(SSU_CASES)))
def test_ssu_matrix(ci):
    case = SSU_CASES[ci]
    dtype = case[5]
    if dtype == torch.float32:
        e1, s1 = _ssu_run(case, 1, ci)
        assert max(e1) < 2e-6 and s1 < 2e-6, (e1, s1)
        e, s = _ssu_run(case, 64, ci)
        assert max(e) < 2e-5 and s < 2e-5, (max(e), s)
    else:
        bar = 1e-2 if dtype == torch.bfloat16 else 2e-3
        e, s = _ssu_run(case, 16, ci)
        assert max(e) < bar and s < bar, (max(e), s)
    print(case, max(e), s)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("width,state_len,seqlen,act,bias", [(4, 4, 1, "silu", True), (2, 1, 1, None, False), (3, 8, 5, "swish", True),
                                                             (4, 3, 7, "silu", False), (4, 6, 2, None, True)])
def test_conv_update_matrix(dtype, width, state_len, seqlen, act, bias):
    gen = torch.Generator().manual_seed(width * 100 + state_len * 10 + seqlen)
    batch, C, pitch = 3, 70, 95
    st = _r(gen, batch, C, state_len).to("cuda", dtype)
    S = st.double()
    w = _r(gen, C, width).to("cuda", dtype)
    b = _r(gen, C).to("cuda", dtype) if bias else None
    for _ in range(3):
        buf = _r(gen, batch, seqlen, pitch).to("cuda", dtype)
        x = buf[..., 2:2 + C].transpose(1, 2)            # (batch, C, seqlen) column slice, time stride pitch
        if seqlen == 1:
            x = x[..., 0]
        out = conv_update_op()(x, st, w, b, act)
        want, S = conv_update_ref64(x.double(), S, w.double(), None if b is None else b.double(), act is not None)
        assert out.shape == x.shape and out.dtype == dtype
        assert torch.equal(st, S.to(dtype)), "conv_state is not the last state_len inputs"
        if dtype == torch.float32:
            assert nrel(out, want) < 2e-6
        else:
            assert torch.allclose(out.double(), want, rtol=1e-2, atol=2e-2)


# ---- in-place writes ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_writes_stay_inside_the_views(dtype):
    from medical_image_classification_b200 import _lib
    from medical_image_classification_b200.selective_state_update import _set
    gen = torch.Generator().manual_seed(7)
    batch, H, P, G, N = 3, 8, 48, 2, 64
    big = _r(gen, batch + 1, H + 1, P + 1, N + 3).to("cuda", dtype)
    state = big[1:, 1:, :P, 2:2 + N]
    before = big.clone()
    a, a64 = ssu_inputs(batch, H, P, G, N, dtype, False, "hp", True, True, 901, gen)
    obuf = torch.full((batch * H * P + 64,), 7.0, dtype=dtype, device="cuda")
    out = obuf[32:32 + batch * H * P].view(batch, H, P)
    want, S = ssu_ref64(state.double(), **a64, dt_softplus=True)
    p = _lib.SsuParams(batch=batch, nheads=H, headdim=P, ngroups=G, dstate=N, dt_softplus=1)
    for k, shape in (("x", (batch, H, P)), ("dt", (batch, H, P)), ("A", (H, P, N)), ("B", (batch, G, N)), ("C", (batch, G, N)),
                     ("D", (H, P)), ("z", (batch, H, P)), ("dt_bias", (H, P))):
        _set(p, k, a[k], shape)
    _set(p, "state", state, (batch, H, P, N))
    _set(p, "out", out, (batch, H, P))
    _lib.launch("b200_selective_state_update", "cuda", ctypes.byref(p))
    torch.cuda.synchronize()
    mask = torch.ones_like(big, dtype=torch.bool)
    mask[1:, 1:, :P, 2:2 + N] = False
    ib = torch.int32 if dtype == torch.float32 else torch.int16
    assert torch.equal(big.view(ib)[mask], before.view(ib)[mask]), "state: write outside the view"
    assert torch.equal(obuf[:32], torch.full((32,), 7.0, dtype=dtype, device="cuda"))
    assert torch.equal(obuf[-32:], torch.full((32,), 7.0, dtype=dtype, device="cuda"))
    bar = 2e-6 if dtype == torch.float32 else 1e-2
    assert nrel(out, want) < bar and nrel(state, S) < bar
    # conv_state inside a wider buffer
    cbig = _r(gen, batch + 1, 70, 9).to("cuda", dtype)
    cst = cbig[1:, 3:67, 2:6]
    cbefore = cbig.clone()
    x = _r(gen, batch, 64).to("cuda", dtype)
    conv_update_op()(x, cst, _r(gen, 64, 4).to("cuda", dtype), None, "silu")
    cmask = torch.ones_like(cbig, dtype=torch.bool)
    cmask[1:, 3:67, 2:6] = False
    assert torch.equal(cbig.view(ib)[cmask], cbefore.view(ib)[cmask]), "conv_state: write outside the view"
    assert torch.equal(cst[..., -1], x)


# ---- transformers' argument sets: one launch each ----------------------------------------------------------------------------
def _hf_step_args(batch, H, P, G, N, W, dtype, gen):
    """causal_conv1d_update and selective_state_update arguments exactly as Mamba2Mixer.cuda_kernels_forward builds them."""
    dim, conv_dim = H * P, H * P + 2 * G * N
    dev = "cuda"
    proj = _r(gen, batch, 2 * dim + 2 * G * N + H).to(dev, dtype)
    gate, xBC, dt = proj.split([dim, conv_dim, H], -1)
    conv_state = _r(gen, batch, conv_dim, W).to(dev, dtype)
    ssm_state = _r(gen, batch, H, P, N).to(dev, dtype)
    w, b = (_r(gen, conv_dim, 1, W) * 0.3).to(dev, dtype).squeeze(1), (_r(gen, conv_dim) * 0.1).to(dev, dtype)
    A_log, D, dt_bias = torch.rand(H, generator=gen).to(dev, dtype), _r(gen, H).to(dev, dtype), (0.3 * _r(gen, H)).to(dev, dtype)

    def ssu_args(xbc):
        x, Bm, Cm = torch.split(xbc, [dim, G * N, G * N], dim=-1)
        A = -torch.exp(A_log.float())
        A = A[:, None, ...][:, :, None].expand(-1, P, N).to(dtype=torch.float32)
        return (ssm_state, x.view(batch, H, P), dt[:, :, None].expand(-1, -1, P), A, Bm.view(batch, G, N), Cm.view(batch, G, N),
                D[:, None, ...].expand(-1, P)), dict(z=None, dt_bias=dt_bias[:, None, ...].expand(-1, P), dt_softplus=True)

    return (xBC, conv_state, w, b, "silu"), ssu_args


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_one_launch_per_call_with_transformers_arguments(dtype):
    from medical_image_classification_b200 import _lib
    gen = torch.Generator().manual_seed(11)
    conv_args, ssu_args = _hf_step_args(4, 24, 64, 1, 128, 4, dtype, gen)
    n0 = _lib.launches()
    xbc = conv_update_op()(*conv_args)
    n1 = _lib.launches()
    args, kw = ssu_args(xbc)
    ssu_op()(*args, **kw)
    n2 = _lib.launches()
    assert (n1 - n0, n2 - n1) == (1, 1)


# ---- prefill then decode -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_prefill_then_decode_equals_longer_prefill():
    from medical_image_classification_b200.conv1d import causal_conv1d_fn
    from medical_image_classification_b200.ssd_combined import mamba_chunk_scan_combined
    gen = torch.Generator().manual_seed(12)
    batch, H, P, G, N, W, L0, k = 2, 8, 64, 2, 64, 4, 100, 6
    dim, conv_dim = H * P, H * P + 2 * G * N
    dev = "cuda"
    xBC = _r(gen, batch, L0 + k, conv_dim).float().to(dev)
    dt = (0.5 * torch.rand(batch, L0 + k, H, generator=gen) - 0.2).to(dev)
    w, b = (_r(gen, conv_dim, W) * 0.3).float().to(dev), (_r(gen, conv_dim) * 0.1).float().to(dev)
    A, D, bias = (-0.5 - torch.rand(H, generator=gen)).to(dev), _r(gen, H).float().to(dev), (0.3 * torch.rand(H, generator=gen)).to(dev)

    def prefill(L):
        xbc = causal_conv1d_fn(xBC[:, :L].transpose(1, 2), w, b, activation="silu").transpose(1, 2)
        x, Bm, Cm = xbc.split([dim, G * N, G * N], -1)
        return mamba_chunk_scan_combined(x.unflatten(-1, (H, P)), dt[:, :L], A, Bm.unflatten(-1, (G, N)), Cm.unflatten(-1, (G, N)), 64,
                                         D=D, dt_bias=bias, dt_softplus=True, return_final_states=True)

    y_full, fin_full = prefill(L0 + k)
    _, state = prefill(L0)
    conv_state = xBC[:, L0 - W:L0].transpose(1, 2).contiguous()
    for i in range(k):
        xbc = conv_update_op()(xBC[:, L0 + i], conv_state, w, b, "silu")
        x, Bm, Cm = xbc.split([dim, G * N, G * N], -1)
        y = ssu_op()(state, x.view(batch, H, P), dt[:, L0 + i, :, None].expand(batch, H, P), A[:, None, None].expand(H, P, N),
                     Bm.view(batch, G, N), Cm.view(batch, G, N), D[:, None].expand(H, P), dt_bias=bias[:, None].expand(H, P),
                     dt_softplus=True)
        assert nrel(y, y_full[:, L0 + i]) < 2e-5, i
    assert nrel(state, fin_full) < 2e-5


# ---- transformers end to end -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_transformers_mixer_decodes_on_these_kernels(monkeypatch):
    from test_oracle_ssd import _hf_mixer
    from medical_image_classification_b200.conv1d import causal_conv1d_fn
    from medical_image_classification_b200.ssd_combined import mamba_chunk_scan_combined, mamba_split_conv1d_scan_combined
    m2 = pytest.importorskip("transformers.models.mamba2.modeling_mamba2")
    cache_cls = pytest.importorskip("transformers").DynamicCache
    heads, headdim, groups, dstate, chunk, L0, k = 8, 64, 2, 64, 64, 37, 8
    ref = _hf_mixer(L0 + k, heads, headdim, groups, dstate, chunk, seed=13)
    mixer = _hf_mixer(L0 + k, heads, headdim, groups, dstate, chunk, seed=13).float().cuda()
    calls = {"ssu": 0, "conv": 0}

    def counted(name, fn):
        def wrapper(*a, **kw):
            calls[name] += 1
            return fn(*a, **kw)
        return wrapper

    monkeypatch.setattr(m2, "selective_state_update", counted("ssu", ssu_op()), raising=False)
    monkeypatch.setattr(m2, "causal_conv1d_update", counted("conv", conv_update_op()), raising=False)
    monkeypatch.setattr(m2, "causal_conv1d_fn", causal_conv1d_fn, raising=False)
    monkeypatch.setattr(m2, "mamba_chunk_scan_combined", mamba_chunk_scan_combined, raising=False)
    monkeypatch.setattr(m2, "mamba_split_conv1d_scan_combined", mamba_split_conv1d_scan_combined, raising=False)
    torch.manual_seed(14)
    hidden = torch.randn(2, L0 + k, heads * headdim // 2, dtype=torch.float64)
    cfg = _hf_cfg(heads, headdim, groups, dstate, chunk)
    try:
        c_ref, c_gpu = cache_cls(config=cfg), cache_cls(config=cfg)
        with torch.no_grad():
            want = [ref.torch_forward(hidden[:, :L0], cache_params=c_ref)]
            want += [ref.torch_forward(hidden[:, t:t + 1], cache_params=c_ref) for t in range(L0, L0 + k)]
            hc = hidden.float().cuda()
            got = [mixer.cuda_kernels_forward(hc[:, :L0], cache_params=c_gpu)]
            got += [mixer.cuda_kernels_forward(hc[:, t:t + 1], cache_params=c_gpu) for t in range(L0, L0 + k)]
    except (TypeError, AttributeError) as exc:     # a cache API this transformers does not have
        pytest.skip(f"transformers' cache API does not fit: {type(exc).__name__}: {str(exc)[:200]}")
    assert calls == {"ssu": k, "conv": k}
    want, got = torch.cat(want, 1), torch.cat(got, 1)
    for t in range(L0 + k):
        assert nrel(got[:, t], want[:, t]) < 2e-5, t


# ---- vLLM cross-check --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("H,G,dtype", [(24, 1, torch.float32), (80, 1, torch.float32), (24, 1, torch.bfloat16)])
def test_matches_vllm_selective_state_update(H, G, dtype):
    mod = pytest.importorskip("vllm.model_executor.layers.mamba.ops.mamba_ssm")
    gen = torch.Generator().manual_seed(H)
    batch, P, N = 8, 64, 128
    a, _ = ssu_inputs(batch, H, P, G, N, dtype, True, "h", False, True, None, gen)
    state = _r(gen, batch, H, P, N).to("cuda", dtype)
    s2 = state.clone()
    out = ssu_op()(state, **a, dt_softplus=True)
    try:
        o2 = torch.empty_like(a["x"])
        r = mod.selective_state_update(s2, a["x"], a["dt"], a["A"], a["B"], a["C"], a["D"], a["dt_bias"], z=a["z"], dt_softplus=True,
                                       out=o2)
        o2 = o2 if r is None else r
    except Exception as exc:   # an API drift or a missing runtime in the installed vLLM is not a failure of this repo
        pytest.skip(f"vLLM selective_state_update not usable here: {type(exc).__name__}: {str(exc)[:200]}")
    bar = 2e-6 if dtype == torch.float32 else 1e-2
    assert nrel(out, o2) < bar and nrel(state, s2) < bar, (nrel(out, o2), nrel(state, s2))


# ---- CUDA graphs -------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_decode_step_in_a_cuda_graph():
    gen = torch.Generator().manual_seed(15)
    conv_args, ssu_args = _hf_step_args(3, 8, 64, 2, 64, 4, torch.float32, gen)
    xBC, conv_state, w, b, act = conv_args
    ssm_state = ssu_args(xBC)[0][0]
    init = (conv_state.clone(), ssm_state.clone())

    def step():
        args, kw = ssu_args(conv_update_op()(xBC, conv_state, w, b, act))
        return ssu_op()(*args, **kw)

    def reset():
        conv_state.copy_(init[0])
        ssm_state.copy_(init[1])

    eager = [step().clone() for _ in range(3)]
    eager_states = (conv_state.clone(), ssm_state.clone())
    reset()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step()
    reset()
    replayed = []
    for _ in range(3):
        g.replay()
        replayed.append(out.clone())
    torch.cuda.synchronize()
    for a, e in zip(replayed, eager):
        assert torch.equal(a, e)
    assert torch.equal(conv_state, eager_states[0]) and torch.equal(ssm_state, eager_states[1])


# ---- errors ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_argument_errors():
    from medical_image_classification_b200 import _lib
    gen = torch.Generator().manual_seed(16)
    batch, H, P, G, N = 2, 4, 16, 2, 32
    a, _ = ssu_inputs(batch, H, P, G, N, torch.float32, True, "h", True, True, None, gen)
    state = torch.zeros(batch, H, P, N, device="cuda")
    x2, cs, w = torch.zeros(2, 8, device="cuda"), torch.zeros(2, 8, 4, device="cuda"), torch.zeros(8, 4, device="cuda")
    before = _lib.launches()
    ssu_cases = [
        (dict(state=state[..., :-1]), "must be"),
        (dict(x=a["x"][:, :, :-1]), "x must be"),
        (dict(B=a["B"][:, :, :-1]), "B must be"),
        (dict(D=torch.zeros(H, device="cuda")), "D must be"),
        (dict(B=torch.zeros(batch, 3, N, device="cuda"), C=torch.zeros(batch, 3, N, device="cuda")), "multiple of ngroups"),
        (dict(state=torch.zeros(batch, H, P, 257, device="cuda"), A=torch.zeros(H, P, 257, device="cuda"),
              B=torch.zeros(batch, G, 257, device="cuda"), C=torch.zeros(batch, G, 257, device="cuda")), "exceeds 256"),
        (dict(state=state.cpu()), "no CPU fallback"),
        (dict(state=state.double()), "unsupported dtype"),
        (dict(state=state[:, :, :1].expand(batch, H, P, N)), "stride-0"),
    ]
    for kw, msg in ssu_cases:
        args = dict(a, state=state)
        args.update(kw)
        with pytest.raises(RuntimeError, match=msg):
            ssu_op()(**args)
    conv_cases = [
        (dict(weight=torch.zeros(8, 5, device="cuda")), "width 5"),
        (dict(weight=torch.zeros(8, 1, device="cuda")), "width 1"),
        (dict(conv_state=torch.zeros(2, 8, 2, device="cuda")), "state_len 2"),
        (dict(conv_state=cs.bfloat16()), "dtype"),
        (dict(conv_state=torch.zeros(2, 7, 4, device="cuda")), "conv_state must be"),
        (dict(weight=torch.zeros(7, 4, device="cuda")), "weight must be"),
        (dict(x=x2.cpu()), "no CPU fallback"),
        (dict(activation="relu"), "activation"),
    ]
    for kw, msg in conv_cases:
        args = dict(x=x2, conv_state=cs, weight=w)
        args.update(kw)
        with pytest.raises(RuntimeError, match=msg):
            conv_update_op()(**args)
    with pytest.raises(NotImplementedError, match="cache_seqlens"):
        conv_update_op()(x2, cs, w, cache_seqlens=torch.zeros(2, dtype=torch.int32, device="cuda"))
    assert _lib.launches() == before


@pytest.mark.gpu
def test_c_entry_point_errors():
    """Bad sizes, dtype codes, NULL pointers, negative strides and dstate > 256 return < 0 with a message and launch nothing."""
    from medical_image_classification_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(1 << 16, device="cuda")
    q = buf.data_ptr()

    def ssu(**kw):
        p = _lib.SsuParams(batch=2, nheads=4, headdim=16, ngroups=2, dstate=32, state=q, x=q, dt=q, A=q, B=q, C=q, out=q)
        for k, v in kw.items():
            if k.endswith("_stride"):
                getattr(p, k)[0] = v
            else:
                setattr(p, k, v)
        return lib.b200_selective_state_update(ctypes.byref(p), None)

    def conv(**kw):
        d = dict(x=q, xd=0, xb=8, xc=1, xl=0, st=q, sb=32, sc=4, sl=1, w=q, wd=0, wc=4, wk=1, b=None, bd=0, bs=1, o=q, ob=8, oc=1,
                 ol=0, B=2, C=8, L=1, S=4, W=4, silu=1)
        d.update(kw)
        return lib.b200_causal_conv1d_update(*d.values(), None)

    before = lib.b200_kernel_launches()
    bad = [(ssu, dict(batch=0), b"batch"), (ssu, dict(nheads=0), b"nheads"), (ssu, dict(headdim=0), b"headdim"),
           (ssu, dict(ngroups=3), b"ngroups"), (ssu, dict(dstate=257), b"dstate"), (ssu, dict(dstate=0), b"dstate"),
           (ssu, dict(state_dtype=5), b"dtype"), (ssu, dict(out_dtype=-1), b"dtype"), (ssu, dict(state=None), b"NULL"),
           (ssu, dict(B=None), b"NULL"), (ssu, dict(state_stride=-1), b"negative"), (ssu, dict(A_stride=-1), b"negative"),
           (conv, dict(W=5), b"width"), (conv, dict(W=1), b"width"), (conv, dict(S=2), b"state_len"), (conv, dict(B=0), b"batch"),
           (conv, dict(C=0), b"dim"), (conv, dict(L=0), b"seqlen"), (conv, dict(xd=3), b"dtype"), (conv, dict(wd=9), b"dtype"),
           (conv, dict(st=None), b"NULL"), (conv, dict(sl=-1), b"negative"), (conv, dict(ob=-8), b"negative")]
    for fn, kw, msg in bad:
        assert fn(**kw) < 0, kw
        assert msg in lib.b200_last_error(), (kw, lib.b200_last_error())
    assert lib.b200_selective_state_update(None, None) < 0
    assert lib.b200_kernel_launches() == before
    assert lib.b200_version() == 4 and lib.b200_sizeof_params(4) == ctypes.sizeof(_lib.SsuParams)
