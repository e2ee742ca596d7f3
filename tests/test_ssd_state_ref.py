"""A float64 restatement of the SSD recurrence, written with differentiable torch ops, so that torch.autograd gives every
gradient of mamba_chunk_scan_combined, including those into initial_states and out of final_states, which the C oracle
(oracle/ssd_oracle.c) does not produce.  tests/test_ssd_state_grads.py checks the kernels against it.

The CPU tests below pin the restatement to the C oracle wherever both define a result (out, final_states, and every
gradient of a loss on out), and check its initial_states gradient against a closed form.
"""
import numpy as np
import pytest
import torch

import oracle


def ssd_ref64(x, dt, A, B, C, D=None, dt_bias=None, dt_softplus=True, dt_limit=(0.0, float("inf")), initial_states=None):
    """float64 tensors x (b,l,h,p), dt (b,l,h), A (h), B/C (b,l,g,n), D (h), dt_bias (h), initial_states (b,h,p,n).
    Returns (out, final_states), evaluated token by token:

        dt'_t = clamp(softplus?(dt_t + dt_bias)),  S_t = exp(dt'_t A) S_{t-1} + dt'_t x_t (outer) B_t,  y_t = S_t C_t + D x_t"""
    batch, L, H, P = x.shape
    G = B.shape[2]
    v = dt + dt_bias if dt_bias is not None else dt
    if dt_softplus:
        v = torch.where(v > 20.0, v, torch.log1p(torch.exp(torch.clamp(v, max=20.0))))
    v = torch.clamp(v, dt_limit[0], dt_limit[1])
    Bh, Ch = B.repeat_interleave(H // G, dim=2), C.repeat_interleave(H // G, dim=2)
    S = initial_states if initial_states is not None else x.new_zeros(batch, H, P, B.shape[3])
    ys = []
    for t in range(L):
        a = torch.exp(v[:, t] * A)
        S = a[:, :, None, None] * S + (v[:, t, :, None] * x[:, t])[..., None] * Bh[:, t, :, None, :]
        ys.append(torch.einsum("bhpn,bhn->bhp", S, Ch[:, t]))
    out = torch.stack(ys, 1)
    if D is not None:
        out = out + x * D[:, None]
    return out, S


def ref_grads(d, dout, dfin=None, init=None, dt_softplus=True, dt_limit=(0.0, float("inf")), device="cpu"):
    """(out, final_states, grads) of ssd_ref64 for the loss <dout, out> + <dfin, final_states>; numpy in, numpy out.
    grads has dx, ddt, dA, dB, dC, dD, ddt_bias and, when init is given, dinit."""
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=device).requires_grad_()
    t = {k: T(d[k]) for k in ("x", "dt", "A", "B", "C", "D", "dt_bias")}
    ti = T(init) if init is not None else None
    out, fin = ssd_ref64(t["x"], t["dt"], t["A"], t["B"], t["C"], t["D"], t["dt_bias"], dt_softplus, dt_limit, ti)
    loss = (out * torch.tensor(np.asarray(dout), dtype=torch.float64, device=device)).sum()
    if dfin is not None:
        loss = loss + (fin * torch.tensor(np.asarray(dfin), dtype=torch.float64, device=device)).sum()
    loss.backward()
    npy = lambda a: a.detach().cpu().numpy()
    g = {"d" + k: npy(v.grad) for k, v in t.items()}
    if ti is not None:
        g["dinit"] = npy(ti.grad)
    return npy(out), npy(fin), g


def _inputs(batch, L, H, P, G, N, seed, dt_scale=0.5):
    r = np.random.RandomState(seed)
    f = lambda *s: r.randn(*s).astype(np.float32)
    return dict(x=f(batch, L, H, P), dt=(dt_scale * r.rand(batch, L, H) - 0.1).astype(np.float32), A=(-0.5 - r.rand(H)).astype(np.float32),
                B=f(batch, L, G, N), C=f(batch, L, G, N), D=f(H), dt_bias=(0.3 * r.rand(H)).astype(np.float32),
                init=f(batch, H, P, N), dout=f(batch, L, H, P), dfin=f(batch, H, P, N))


def _rel(a, b):
    return float(np.abs(np.asarray(a, np.float64) - b).max() / max(np.abs(b).max(), 1e-30))


# (softplus, dt_limit): dt in [-0.1, 0.4) without softplus so that a (0, 0.3) limit clamps both ends
OPTIONS = [(True, (0.0, float("inf"))), (False, (0.0, float("inf"))), (True, (0.75, 0.9)), (False, (0.0, 0.3))]


@pytest.mark.parametrize("softplus,limit", OPTIONS)
@pytest.mark.parametrize("with_init", [False, True])
def test_restatement_matches_c_oracle(softplus, limit, with_init):
    d = _inputs(2, 37, 4, 3, 2, 5, seed=int(softplus) + 2 * int(with_init) + 7 * int(limit[0] * 100))
    init = d["init"] if with_init else None
    kw = dict(D=d["D"], dt_bias=d["dt_bias"], dt_softplus=softplus, dt_limit=limit, initial_states=init)
    ref, rfin = oracle.ssd_fwd(d["x"], d["dt"], d["A"], d["B"], d["C"], **kw)
    g = oracle.ssd_bwd(d["x"], d["dt"], d["A"], d["B"], d["C"], dout=d["dout"], **kw)
    out, fin, r = ref_grads(d, d["dout"], init=init, dt_softplus=softplus, dt_limit=limit)
    errs = dict(out=_rel(ref, out), fin=_rel(rfin, fin))
    errs.update({k: _rel(g[k], r[k]) for k in ("dx", "ddt", "dA", "dB", "dC", "dD", "ddt_bias")})
    assert all(v < 2e-6 for v in errs.values()), errs


@pytest.mark.parametrize("softplus,limit", OPTIONS)
def test_initial_states_gradient_closed_form(softplus, limit):
    """S_{-1} reaches y_t as exp(A sum_{s<=t} dt'_s) C_t and the final state as exp(A sum_s dt'_s): dinit[b,h,p,n] =
    sum_t dout[b,t,h,p] C[b,t,g,n] exp(A_h cs_t) + dfin[b,h,p,n] exp(A_h cs_{L-1})."""
    batch, L, H, P, G, N = 2, 29, 4, 3, 2, 5
    d = _inputs(batch, L, H, P, G, N, seed=3)
    _, _, r = ref_grads(d, d["dout"], dfin=d["dfin"], init=d["init"], dt_softplus=softplus, dt_limit=limit)
    v = d["dt"].astype(np.float64) + d["dt_bias"]
    if softplus:
        v = np.where(v > 20.0, v, np.log1p(np.exp(np.minimum(v, 20.0))))
    v = np.clip(v, limit[0], limit[1])
    cs = np.cumsum(v, axis=1) * d["A"]                                   # (b, l, h)
    Ch = np.repeat(d["C"].astype(np.float64), H // G, axis=2)             # (b, l, h, n)
    want = np.einsum("blhp,blhn,blh->bhpn", d["dout"], Ch, np.exp(cs)) + d["dfin"] * np.exp(cs[:, -1])[:, :, None, None]
    assert _rel(r["dinit"], want) < 1e-12


def test_final_states_gradient_equals_appended_readout():
    """<dfin, S_{L-1}> as a loss equals the output of N extra tokens with dt' = 0 (no decay, no input), C = e_n and
    dout = dfin[..., n]: the restatement's gradients for a final-state loss match those of that output loss."""
    batch, L, H, P, G, N = 1, 23, 2, 3, 1, 4
    d = _inputs(batch, L, H, P, G, N, seed=5)
    _, _, r = ref_grads(d, d["dout"], dfin=d["dfin"], init=d["init"], dt_softplus=False)
    e = dict(d)
    e["x"] = np.concatenate([d["x"], np.zeros((batch, N, H, P), np.float32)], 1)
    e["dt"] = np.concatenate([d["dt"], np.full((batch, N, H), -d["dt_bias"][None, None] - 1.0, np.float32)], 1)  # clamps to 0
    e["B"] = np.concatenate([d["B"], np.zeros((batch, N, G, N), np.float32)], 1)
    e["C"] = np.concatenate([d["C"], np.broadcast_to(np.eye(N, dtype=np.float32)[None, :, None], (batch, N, G, N))], 1)
    dout = np.concatenate([d["dout"], np.moveaxis(d["dfin"], 3, 1)], 1)     # token L + n reads dfin[..., n]
    _, _, s = ref_grads(e, dout, init=d["init"], dt_softplus=False)
    for k in ("dinit", "dA", "dD", "ddt_bias", "dB", "dC", "ddt", "dx"):
        b = s[k][:, :L] if k in ("dB", "dC", "ddt", "dx") else s[k]
        assert _rel(r[k], b) < 1e-12, k
