"""Gradients into initial_states and out of final_states of the SSD chunk scan (mamba_chunk_scan_combined), against the float64
restatement of tests/test_ssd_state_ref.py differentiated by torch.autograd.

Bars as in test_ssd_parity.py: norm-wise relative error 2e-5 (2e-4 for the per-head sums dA / ddt_bias) at precision 0, 5e-3
(5e-2) at precision 1; bf16 I/O rtol 3e-2 / atol 5e-2 against the restatement on the bf16-rounded inputs.

dA and ddt_bias sum b*L*P terms of both signs.  With a final_states gradient, the chunked backward's last-chunk term
dcsQ = <dfin, final_states>, carried to every position of the chunk, contributes |dcsQ| * sum(dt') per (batch, head) to dA
(times |A| to ddt_bias), and the per-position terms cancel most of it, as the chunked forward's derivative does in mamba_ssm.
Their error is therefore measured against the larger of that contribution and the gradient itself.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from test_ssd_parity import CASES, make, rel, to_dev
from test_ssd_state_ref import ssd_ref64
from test_ssd_varlen import ids_from_bounds, segments

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOOSE = ("dA", "ddt_bias")
MODES = ("init", "dfin", "both")
# the parity shapes, and one whose P * N is not a multiple of 4 (the element-wise state-passing kernels)
STATE_CASES = CASES + [(2, 100, 2, 6, 1, 7, 32)]
KEYS = ("x", "dt", "A", "B", "C", "D", "dt_bias")


def scan():
    from medical_image_classification_b200.ssd_combined import mamba_chunk_scan_combined
    return mamba_chunk_scan_combined


def state_inputs(batch, H, P, N, seed):
    r = np.random.RandomState(seed)
    return r.randn(batch, H, P, N).astype(np.float32), r.randn(batch, H, P, N).astype(np.float32)


def init_tensor(init, model_layout, dtype=torch.float32):
    """initial_states as a leaf; in the model layout a transposed view (non-contiguous strides)."""
    t = torch.tensor(init, device="cuda", dtype=dtype)
    if model_layout:
        t = t.transpose(2, 3).contiguous().transpose(2, 3)
    return t.requires_grad_()


def reference(d, dout, dfin=None, init=None, segs=None):
    """Gradients of <dout, out> + <dfin, final_states> of the float64 restatement on the GPU.  segs: per row, the (start, end,
    id) segments of a packed row, each run alone (initial_states for a leading id 0, dfin from the row's last segment)."""
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device="cuda").requires_grad_()
    t = {k: T(d[k]) for k in KEYS}
    ti = T(init) if init is not None else None
    go = torch.tensor(np.asarray(dout), dtype=torch.float64, device="cuda")
    gf = torch.tensor(np.asarray(dfin), dtype=torch.float64, device="cuda") if dfin is not None else None
    batch, L = d["x"].shape[:2]
    segs = segs if segs is not None else [[(0, L, 0)]] * batch
    loss, outs, fins = 0.0, [], []
    for b, row in enumerate(segs):
        parts = []
        for j, (s, e, sid) in enumerate(row):
            sl = (slice(b, b + 1), slice(s, e))
            ini = ti[b:b + 1] if (ti is not None and s == 0 and sid == 0) else None
            o, f = ssd_ref64(t["x"][sl], t["dt"][sl], t["A"], t["B"][sl], t["C"][sl], t["D"], t["dt_bias"], True,
                             (0.0, float("inf")), ini)
            loss = loss + (o * go[sl]).sum()
            parts.append(o)
            if j == len(row) - 1:
                fins.append(f)
                if gf is not None:
                    loss = loss + (f * gf[b:b + 1]).sum()
        outs.append(torch.cat(parts, 1))
    loss.backward()
    npy = lambda a: a.detach().cpu().numpy()
    g = {"d" + k: npy(v.grad) for k, v in t.items()}
    if ti is not None:
        g["dinit"] = npy(ti.grad) if ti.grad is not None else np.zeros_like(init)
    return npy(torch.cat(outs)), npy(torch.cat(fins)), g


def run_kernels(d, chunk, model_layout, dout, dfin=None, init=None, seq_idx=None, dtype=torch.float32, init_dtype=torch.float32):
    t = {k: to_dev(d[k], model_layout, dtype if k in ("x", "dt", "B", "C") else torch.float32) for k in KEYS}
    ti = init_tensor(init, model_layout, init_dtype) if init is not None else None
    si = torch.tensor(seq_idx, device="cuda", dtype=torch.int32) if seq_idx is not None else None
    out, fin = scan()(t["x"], t["dt"], t["A"], t["B"], t["C"], chunk, D=t["D"], dt_bias=t["dt_bias"], initial_states=ti, seq_idx=si,
                      dt_softplus=True, return_final_states=True)
    assert fin.requires_grad
    outs, grads = ([out], [torch.tensor(dout, device="cuda", dtype=out.dtype)]) if dout is not None else ([], [])
    if dfin is not None:
        outs.append(fin)
        grads.append(torch.tensor(dfin, device="cuda"))
    torch.autograd.backward(outs, grads)
    g = {"d" + k: v.grad for k, v in t.items()}
    if ti is not None:
        assert ti.grad is not None and ti.grad.dtype == init_dtype and ti.grad.shape == ti.shape
        g["dinit"] = ti.grad
    return out, fin, g


def errors(got, want):
    out, fin, g = got
    rout, rfin, rg = want
    errs = dict(out=rel(out, rout), fin=rel(fin, rfin))
    errs.update({k: rel(v, rg[k]) for k, v in g.items()})
    return errs


def with_state_scale(errs, got, want, d, dfin, chunk):
    """Re-measure dA / ddt_bias against max(|gradient|, max_h sum_b |dcsQ_b,h| sum_{l in last chunk} dt'_b,l,h (* |A_h|))."""
    if dfin is None:
        return errs
    _, rfin, rg = want
    v = d["dt"].astype(np.float64) + d["dt_bias"]
    v = np.where(v > 20.0, v, np.log1p(np.exp(np.minimum(v, 20.0))))
    L = v.shape[1]
    last = v[:, (L - 1) // chunk * chunk:].sum(1)                                         # (b, h)
    term = (np.abs(np.einsum("bhpn,bhpn->bh", dfin, rfin)) * last).sum(0)               # (h)
    for k, w in (("dA", term), ("ddt_bias", term * np.abs(d["A"]))):
        a = got[2][k].detach().float().cpu().numpy()
        errs[k] = float(np.abs(a - rg[k]).max() / max(np.abs(rg[k]).max(), w.max()))
    return errs


def check(errs, bar=2e-5):
    print(" ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert all(v < (10 * bar if k in LOOSE else bar) for k, v in errs.items()), errs


def case_inputs(case, mode, seed_extra=0):
    batch, L, H, P, G, N, chunk = case
    d = make(batch, L, H, P, G, N, seed=L + N + seed_extra)
    init, dfin = state_inputs(batch, H, P, N, seed=L + 2 * N + seed_extra)
    return d, (init if mode in ("init", "both") else None), (dfin if mode in ("dfin", "both") else None)


# ---- 1. against the float64 restatement ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("model_layout", [True, False])
@pytest.mark.parametrize("case", STATE_CASES)
def test_state_grads_match_fp64_reference(case, model_layout, mode):
    d, init, dfin = case_inputs(case, mode)
    want = reference(d, d["dout"], dfin, init)
    got = run_kernels(d, case[-1], model_layout, d["dout"], dfin, init)
    check(with_state_scale(errors(got, want), got, want, d, dfin, case[-1]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", STATE_CASES)
def test_state_grads_tf32_mode(case):
    from medical_image_classification_b200 import ssd_combined
    d, init, dfin = case_inputs(case, "both", seed_extra=1)
    want = reference(d, d["dout"], dfin, init)
    ssd_combined.set_precision(1)
    try:
        got = run_kernels(d, case[-1], True, d["dout"], dfin, init)
    finally:
        ssd_combined.set_precision(None)
    errs = errors(got, want)
    # dA / ddt_bias are printed, not asserted: single-pass TF32 products (relative error ~1e-3) on their cancelling terms leave
    # them beyond 5e-2 at some shapes with state gradients; the precision-0 tests above hold them to 2e-4
    print("per-head sums:", {k: f"{errs.pop(k):.2e}" for k in LOOSE})
    check(errs, bar=5e-3)


@pytest.mark.gpu
def test_state_grads_bf16_io():
    """bf16 x / dt / B / C and a bf16 initial_states: its gradient comes back bf16.  ddt, dA and ddt_bias are not compared
    element-wise: the backward derives d(cumsum) from the stored forward output, which is bf16 here, as on the default path."""
    case = (2, 130, 4, 32, 2, 24, 64)
    d, init, dfin = case_inputs(case, "both", seed_extra=2)
    rb = lambda a: torch.tensor(a).bfloat16().float().numpy()
    db = dict(d, x=rb(d["x"]), dt=rb(d["dt"]), B=rb(d["B"]), C=rb(d["C"]))
    out, fin, g = run_kernels(d, 64, True, d["dout"], dfin, rb(init), dtype=torch.bfloat16, init_dtype=torch.bfloat16)
    assert out.dtype == torch.bfloat16 and g["dinit"].dtype == torch.bfloat16
    rout, rfin, rg = reference(db, rb(d["dout"]), dfin, rb(init))
    f = lambda a: a.detach().float().cpu().numpy()
    assert np.allclose(f(out), rout, rtol=3e-2, atol=5e-2) and np.allclose(f(fin), rfin, rtol=3e-2, atol=5e-2)
    for k, v in g.items():
        if k not in ("ddt", "dA", "ddt_bias"):
            assert np.allclose(f(v), rg[k], rtol=3e-2, atol=5e-2), k
    assert rel(g["ddt"], rg["ddt"]) < 3e-2


# ---- 2. the mma.sync engine --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_mma_sync_engine_in_child_process():
    """B200_SSD_TC is read once per process: the matrix above runs again in a child with the mma.sync tiles."""
    env = dict(os.environ, B200_SSD_TC="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", os.path.abspath(__file__), "-k",
                        "test_state_grads_match_fp64_reference or test_state_grads_tf32_mode or test_chained or test_packed"],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and " skipped" not in r.stdout, r.stdout[-500:]


# ---- 3. chained calls equal one call ------------------------------------------------------------------------------------------
def _leaves(d, model_layout):
    return {k: to_dev(d[k], model_layout) for k in KEYS}


def _chain(t, cuts, chunk, init=None):
    """Outputs of consecutive calls over [cuts[i], cuts[i+1]), each starting from the previous call's final_states."""
    outs, state = [], init
    for s, e in zip(cuts[:-1], cuts[1:]):
        out, state = scan()(t["x"][:, s:e], t["dt"][:, s:e], t["A"], t["B"][:, s:e], t["C"][:, s:e], chunk, D=t["D"],
                            dt_bias=t["dt_bias"], initial_states=state, dt_softplus=True, return_final_states=True)
        outs.append(out)
    return torch.cat(outs, 1), state


@pytest.mark.gpu
@pytest.mark.parametrize("model_layout", [True, False])
@pytest.mark.parametrize("cuts,learned_init", [((0, 100, 300), False), ((0, 77, 200, 300), True), ((0, 256, 300), False)],
                         ids=["two", "three_learned_init", "two_on_chunk_edge"])
def test_chained_calls_equal_one_call(cuts, learned_init, model_layout):
    chunk, batch, L, H, P, G, N = 128, 2, 300, 4, 64, 2, 40
    d = make(batch, L, H, P, G, N, seed=21)
    init, dfin = state_inputs(batch, H, P, N, seed=22)
    one, many = _leaves(d, model_layout), _leaves(d, model_layout)
    i1 = init_tensor(init, model_layout) if learned_init else None
    i2 = init_tensor(init, model_layout) if learned_init else None
    out1, fin1 = _chain(one, (0, L), chunk, i1)
    out2, fin2 = _chain(many, cuts, chunk, i2)
    g, gf = torch.tensor(d["dout"], device="cuda"), torch.tensor(dfin, device="cuda")
    torch.autograd.backward([out1, fin1], [g, gf])
    torch.autograd.backward([out2, fin2], [g, gf])
    errs = dict(out=rel(out2, out1.detach().cpu().numpy()), fin=rel(fin2, fin1.detach().cpu().numpy()))
    errs.update({"d" + k: rel(many[k].grad, one[k].grad.cpu().numpy()) for k in KEYS})
    if learned_init:
        errs["dinit"] = rel(i2.grad, i1.grad.cpu().numpy())
    check(errs)


# ---- 4. packed rows -------------------------------------------------------------------------------------------------------------
PACKED_L, PACKED_Q = 300, 64
PACKED_ROWS = [
    ids_from_bounds(PACKED_L, [40, 64, 150], first=1),            # first id not 0: no initial_states gradient at all
    ids_from_bounds(PACKED_L, [10, 64, 170]),                     # id changes inside chunk 0, on a chunk edge, mid-chunk
    ids_from_bounds(PACKED_L, [128, 200, 299]) + np.where(np.arange(PACKED_L) >= 200, 1, 0),   # an empty segment (id 2), last of length 1
    ids_from_bounds(PACKED_L, [256]),                             # last segment starts on a chunk edge, first spans four chunks
]


@pytest.mark.gpu
@pytest.mark.parametrize("model_layout", [True, False])
@pytest.mark.parametrize("mode", MODES)
def test_packed_rows_state_grads(mode, model_layout):
    seq_idx = np.stack(PACKED_ROWS)
    batch, H, P, G, N = len(PACKED_ROWS), 4, 32, 1, 24
    d = make(batch, PACKED_L, H, P, G, N, seed=31)
    init, dfin = state_inputs(batch, H, P, N, seed=32)
    init = init if mode in ("init", "both") else None
    dfin = dfin if mode in ("dfin", "both") else None
    got = run_kernels(d, PACKED_Q, model_layout, d["dout"], dfin, init, seq_idx=seq_idx)
    segs = [segments(r) for r in seq_idx]
    want = reference(d, d["dout"], dfin, init, segs=segs)
    check(with_state_scale(errors(got, want), got, want, d, dfin, PACKED_Q))
    if init is not None:
        assert not got[2]["dinit"][0].any()                        # exactly zero: row 0 starts with id 1
        assert got[2]["dinit"][1:].abs().amax((1, 2, 3)).min() > 0


# ---- 5. the path the models run --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", [CASES[0], CASES[5]])
def test_unused_final_states_runs_the_default_backward(case):
    """A returned final_states that takes no part in the loss reaches backward as None: the same launches, and the same dx / dB / dC
    bit for bit.  ddt, dA, dD and ddt_bias sum atomically accumulated partials, whose order varies from run to run, so they are
    compared at that spread (up to 2e-6 of their largest magnitude between two runs of the same code)."""
    from medical_image_classification_b200 import _lib
    batch, L, H, P, G, N, chunk = case
    d = make(batch, L, H, P, G, N, seed=41)
    res = []
    for ret in (False, True):
        t = _leaves(d, True)
        r = scan()(t["x"], t["dt"], t["A"], t["B"], t["C"], chunk, D=t["D"], dt_bias=t["dt_bias"], dt_softplus=True,
                   return_final_states=ret)
        out = r[0] if ret else r
        torch.cuda.synchronize()
        n0 = _lib.launches()
        out.backward(torch.tensor(d["dout"], device="cuda"))
        torch.cuda.synchronize()
        res.append((_lib.launches() - n0, {k: v.grad.clone() for k, v in t.items()}))
    (n_off, g_off), (n_on, g_on) = res
    assert n_on == n_off
    for k in ("x", "B", "C"):
        assert torch.equal(g_on[k], g_off[k]), k
    for k in ("dt", "A", "D", "dt_bias"):
        assert rel(g_on[k], g_off[k].cpu().numpy()) < 1e-5, k


@pytest.mark.gpu
def test_state_grads_launch_the_same_kernels():
    """Asking for the state gradients changes what the backward's kernels compute, not which kernels run."""
    from medical_image_classification_b200 import _lib
    case = CASES[3]
    counts = []
    for mode in (None,) + MODES:
        d, init, dfin = case_inputs(case, mode or "init")
        if mode is None:
            init = None
        t = _leaves(d, True)
        ti = init_tensor(init, True) if init is not None else None
        out, fin = scan()(t["x"], t["dt"], t["A"], t["B"], t["C"], case[-1], D=t["D"], dt_bias=t["dt_bias"], initial_states=ti,
                          dt_softplus=True, return_final_states=True)
        outs, grads = [out], [torch.tensor(d["dout"], device="cuda")]
        if dfin is not None:
            outs.append(fin)
            grads.append(torch.tensor(dfin, device="cuda"))
        torch.cuda.synchronize()
        n0 = _lib.launches()
        torch.autograd.backward(outs, grads)
        torch.cuda.synchronize()
        counts.append(_lib.launches() - n0)
    assert len(set(counts)) == 1, counts


@pytest.mark.gpu
def test_loss_on_final_states_only_and_varlen_states_stay_non_differentiable():
    case = CASES[0]
    d, init, dfin = case_inputs(case, "both")
    out, fin, g = run_kernels(d, case[-1], False, None, dfin, init)     # out's gradient arrives as None
    want = reference(d, np.zeros_like(d["dout"]), dfin, init)
    check(errors((out, fin, g), want))
    t = {k: torch.tensor(v, device="cuda") for k, v in make(1, 64, 2, 8, 1, 8, seed=1).items()}
    _, vs = scan()(t["x"], t["dt"], t["A"], t["B"], t["C"], 32, seq_idx=torch.zeros(1, 64, dtype=torch.int32, device="cuda"),
                   cu_seqlens=torch.tensor([0, 64], device="cuda"), return_varlen_states=True)
    assert not vs.requires_grad


# ---- 6. the C ABI ---------------------------------------------------------------------------------------------------------------------
def _bwd_params(batch=1, L=64, H=2, P=8, G=1, N=8, Q=32):
    from medical_image_classification_b200 import _lib
    q = _lib.SsdBwdParams()
    p = q.f
    p.batch, p.seqlen, p.nheads, p.headdim, p.n_groups, p.dstate, p.chunk_size = batch, L, H, P, G, N, Q
    p.x = p.dt = p.A = p.B = p.C = p.out = 16
    p.workspace = 256
    q.dout = q.dx = q.ddt = q.dB = q.dC = q.dA = q.scratch = 256
    return q


def test_c_entry_point_refuses_state_grads_without_their_inputs():
    """Checked before any launch: an error code, a message, and nothing launched."""
    from medical_image_classification_b200 import _lib
    lib = _lib.load()
    n0 = _lib.launches()
    q = _bwd_params()
    q.dfinal_states = 512
    assert lib.b200_ssd_bwd(ctypes.byref(q), None) != 0
    assert b"final_states" in lib.b200_last_error()
    q = _bwd_params()
    q.dinitial_states = 512
    assert lib.b200_ssd_bwd(ctypes.byref(q), None) != 0
    assert b"initial_states" in lib.b200_last_error()
    assert _lib.launches() == n0


@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 1], ids=["aligned", "unaligned"])
def test_dinitial_states_written_exactly_within_its_shape(offset):
    """Through the C ABI, dfinal_states and dinitial_states in NaN-filled buffers at an offset of 0 or 1 float (the vector
    or the element-wise state-passing kernel): dinitial_states is written exactly within (batch, H, P, N), the reads of
    dfinal_states stop at its end, and both paths give the restatement's gradient."""
    from medical_image_classification_b200 import _lib, ssd_combined
    batch, L, H, P, G, N, Q = 2, 100, 2, 16, 1, 12, 32
    d = make(batch, L, H, P, G, N, seed=51)
    init, dfin = state_inputs(batch, H, P, N, seed=52)
    t = {k: torch.tensor(d[k], device="cuda") for k in KEYS + ("dout",)}
    ti = torch.tensor(init, device="cuda")
    n = batch * H * P * N
    out = torch.empty_like(t["x"])
    fin = torch.empty(batch, H, P, N, device="cuda")
    ws = torch.empty(_lib.load().b200_ssd_workspace_bytes(batch, L, H, P, G, N, Q) // 4, device="cuda")
    p = _lib.SsdFwdParams()
    ssd_combined._fill_fwd(p, t["x"], t["dt"], t["A"], t["B"], t["C"], t["D"], t["dt_bias"], Q, True, (0.0, float("inf")), ti, 0, None)
    p.out_stride[:] = list(out.stride())
    p.out, p.final_states, p.workspace = out.data_ptr(), fin.data_ptr(), ws.data_ptr()
    _lib.launch("b200_ssd_fwd", t["x"].device, ctypes.byref(p))
    dinit_buf = torch.full((n + 8,), float("nan"), device="cuda")
    dfin_buf = torch.full((n + 8,), float("nan"), device="cuda")
    dfin_buf[offset:offset + n] = torch.tensor(dfin, device="cuda").flatten()
    grads = {k: torch.empty_like(t[k]) for k in ("x", "dt", "B", "C")}
    dA, dD, dbias = (torch.zeros(H, device="cuda") for _ in range(3))
    q = _lib.SsdBwdParams()
    q.f = p
    q.dout_stride[:] = list(t["dout"].stride())
    q.dout = t["dout"].data_ptr()
    q.dx, q.ddt, q.dB, q.dC = (grads[k].data_ptr() for k in ("x", "dt", "B", "C"))
    q.dA, q.dD, q.ddt_bias = dA.data_ptr(), dD.data_ptr(), dbias.data_ptr()
    scratch = torch.empty(_lib.load().b200_ssd_bwd_scratch_bytes(batch, L, H, P, G, N, Q) // 4, device="cuda")
    q.scratch = scratch.data_ptr()
    q.final_states, q.dfinal_states = fin.data_ptr(), dfin_buf[offset:].data_ptr()
    q.dinitial_states = dinit_buf[offset:].data_ptr()
    _lib.launch("b200_ssd_bwd", t["x"].device, ctypes.byref(q))
    torch.cuda.synchronize()
    assert torch.isnan(dinit_buf[:offset]).all() and torch.isnan(dinit_buf[offset + n:]).all()
    dinit = dinit_buf[offset:offset + n].view(batch, H, P, N)
    assert torch.isfinite(dinit).all()
    _, _, rg = reference(d, d["dout"], dfin, init)
    check(dict(dinit=rel(dinit, rg["dinit"]), dx=rel(grads["x"], rg["dx"]), ddt=rel(grads["dt"], rg["ddt"]), dA=rel(dA, rg["dA"])))
