"""Model-level parity of the BENCHMARKED configuration (VERDICT r1, row x1; north_star: "a stated bf16 tolerance for both
activations and gradients, equal top-1 on a fixed synthetic eval batch").

bench.py trains MedMamba-T under torch.autocast(bfloat16): bf16 Linear / conv / residual stream, TF32 folded x_proj / dt_proj,
fp32 selective scan (as the reference calls it, MedMamba.py:403-418).  The reference itself trains in fp32
(train.py:40,59-60).  Golden = the UNMODIFIED reference VSSM at MedMamba-T's real widths (dims 96-768, d_state 16, 224 x 224,
depths 1-1-1-1, batch 4) in fp32 on CPU (tests/golden/medmamba_real_dims.npz, oracle/make_golden.py::medmamba_real_dims_case;
weights = the product model's seeded CPU initialisation, re-created here and checked by checksum).

Stated tolerances (norm-wise relative error max|a - b| / max|b| unless noted):
  fp32 product vs fp32 reference : logits 1e-4, loss 1e-5, every parameter gradient: cosine >= 0.9999 on the stored samples
  bf16-autocast product (the bench's code path, entered exactly as bench.py::fwd_bwd_opt does) vs fp32 reference:
      logits rtol 3e-2 / atol 5e-2 -- the reference's own bf16 bar (test_selective_scan.py:398-400);
      equal top-1 on the eval batch; loss within 2e-2; parameter gradients: global cosine >= 0.99, per-parameter cosine >= 0.95
      for every parameter whose gradient norm is above 1e-3 of the largest (bf16 keeps 8 bits: this is what 8 bits give, measured
      values are printed with -s and recorded in DESIGN.md)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

KW = dict(num_classes=6, depths=[1, 1, 1, 1], dims=[96, 192, 384, 768], drop_path_rate=0.0)


def _sample(t, n=4096):
    f = t.detach().flatten()
    if f.numel() <= n:
        return f.float().cpu().numpy()
    return f[torch.arange(0, f.numel(), f.numel() // n, device=f.device)[:n]].float().cpu().numpy()


def _setup():
    from medical_image_classification_b200.models import VSSM
    g = np.load(os.path.join(GOLDEN, "medmamba_real_dims.npz"))
    torch.manual_seed(int(g["seed"]))
    net = VSSM(**KW)                                    # CPU init, the same RNG stream the golden script consumed
    chk = np.array([float(sum(p.double().sum() for p in net.parameters())), float(sum(p.double().abs().sum() for p in net.parameters()))])
    assert np.allclose(chk, g["param_checksum"], rtol=1e-9), "seeded initialisation differs from the one the goldens were made with"
    gen = torch.Generator().manual_seed(int(g["seed"]) + 1)
    x = torch.randn(4, 3, 224, 224, generator=gen)
    y = torch.randint(0, 6, (4,), generator=gen)
    assert np.array_equal(y.numpy(), g["y"])
    return net.cuda(), x.cuda(), y.cuda(), g


def _cos(a, b):
    a, b = a.astype(np.float64).ravel(), b.astype(np.float64).ravel()
    return float(a @ b / max(np.linalg.norm(a) * np.linalg.norm(b), 1e-300))


def _grad_report(net, g):
    names = [k for k, p in net.named_parameters() if p.grad is not None and "grad." + k in g.files]
    gmax = max(float(g["gnorm." + k]) for k in names)
    cos, allg, allr = {}, [], []
    for k, p in net.named_parameters():
        if k in names:
            got, ref = _sample(p.grad), g["grad." + k]
            allg.append(got); allr.append(ref)
            if float(g["gnorm." + k]) > 1e-3 * gmax:
                cos[k] = _cos(got, ref)
    return cos, _cos(np.concatenate(allg), np.concatenate(allr)), len(names)


@pytest.fixture
def strict_fp32():
    """cuDNN convolutions default to TF32 on this hardware (torch.backends.cudnn.allow_tf32): switch it off for the fp32 bar."""
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev


def test_fp32_model_matches_reference(strict_fp32):
    net, x, y, g = _setup()
    net.eval()
    with torch.no_grad():
        le = net(x).float().cpu().numpy()
    assert np.abs(le - g["logits_eval"]).max() / np.abs(g["logits_eval"]).max() < 1e-4
    assert np.array_equal(le.argmax(-1), g["logits_eval"].argmax(-1))
    net.train()
    logits = net(x)
    loss = torch.nn.functional.cross_entropy(logits.float(), y)
    loss.backward()
    assert np.abs(logits.detach().cpu().numpy() - g["logits_train"]).max() / np.abs(g["logits_train"]).max() < 1e-4
    assert abs(float(loss) - float(g["loss"])) < 1e-5 * max(1.0, abs(float(g["loss"])))
    cos, cos_all, n = _grad_report(net, g)
    worst = min(cos, key=cos.get)
    print(f"fp32: {n} parameters, global grad cosine {cos_all:.7f}, worst per-parameter cosine {cos[worst]:.7f} ({worst})")
    assert n > 60 and cos_all > 0.99999 and cos[worst] > 0.9999, (cos_all, worst, cos[worst])


def test_bf16_autocast_model_matches_reference():
    """The bench's code path: bench.py::fwd_bwd_opt -- forward and loss inside torch.autocast(bfloat16), backward outside."""
    net, x, y, g = _setup()
    net.eval()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        le = net(x).float().cpu().numpy()
    ref = g["logits_eval"]
    assert np.all(np.abs(le - ref) <= 5e-2 + 3e-2 * np.abs(ref)), np.abs(le - ref).max()
    assert np.array_equal(le.argmax(-1), ref.argmax(-1)), "top-1 differs on the fixed synthetic eval batch"
    net.train()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        logits = net(x)
        loss = torch.nn.functional.cross_entropy(logits.float(), y)
    loss.backward()
    lt, rt = logits.detach().float().cpu().numpy(), g["logits_train"]
    assert np.all(np.abs(lt - rt) <= 5e-2 + 3e-2 * np.abs(rt)), np.abs(lt - rt).max()
    assert abs(float(loss) - float(g["loss"])) < 2e-2
    cos, cos_all, n = _grad_report(net, g)
    worst = min(cos, key=cos.get)
    print(f"bf16 autocast: eval logits max |err| {np.abs(le - ref).max():.2e}, train logits max |err| {np.abs(lt - rt).max():.2e}, "
          f"loss err {abs(float(loss) - float(g['loss'])):.2e}, global grad cosine {cos_all:.5f}, "
          f"worst per-parameter cosine {cos[worst]:.5f} ({worst}) over {len(cos)} parameters")
    assert cos_all > 0.99 and cos[worst] > 0.95, (cos_all, worst, cos[worst])


def test_backward_inside_autocast_region_is_safe():
    """ADVICE r1: loss.backward() called INSIDE the autocast block runs the custom backwards under autocast; the ctypes-backed
    Functions must not hand re-cast (bf16) buffers to fp32 kernels.  Gradients must equal the backward-outside run up to the order
    of the fp32 atomics, and meet the bf16 bars against the fp32 reference golden.  The two runs are compared by direction
    (cosine) rather than element by element: under bf16 autocast a last-bit difference from the atomics can flip one bf16
    rounding downstream and move single elements by ~2^-8 of their magnitude, while a mis-cast buffer scrambles whole tensors."""
    net, x, y, g = _setup()
    net.train()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss = torch.nn.functional.cross_entropy(net(x).float(), y)
    loss.backward()
    ref = {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None}
    net.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss2 = torch.nn.functional.cross_entropy(net(x).float(), y)
        loss2.backward()
    assert set(ref) == {k for k, p in net.named_parameters() if p.grad is not None}
    nmax = max(float(v.float().norm()) for v in ref.values())
    cos, allg, allr = {}, [], []
    for k, p in net.named_parameters():
        if p.grad is None:
            continue
        assert torch.isfinite(p.grad).all(), k
        a, b = p.grad.float().cpu().numpy(), ref[k].float().cpu().numpy()
        allg.append(a.ravel()); allr.append(b.ravel())
        if float(ref[k].float().norm()) > 1e-3 * nmax:
            cos[k] = _cos(a, b)
    worst = min(cos, key=cos.get)
    cos_all = _cos(np.concatenate(allg), np.concatenate(allr))
    gcos, gcos_all, n = _grad_report(net, g)
    gworst = min(gcos, key=gcos.get)
    print(f"backward inside vs outside autocast: global grad cosine {cos_all:.7f}, worst per-parameter cosine {cos[worst]:.7f} ({worst}) "
          f"over {len(cos)} parameters; vs the fp32 golden: global {gcos_all:.5f}, worst {gcos[gworst]:.5f} ({gworst})")
    # same kernels, same inputs: only the order of the fp32 atomics differs between the two runs
    assert cos_all > 0.99999 and cos[worst] > 0.999, (cos_all, worst, cos[worst])
    assert n > 60 and gcos_all > 0.99 and gcos[gworst] > 0.95, (gcos_all, gworst, gcos[gworst])
