"""The fused Mamba-2 mixer (mamba_split_conv1d_scan_combined) against the same steps composed, CUDA events.

Shapes: a Mamba-2-130m-like layer (d_model 768: dim 1536, 24 heads of 64, d_state 128, width 4, L 2048, batch 8) and MedSSD's four
SS2D_with_SSD stages flattened to 1-D (d_model 96 / 192 / 384 / 768: dim 192 / 384 / 768 / 1536, heads of 64, d_state 128, width 3,
L 3136 / 784 / 196 / 49, batch 64).  Everything runs under bf16 autocast (zxbcdt bf16, parameters fp32, single-pass TF32 SSD), with
a gated RMSNorm (norm after the gate) and out_proj, as transformers' Mamba2Mixer calls the operator.  Per shape, forward + backward
time (best of several rounds, arms alternated), the memory held from the forward to the backward (output and saved tensors: what a
stack of layers accumulates) and the peak memory of one forward + backward, both above the inputs, of
  fused     mamba_split_conv1d_scan_combined
  composed  causal_conv1d_fn -> mamba_chunk_scan_combined -> rmsnorm_fn -> F.linear
  torchconv the same with nn.Conv1d + SiLU in place of causal_conv1d_fn
and the conv kernels alone (b200_causal_conv1d_fwd / _bwd) in GB/s of the bytes they must move (computed from the shapes below),
next to the device-to-device copy rate measured in the same run.  Each timed pass cycles over enough input sets to exceed the 126 MB
L2.  Prints one JSON line per shape, then the copy rate, the device name and its power limit.

    python tools/bench_split_conv1d.py [--iters N] [--rounds R]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from medical_image_classification_b200.conv1d import causal_conv1d_fn, conv_bwd, conv_fwd  # noqa: E402
from medical_image_classification_b200.ssd_combined import (mamba_chunk_scan_combined, mamba_split_conv1d_scan_combined,  # noqa: E402
                                                            rmsnorm_fn)

dev = "cuda"
L2_BYTES = 126 << 20
# (name, batch, L, d_model, headdim, d_state, width)
SHAPES = [("mamba2-130m", 8, 2048, 768, 64, 128, 4)] + [(f"medssd-stage{i + 1}", 64, L, dm, 64, 128, 3)
                                                       for i, (L, dm) in enumerate([(3136, 96), (784, 192), (196, 384), (49, 768)])]


def make(batch, L, d_model, P, N, width, copies):
    dim = 2 * d_model
    H, conv_dim = dim // P, dim + 2 * N
    prm = dict(conv_w=torch.randn(conv_dim, width, device=dev) * 0.3, conv_b=torch.randn(conv_dim, device=dev) * 0.1,
               dt_bias=torch.rand(H, device=dev) * 0.5, A=-0.5 - torch.rand(H, device=dev), D=torch.randn(H, device=dev),
               rms_w=torch.ones(dim, device=dev), W=torch.randn(d_model, dim, device=dev) / dim ** 0.5)
    for v in prm.values():
        v.requires_grad_()
    zx = [torch.randn(batch, L, dim + conv_dim + H, device=dev, dtype=torch.bfloat16).requires_grad_() for _ in range(copies)]
    g = torch.randn(batch, L, d_model, device=dev, dtype=torch.bfloat16)
    return prm, zx, g, (H, dim, conv_dim)


def fused(p, zx, P):
    return mamba_split_conv1d_scan_combined(zx, p["conv_w"], p["conv_b"], p["dt_bias"], p["A"], p["D"], 256, rmsnorm_weight=p["rms_w"],
                                            outproj_weight=p["W"], headdim=P, norm_before_gate=False)


def composed(p, zx, P, N, dims, torch_conv):
    H, dim, conv_dim = dims
    z, xBC, dt = zx.split([dim, conv_dim, H], -1)
    if torch_conv:
        w = p["conv_w"].shape[1]
        xbc = F.silu(F.conv1d(xBC.transpose(1, 2), p["conv_w"].unsqueeze(1), p["conv_b"], padding=w - 1, groups=conv_dim)[..., :zx.shape[1]])
    else:
        xbc = causal_conv1d_fn(xBC.transpose(1, 2), p["conv_w"], p["conv_b"], activation="silu")
    xbc = xbc.transpose(1, 2)
    x, Bm, Cm = xbc.split([dim, N, N], -1)
    y = mamba_chunk_scan_combined(x.unflatten(-1, (H, P)), dt, p["A"], Bm.unflatten(-1, (1, N)), Cm.unflatten(-1, (1, N)), 256, D=p["D"],
                                  dt_bias=p["dt_bias"], dt_softplus=True)
    o = rmsnorm_fn(y.flatten(2), p["rms_w"], None, z=z, norm_before_gate=False)
    return F.linear(o, p["W"])


def timed(step, copies, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        step(i % copies)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def memory(fwd, bwd):
    """(bytes held between forward and backward: the output and what autograd saved, peak bytes of forward + backward), both
    above what was allocated before."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = fwd(0)
    torch.cuda.synchronize()
    held = torch.cuda.memory_allocated() - base
    bwd(0, out)
    del out
    torch.cuda.synchronize()
    return held, torch.cuda.max_memory_allocated() - base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    for name, batch, L, d_model, P, N, width in SHAPES:
        dim = 2 * d_model
        one = batch * L * (2 * dim + 2 * N + dim // P) * 2
        copies = max(1, -(-2 * L2_BYTES // one))
        p, zxs, g, dims = make(batch, L, d_model, P, N, width, copies)
        leaves = list(p.values())

        def arm(fn):
            def fwd(i):
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    return fn(zxs[i])
            return fwd, lambda i, out: torch.autograd.grad(out, [zxs[i]] + leaves, g)

        fns = {"fused": arm(lambda zx: fused(p, zx, P)), "composed": arm(lambda zx: composed(p, zx, P, N, dims, False)),
               "torchconv": arm(lambda zx: composed(p, zx, P, N, dims, True))}
        arms = {k: (lambda f, b: lambda i: b(i, f(i)))(f, b) for k, (f, b) in fns.items()}
        for s in arms.values():
            s(0), s(0)
        best = {k: float("inf") for k in arms}
        for _ in range(args.rounds):
            for k, s in arms.items():
                best[k] = min(best[k], timed(s, copies, args.iters))
        mem = {k: memory(*fb) for k, fb in fns.items()}
        # the conv kernels alone, on the xBC slices of the zxbcdt copies (read in place)
        H, _, conv_dim = dims
        w32, b32 = p["conv_w"].detach(), p["conv_b"].detach()
        outs = torch.empty(batch, L, conv_dim, device=dev, dtype=torch.bfloat16)
        gbuf = torch.randn(batch, L, conv_dim, device=dev)
        dx = torch.empty_like(outs)
        xbcs = [zx.detach()[..., dim:dim + conv_dim] for zx in zxs]
        kf = lambda i: conv_fwd(xbcs[i], w32, b32, None, True, outs)
        kb = lambda i: conv_bwd(gbuf, xbcs[i], w32, b32, None, True, dx)
        kf(0), kb(0)
        t_f = min(timed(kf, copies, 5 * args.iters) for _ in range(args.rounds))
        t_b = min(timed(kb, copies, 5 * args.iters) for _ in range(args.rounds))
        n = batch * L * conv_dim
        bytes_f, bytes_b = n * (2 + 2), n * (2 + 4 + 2)      # x in, y out / x and fp32 dy in, dx out
        print(json.dumps({"shape": name, "batch": batch, "L": L, "dim": dim, "heads": H, "d_state": N, "width": width,
                          "zxbcdt_row_pitch": zxs[0].shape[-1], "fwd_bwd_ms": {k: round(v, 3) for k, v in best.items()},
                          "held_fwd_to_bwd_MiB": {k: round(v[0] / 2**20, 1) for k, v in mem.items()},
                          "peak_MiB_above_inputs": {k: round(v[1] / 2**20, 1) for k, v in mem.items()}, "conv_fwd_ms": round(t_f, 4), "conv_bwd_ms": round(t_b, 4),
                          "conv_fwd_GBps": round(bytes_f / t_f / 1e6, 1), "conv_bwd_GBps": round(bytes_b / t_b / 1e6, 1)}), flush=True)
        del p, zxs, g, outs, gbuf, dx, xbcs, leaves, arms, fns
        torch.cuda.empty_cache()
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    t_c = min(timed(lambda i: dst.copy_(src), 1, 20) for _ in range(3))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"copy_GBps": round(2 * src.numel() / t_c / 1e6, 1), "device": torch.cuda.get_device_name(),
                      "nvidia_smi": q.stdout.strip()}))


if __name__ == "__main__":
    main()
