"""Cost of the state gradients in the SSD backward (mamba_chunk_scan_combined: initial_states in, final_states out), CUDA events.

At MedSSD's four stage shapes (L = 3136 / 784 / 196 / 49, H' = 8 / 16 / 32 / 64 heads of 64, N' = 512, one group, chunk 256,
batch 64, single-pass TF32 as under bf16 autocast; the reference's layout: channel-major storage, (b, l, .) views), the backward
alone (one forward, then repeated torch.autograd.grad over its graph) of
  plain   as the models call it: no initial_states, final_states not returned
  states  initial_states that require a gradient, and a gradient for the returned final_states as well as for out
Arms are alternated; each reports its best round.  Prints one JSON line per stage, then the device name and power limit.

    python tools/bench_ssd_states.py [--iters N] [--rounds R] [--batch B]
    python tools/bench_ssd_states.py --dump OUT.npz [--stage K]

--dump runs one seeded `plain` backward at stage K (default 1) and writes its inputs' gradients to OUT.npz, so that two trees can
be compared on the same inputs; it writes nothing else."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from medical_image_classification_b200 import ssd_combined  # noqa: E402
from medical_image_classification_b200.ssd_combined import mamba_chunk_scan_combined  # noqa: E402

Q, P, N = 256, 64, 512
STAGES = [(3136, 8), (784, 16), (196, 32), (49, 64)]
dev = "cuda"


def inputs(batch, L, H):
    x = torch.randn(batch, H * P, L, device=dev).permute(0, 2, 1).unflatten(2, (H, P)).requires_grad_()
    Bm = torch.randn(batch, N, L, device=dev).permute(0, 2, 1).unflatten(2, (1, N)).requires_grad_()
    Cm = torch.randn(batch, N, L, device=dev).permute(0, 2, 1).unflatten(2, (1, N)).requires_grad_()
    dt = (0.5 * torch.rand(batch, H, L, device=dev)).permute(0, 2, 1).requires_grad_()
    A = (-0.5 - torch.rand(H, device=dev)).requires_grad_()
    D = torch.randn(H, device=dev).requires_grad_()
    bias = (0.3 * torch.rand(H, device=dev)).requires_grad_()
    return (x, dt, A, Bm, Cm, D, bias), torch.randn(batch, L, H, P, device=dev)


def backward_fn(t, g, with_states):
    """A closure running the backward of one forward, keeping the graph."""
    x, dt, A, Bm, Cm, D, bias = t
    batch, L, H, _ = x.shape
    if not with_states:
        out = mamba_chunk_scan_combined(x, dt, A, Bm, Cm, Q, D=D, dt_bias=bias, dt_softplus=True)
        return lambda: torch.autograd.grad(out, t, g, retain_graph=True)
    init = torch.randn(batch, H, P, N, device=dev, requires_grad=True)
    out, fin = mamba_chunk_scan_combined(x, dt, A, Bm, Cm, Q, D=D, dt_bias=bias, initial_states=init, dt_softplus=True,
                                         return_final_states=True)
    gf = torch.randn_like(fin)
    return lambda: torch.autograd.grad((out, fin), t + (init,), (g, gf), retain_graph=True)


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def best_of(arms, iters, rounds):
    for fn in arms.values():     # warm-up: module load, allocator
        fn(); fn()
    torch.cuda.synchronize()
    best = {k: float("inf") for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            best[k] = min(best[k], time_ms(fn, iters))
    return best


def dump(path, stage, batch):
    torch.manual_seed(0)
    L, H = STAGES[stage]
    t, g = inputs(batch, L, H)
    grads = backward_fn(t, g, False)()
    np.savez(path, **{k: v.detach().cpu().numpy() for k, v in zip(("dx", "ddt", "dA", "dB", "dC", "dD", "ddt_bias"), grads)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--dump", default=None)
    ap.add_argument("--stage", type=int, default=1)
    args = ap.parse_args()
    ssd_combined.set_precision(1)
    if args.dump:
        dump(args.dump, args.stage, args.batch)
        return
    for L, H in STAGES:
        t, g = inputs(args.batch, L, H)
        best = best_of({"plain": backward_fn(t, g, False), "states": backward_fn(t, g, True)}, args.iters, args.rounds)
        print(json.dumps({"L": L, "H": H, "N": N, "batch": args.batch, "bwd_ms": {k: round(v, 4) for k, v in best.items()},
                          "states_over_plain": round(best["states"] / best["plain"] - 1.0, 4)}), flush=True)
        del t, g
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}))


if __name__ == "__main__":
    main()
