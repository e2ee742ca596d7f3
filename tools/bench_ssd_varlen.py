"""Cost of packed variable-length sequences in the SSD chunk scan (mamba_chunk_scan_combined's seq_idx), CUDA events.

At MedSSD's four stage shapes (L = 3136 / 784 / 196 / 49, H' = 8 / 16 / 32 / 64 heads of 64, N' = 512, one group, chunk 256,
batch 64, single-pass TF32 as under bf16 autocast; the reference's layout: channel-major storage, (b, l, .) views), forward and
forward + backward of
  none    seq_idx=None
  zeros   an all-zero seq_idx (the masked kernels with nothing masked: their cost over `none`)
  four    four equal segments per row
then one packed row of mixed-length sequences (the four stage lengths, several of each, at stage 0's head shape) against one call per
sequence.  Arms are alternated; each reports its best round.
    python tools/bench_ssd_varlen.py [--iters N] [--rounds R] [--batch B]
Prints one JSON line per measurement, then the device name and power limit."""
import argparse
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
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


def fwd_fn(t, seq_idx):
    x, dt, A, Bm, Cm, D, bias = t
    return lambda: mamba_chunk_scan_combined(x, dt, A, Bm, Cm, Q, D=D, dt_bias=bias, dt_softplus=True, seq_idx=seq_idx)


def fwd_bwd_fn(t, g, seq_idx):
    f = fwd_fn(t, seq_idx)
    return lambda: torch.autograd.grad(f(), t, g)


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    args = ap.parse_args()
    ssd_combined.set_precision(1)
    for L, H in STAGES:
        t, g = inputs(args.batch, L, H)
        seqs = {"none": None, "zeros": torch.zeros(args.batch, L, dtype=torch.int32, device=dev),
                "four": (torch.arange(L, device=dev) * 4 // L).to(torch.int32).expand(args.batch, L)}
        with torch.no_grad():
            fwd = best_of({k: fwd_fn(t, s) for k, s in seqs.items()}, args.iters, args.rounds)
        both = best_of({k: fwd_bwd_fn(t, g, s) for k, s in seqs.items()}, args.iters, args.rounds)
        for k in seqs:
            print(json.dumps({"L": L, "H": H, "N": N, "batch": args.batch, "seq_idx": k, "fwd_ms": round(fwd[k], 3),
                              "bwd_ms": round(both[k] - fwd[k], 3), "fwd_bwd_ms": round(both[k], 3)}), flush=True)
        del t, g
    # one packed row of mixed lengths vs one call per sequence, stage-0 heads
    lengths = [3136] * 2 + [784] * 6 + [196] * 12 + [49] * 24
    H = STAGES[0][1]
    t, g = inputs(1, sum(lengths), H)
    seq_idx = torch.repeat_interleave(torch.arange(len(lengths), device=dev, dtype=torch.int32),
                                      torch.tensor(lengths, device=dev))[None]
    parts, o = [], 0
    for n in lengths:
        x, dt, A, Bm, Cm, D, bias = t
        parts.append(((x[:, o:o + n], dt[:, o:o + n], A, Bm[:, o:o + n], Cm[:, o:o + n], D, bias), g[:, o:o + n]))
        o += n
    packed = fwd_bwd_fn(t, g, seq_idx)
    calls = [fwd_bwd_fn(pt, pg, None) for pt, pg in parts]
    res = best_of({"packed": packed, "per_sequence": lambda: [c() for c in calls]}, args.iters, args.rounds)
    print(json.dumps({"packed_row": {"sequences": len(lengths), "tokens": sum(lengths), "H": H, "N": N},
                      "fwd_bwd_ms": {k: round(v, 3) for k, v in res.items()}}), flush=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"device": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}))


if __name__ == "__main__":
    main()
