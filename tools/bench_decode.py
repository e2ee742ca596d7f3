"""Recurrent decoding: selective_state_update and causal_conv1d_update per call, CUDA events.

Shapes: a Mamba-2-130m-like layer (24 heads of 64, d_state 128, conv_dim 1792), a Mamba-2-2.7b-like layer (80 heads of 64, d_state
128, conv_dim 5376) and a Mamba-1-130m-like layer (dim 1536, d_state 16, conv over the 1536 channels), each at batch 1, 8, 64 and
256 with an fp32 and a bf16 state (the activations in the state's dtype, A in fp32), with transformers' argument sets: A, dt,
dt_bias and D expanded, x, B and C column slices of the conv output, the conv input a column slice of in_proj's output.

Per shape, the time per call of
  ssu        this package's selective_state_update (csrc/state_update.cu)
  conv       this package's causal_conv1d_update (csrc/conv1d.cu)
  vllm       vLLM's Triton selective_state_update on the same inputs (when vLLM is importable)
  torch      a composed-PyTorch restatement of selective_state_update
  mixer      one decode step of transformers' Mamba2Mixer.cuda_kernels_forward with this package's five kernels patched in,
             against its torch_forward (Mamba-2 shapes only)
with GB/s of the bytes each op must move (computed from the shapes below).  Each op is captured in a CUDA graph of `iters` calls
and the graph is replayed, so the times are GPU time per call without the Python launch cost.  When the state exceeds the 126 MB
L2, the calls cycle over enough state copies that every pass reads the state from HBM ("state_copies" > 1 says so).  Prints one
JSON line per shape, then the device-to-device copy rate measured in the same run, the device name and its power limit.

    python tools/bench_decode.py [--iters N] [--rounds R]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from medical_image_classification_b200.conv1d import causal_conv1d_fn, causal_conv1d_update  # noqa: E402
from medical_image_classification_b200.selective_state_update import selective_state_update  # noqa: E402
from medical_image_classification_b200.ssd_combined import mamba_chunk_scan_combined, mamba_split_conv1d_scan_combined  # noqa: E402

dev = "cuda"
L2_BYTES = 126 << 20
# (name, heads (None: Mamba-1), headdim (Mamba-1: dim), d_state, conv_dim)
SHAPES = [("mamba2-130m", 24, 64, 128, 1792), ("mamba2-2.7b", 80, 64, 128, 5376), ("mamba1-130m", None, 1536, 16, 1536)]
BATCHES = [1, 8, 64, 256]
WIDTH = 4


def graph_time(fn, iters, rounds):
    """ms per call of fn(i), i = 0 .. iters-1, captured in one CUDA graph and replayed (best of rounds)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(2):
            fn(i)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(iters):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    best = float("inf")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / iters)
    return best


def torch_ssu(state, x, dt, A, B, C, D, dt_bias):
    """The composed-PyTorch restatement (Mamba-2 form, ngroups 1, softplus), state updated in place."""
    v = F.softplus(dt.float() + dt_bias.float())
    new = state.float() * torch.exp(A * v[..., None]) + B.float()[:, :, None] * v[..., None] * x.float()[..., None]
    state.copy_(new)
    return ((new * C.float()[:, :, None]).sum(-1) + D.float() * x.float()).to(x.dtype)


def mixer_times(H, P, N, batch, dtype, iters, rounds):
    """(cuda_kernels_forward, torch_forward) ms of one graph-captured decode step of transformers' Mamba2Mixer."""
    import transformers
    from transformers.models.mamba2 import modeling_mamba2 as m2
    cfg = transformers.Mamba2Config(num_heads=H, head_dim=P, hidden_size=H * P // 2, state_size=N, expand=2, n_groups=1, chunk_size=256,
                                    conv_kernel=WIDTH, num_hidden_layers=1, vocab_size=16, use_conv_bias=True, use_bias=False)
    mixer = m2.Mamba2Mixer(cfg, layer_idx=0).to(dev, dtype).eval()
    # after the mixer's constructor, which sets these module globals from the mamba_ssm / causal-conv1d packages it finds
    for name, fn in (("selective_state_update", selective_state_update), ("causal_conv1d_update", causal_conv1d_update),
                     ("causal_conv1d_fn", causal_conv1d_fn), ("mamba_chunk_scan_combined", mamba_chunk_scan_combined),
                     ("mamba_split_conv1d_scan_combined", mamba_split_conv1d_scan_combined)):
        setattr(m2, name, fn)
    out = []
    for fwd in (mixer.cuda_kernels_forward, mixer.torch_forward):
        cache = transformers.DynamicCache(config=cfg)
        h = torch.randn(batch, 1, H * P // 2, device=dev, dtype=dtype)
        with torch.no_grad():
            mixer.cuda_kernels_forward(torch.randn(batch, 8, H * P // 2, device=dev, dtype=dtype), cache_params=cache)
            out.append(graph_time(lambda i: fwd(h, cache_params=cache), iters, rounds))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    try:
        from vllm.model_executor.layers.mamba.ops.mamba_ssm import selective_state_update as vllm_ssu
    except Exception as exc:  # vLLM absent or unusable on this machine: its column reports why
        vllm_ssu, vllm_err = None, f"{type(exc).__name__}: {str(exc)[:120]}"
    for name, H, P, N, conv_dim in SHAPES:
        mamba1 = H is None
        Hh = 1 if mamba1 else H
        for dtype in (torch.float32, torch.bfloat16):
            es = 4 if dtype == torch.float32 else 2
            for batch in BATCHES:
                dim = Hh * P
                G = 1
                sbytes = batch * dim * N * es
                copies = max(1, -(-2 * L2_BYTES // sbytes))
                states = [torch.randn(batch, Hh, P, N, device=dev).to(dtype) * 0.1 for _ in range(copies)]
                proj = torch.randn(batch, dim + conv_dim + Hh, device=dev).to(dtype)     # (gate, xBC, dt) of in_proj's output
                xBC = proj[:, dim:dim + conv_dim]
                dt = proj[:, dim + conv_dim:dim + conv_dim + Hh]
                conv_out = torch.randn(batch, conv_dim if not mamba1 else dim + 2 * N, device=dev).to(dtype)
                x = conv_out[:, :dim].view(batch, Hh, P)
                Bm, Cm = conv_out[:, dim:dim + N].view(batch, G, N), conv_out[:, dim + N:dim + 2 * N].view(batch, G, N)
                if mamba1:     # Mamba-1: A (dim, N), dt, dt_bias, D per channel
                    A = -torch.rand(Hh, P, N, device=dev) - 0.5
                    dtv, bias, D = torch.rand(batch, Hh, P, device=dev).to(dtype), torch.rand(Hh, P, device=dev), torch.randn(Hh, P, device=dev)
                else:
                    A = (-torch.rand(Hh, device=dev) - 0.5)[:, None, None].expand(Hh, P, N)
                    dtv = dt[:, :, None].expand(batch, Hh, P)
                    bias = torch.rand(Hh, device=dev).to(dtype)[:, None].expand(Hh, P)
                    D = torch.randn(Hh, device=dev).to(dtype)[:, None].expand(Hh, P)
                ops = {
                    "ssu": lambda i: selective_state_update(states[i % copies], x, dtv, A, Bm, Cm, D, dt_bias=bias, dt_softplus=True),
                }
                if not mamba1:
                    ops["torch"] = lambda i: torch_ssu(states[i % copies], x, dtv, A, Bm, Cm, D, bias)
                if vllm_ssu is not None:
                    vout = torch.empty_like(x)
                    ops["vllm"] = lambda i: vllm_ssu(states[i % copies], x, dtv, A, Bm, Cm, D, bias, dt_softplus=True, out=vout)
                conv_states = [torch.randn(batch, conv_dim, WIDTH, device=dev).to(dtype) for _ in range(copies)]
                cw, cb = torch.randn(conv_dim, WIDTH, device=dev).to(dtype), torch.randn(conv_dim, device=dev).to(dtype)
                ops["conv"] = lambda i: causal_conv1d_update(xBC, conv_states[i % copies], cw, cb, "silu")
                ms, n = {}, max(args.iters, copies)
                for k, fn in ops.items():
                    try:
                        ms[k] = round(graph_time(fn, n, args.rounds), 5)
                    except Exception as exc:
                        ms[k] = f"failed: {type(exc).__name__}: {str(exc)[:120]}"
                # bytes each op must move: the state read and written, x, dt, B, C and out once (A, D, dt_bias and the conv weights stay in L2)
                ssu_bytes = 2 * sbytes + batch * (2 * dim * es + 2 * G * N * es + (dim if mamba1 else Hh) * es)
                conv_bytes = batch * conv_dim * (2 * WIDTH * es + 2 * es)
                gbps = lambda b, t: round(b / t / 1e6, 1) if isinstance(t, float) else None
                rec = {"shape": name, "batch": batch, "state_dtype": str(dtype).replace("torch.", ""), "heads": H, "headdim": P,
                       "d_state": N, "conv_dim": conv_dim, "state_MB": round(sbytes / 1e6, 2), "state_copies": copies, "ms": ms,
                       "ssu_GBps": gbps(ssu_bytes, ms.get("ssu")), "conv_GBps": gbps(conv_bytes, ms.get("conv")),
                       "vllm_GBps": gbps(ssu_bytes, ms.get("vllm")) if vllm_ssu is not None else f"vLLM not usable: {vllm_err}"}
                if not mamba1:
                    try:
                        kern, ref = mixer_times(H, P, N, batch, dtype, 10, args.rounds)
                        rec["mixer_step_ms"] = {"cuda_kernels_forward": round(kern, 4), "torch_forward": round(ref, 4)}
                    except Exception as exc:
                        rec["mixer_step_ms"] = f"failed: {type(exc).__name__}: {str(exc)[:160]}"
                print(json.dumps(rec), flush=True)
                del states, conv_states, ops
                torch.cuda.empty_cache()
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_c = float("inf")
    for _ in range(3):          # eagerly, as tools/bench_split_conv1d.py does (a copy captured in a graph ran at half this rate)
        e0.record()
        for _ in range(20):
            dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        t_c = min(t_c, e0.elapsed_time(e1) / 20)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"copy_GBps": round(2 * src.numel() / t_c / 1e6, 1), "device": torch.cuda.get_device_name(),
                      "nvidia_smi": q.stdout.strip()}))


if __name__ == "__main__":
    main()
