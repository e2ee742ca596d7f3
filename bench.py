#!/usr/bin/env python
"""bench.py -- MedMamba-T training throughput on B200 (BASELINE.json metric) + selective-scan roofline.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (port)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write the last timed step's results (dump_outputs)

A "step" is one training step (forward, CrossEntropy, backward, Adam) of MedMamba-T
(MedMamba.py VSSM, depths 2-2-4-2, dims 96-768, 6 classes) on synthetic 3x224x224 images,
batch 64 per GPU, bf16 autocast (BASELINE.json configs[1]); N > 1 = ddp_train.py-style data
parallelism (one process per GPU, NCCL gradient all-reduce overlapped with backward).

One JSON line on rank 0:
  value      images/s over all ranks, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric with the step's input copied from pinned host memory and the loss read
             back to the host inside the timed region
  roofline   dominant libb200ssm kernel (selective scan): algorithmic bytes (SURVEY.md 8d formula)
             / CUDA-event time per launch, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference's CPU data flow (oracle/cpu_path.py: PyTorch CPU ops + the C
             restatement of selective_scan_ref) on a bounded sample, rank 0, N=1
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "images/s"
PER_GPU_BATCH = 64
NUM_CLASSES = 6
REF_BATCH = 8      # BASELINE.json configs[0]: the reference's own CPU-runnable case is batch 8
MODELS = {
    # default: the configuration BASELINE.json's metric is quoted on (configs[1])
    "medmamba_t": dict(metric="MedMamba-T train images/sec @224",
                       workload=("MedMamba-T (VSSM depths 2-2-4-2, dims 96-768, 6 classes) bf16-autocast training step, "
                                 "batch 64 per GPU, synthetic 3x224x224 (BASELINE.json configs[1])")),
    # BASELINE.json configs[2]: the Mamba-2 SSD family
    "medssd": dict(metric="MedSSD train images/sec @224",
                   workload=("MedSSD (SSD/MedSSD.py VSSM depths 2-2-4-2, dims 128-1024, d_state 128 -> N' = 512, 6 classes) bf16-autocast "
                             "training step, batch 64 per GPU, synthetic 3x224x224 (BASELINE.json configs[2])")),
    # BASELINE.json configs[3], first half: MedSSD_kan (the CrossMamba VFEFM fusion network of the second half is not mirrored)
    "medssd_kan": dict(metric="MedSSD_kan train images/sec @224",
                       workload=("MedSSD_kan (MedSSD_kan/MedSSD_kan.py VSSM depths 2-2-4-2, dims 128-1024, d_state 16 -> N' = 64, KAN head, "
                                 "6 classes) bf16-autocast training step, synthetic 3x224x224 (BASELINE.json configs[3])")),
}
METRIC = MODELS["medmamba_t"]["metric"]
WORKLOAD = MODELS["medmamba_t"]["workload"]


def build_model(name):
    from medical_image_classification_b200 import models
    return getattr(models, name)(num_classes=NUM_CLASSES)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak_tf32():
    """TF32 dense peak taken as half the measured sustained bf16 figure (the SSD kernels run inside a long step)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["bf16_tflops_sustained"]) / 2, "measured (MEASURED_PEAKS.json bf16_tflops_sustained / 2 = TF32)"
    except Exception:
        return 1400.0 / 2, "fallback (B200_PROFILING.md sustained bf16 1.4 PFLOP/s / 2 = TF32)"


# ------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi's numbers through NVML)
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {
        0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting",
    }

    def __init__(self, index: int, period: float = 0.2):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        while not self._halt.is_set():
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                try:
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set()
        if self.is_alive():
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# per-launch CUDA-event timing of the libb200ssm selective-scan kernels
# ------------------------------------------------------------------------------------------------
class ScanProfiler:
    """Wraps selective_scan_interface.launch_fwd/launch_bwd with torch.cuda events on the stream the
    kernels are launched on (torch's current stream), and records the algorithmic bytes per launch."""

    def __init__(self):
        import torch
        from medical_image_classification_b200 import selective_scan_interface as ssi
        from medical_image_classification_b200 import _lib
        self.torch, self.ssi, self.lib = torch, ssi, _lib.load()
        self.records = []  # (key, bytes, start_event, end_event)
        self.enabled = False

    @staticmethod
    def algorithmic_bytes(kind, u, delta, Bm, L=None):
        """SURVEY.md section 8(d): s = bytes per I/O element, E = B*KD*L, Ebc = B*K*N*L.
        fwd: s*(3E + 2Ebc) + 4*(KD*N + 2KD);  bwd: s*(5E + 2Ebc) + 4*2Ebc + 4*(2KD*N + 4KD)."""
        s = u.element_size()
        batch, KD = delta.shape[0], delta.numel() // (delta.shape[0] * delta.shape[-1])   # (B, KD, L) or a (B, K, D, L) view
        L = L or delta.shape[-1]                # the TRUE sequence length when rows are padded to a 16-byte pitch (49 -> 52)
        G, N = Bm.shape[1], Bm.shape[2]
        E, Ebc = batch * KD * L, batch * G * N * L
        if kind.startswith("fwd"):
            return s * (3 * E + 2 * Ebc) + 4 * (KD * N + 2 * KD)
        return s * (5 * E + 2 * Ebc) + 4 * 2 * Ebc + 4 * (2 * KD * N + 4 * KD)

    def install(self):
        self.ssi.set_profiler(self)

    def begin(self):
        if not self.enabled:
            return None
        e0 = self.torch.cuda.Event(enable_timing=True)
        e0.record()
        return e0

    def end(self, e0, kind, u, delta, Bm, algo_len=None):
        if e0 is None:
            return
        e1 = self.torch.cuda.Event(enable_timing=True)
        e1.record()
        gen = "2" if self.lib.b200_sscan_last_variant() == 2 else ""
        key = (kind + gen, (delta.shape[0], delta.numel() // (delta.shape[0] * delta.shape[-1]), algo_len or delta.shape[-1]), Bm.shape[2], str(u.dtype))
        self.records.append((key, self.algorithmic_bytes(kind, u, delta, Bm, algo_len), e0, e1))

    def summary(self, peak_gbs, peak_src, steps):
        """Per (kernel, shape): launches, mean ms between events recorded immediately around the
        C-ABI launch on the launching stream, achieved GB/s."""
        agg = {}
        for key, nbytes, e0, e1 in self.records:
            ms = e0.elapsed_time(e1)
            a = agg.setdefault(key, [0, 0.0, nbytes])
            a[0] += 1
            a[1] += ms
        if not agg:
            return None, None
        rows = []
        for key, (n, ms, nbytes) in agg.items():
            rows.append({"kernel": f"sscan_{key[0]}_kernel", "shape_b_kd_l": list(key[1]), "dstate": key[2],
                         "io": key[3].replace("torch.", ""), "launches": n, "ms_per_launch": ms / n,
                         "bytes_per_launch": nbytes, "gbs": nbytes / (ms / n) / 1e6})
        rows.sort(key=lambda r: -r["ms_per_launch"] * r["launches"])
        top = rows[0]
        tot_bytes = sum(r["bytes_per_launch"] * r["launches"] for r in rows)
        tot_ms = sum(r["ms_per_launch"] * r["launches"] for r in rows)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as fh:
                traffic = json.load(fh).get(top["kernel"] + ":" + "x".join(map(str, top["shape_b_kd_l"])))
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": top["kernel"], "shape_b_kd_l": top["shape_b_kd_l"],
                "achieved": round(top["gbs"], 1), "peak": peak_gbs, "unit": "GB/s",
                "frac": round(top["gbs"] / peak_gbs, 4), "traffic": traffic,
                "bytes_per_launch": top["bytes_per_launch"], "ms_per_launch": round(top["ms_per_launch"], 4),
                "peak_source": peak_src, "formula": "SURVEY.md 8(d) API-boundary bytes, fp32 I/O (s=4)",
                "timing": "CUDA events around the C-ABI launch in an eager single-stream twin of the same K steps (the kernel alone; in the "
                          "timed step it shares the GPU with the other branch's kernels)"}
        allscan = {"launches_per_step": round(sum(r["launches"] for r in rows) / steps, 1),
                   "bytes_per_step": tot_bytes / steps, "ms_per_step": round(tot_ms / steps, 4),
                   "achieved": round(tot_bytes / tot_ms / 1e6, 1), "unit": "GB/s",
                   "frac": round(tot_bytes / tot_ms / 1e6 / peak_gbs, 4),
                   "per_kernel": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items()} for r in rows]}
        return roof, allscan


class SsdProfiler:
    """Same idea for the SSD operator (b200_ssd_fwd / b200_ssd_bwd: 5 + 6 kernels per call): CUDA events immediately around the
    C-ABI call, algorithmic FLOPs and bytes per call from SURVEY.md 8(d)."""

    def __init__(self):
        import torch
        from medical_image_classification_b200 import ssd_combined
        self.torch, self.mod = torch, ssd_combined
        self.records, self.enabled = [], False

    @staticmethod
    def work(kind, batch, L, H, P, G, N, Q, s=4):
        nq = [min(Q, L - c) for c in range(0, L, Q)]
        if kind == "fwd":
            flops = batch * sum(2 * q * q * N * G + H * (2 * q * q * P + 4 * q * N * P) for q in nq)
            nbytes = s * (2 * batch * L * H * P + 2 * batch * L * G * N + batch * L * H)
        else:
            flops = batch * sum(6 * q * q * N * G + H * (4 * q * q * P + 10 * q * N * P) for q in nq)
            nbytes = s * (3 * batch * L * H * P + 4 * batch * L * G * N + 2 * batch * L * H)
        return flops, nbytes

    def install(self):
        self.mod.set_profiler(self)

    def begin(self):
        if not self.enabled:
            return None
        e0 = self.torch.cuda.Event(enable_timing=True)
        e0.record()
        return e0

    def end(self, e0, kind, shape):
        if e0 is None:
            return
        e1 = self.torch.cuda.Event(enable_timing=True)
        e1.record()
        self.records.append(((kind,) + tuple(shape), e0, e1))

    def summary(self, hbm_peak, hbm_src, steps):
        agg = {}
        for key, e0, e1 in self.records:
            a = agg.setdefault(key, [0, 0.0])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
        if not agg:
            return None, None
        tpk, tsrc = tensor_peak_tf32()
        rows = []
        for key, (n, ms) in agg.items():
            kind, batch, L, H, P, G, N, Q, prec = key
            flops, nbytes = self.work(kind, batch, L, H, P, G, N, Q)
            t = ms / n
            rows.append({"op": f"b200_ssd_{kind}", "shape_b_l_h_p_g_n_q": [batch, L, H, P, G, N, Q], "precision": "tf32" if prec else "3xtf32",
                         "launches": n, "ms_per_call": round(t, 4), "flops_per_call": flops, "bytes_per_call": nbytes,
                         "tflops": round(flops / t / 1e9, 2), "gbs": round(nbytes / t / 1e6, 1),
                         "t_tensor_ms": round(flops / tpk / 1e9, 4), "t_hbm_ms": round(nbytes / hbm_peak / 1e6, 4)})
        rows.sort(key=lambda r: -r["ms_per_call"] * r["launches"])
        top = rows[0]
        bound = "tensor" if top["t_tensor_ms"] >= top["t_hbm_ms"] else "hbm"
        if bound == "tensor":
            roof = {"bound": "tensor", "achieved": top["tflops"], "peak": tpk, "unit": "TFLOP/s", "frac": round(top["tflops"] / tpk, 4),
                    "peak_source": tsrc}
        else:
            roof = {"bound": "hbm", "achieved": top["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": round(top["gbs"] / hbm_peak, 4),
                    "peak_source": hbm_src}
        roof.update({"kernel": top["op"] + " (all kernels of the call)", "shape_b_l_h_p_g_n_q": top["shape_b_l_h_p_g_n_q"],
                     "precision": top["precision"], "ms_per_launch": top["ms_per_call"], "flops_per_launch": top["flops_per_call"],
                     "bytes_per_launch": top["bytes_per_call"], "traffic": None,
                     "formula": "SURVEY.md 8(d): max(HBM time, tensor time) of the SSD call; FLOPs sum_c 2 q^2 N G + H (2 q^2 P + 4 q N P) fwd, "
                                "6 / 4 / 10 bwd; bytes at fp32 I/O"})
        tot_ms = sum(r["ms_per_call"] * r["launches"] for r in rows)
        allssd = {"calls_per_step": round(sum(r["launches"] for r in rows) / steps, 1), "ms_per_step": round(tot_ms / steps, 4),
                  "tflops": round(sum(r["flops_per_call"] * r["launches"] for r in rows) / tot_ms / 1e9, 2), "per_call": rows}
        return roof, allssd


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference's CPU data flow (port)
# ------------------------------------------------------------------------------------------------
def cpu_train_step_time(batch: int, steps: int = 1, warmup: int = 0, threads: int | None = None, model: str = "medmamba_t"):
    import torch
    import oracle
    from oracle.cpu_path import bind_cpu_core
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    net = build_model(model)
    bind_cpu_core(net)
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    x = torch.randn(batch, 3, 224, 224)
    y = torch.randint(0, NUM_CLASSES, (batch,))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = torch.nn.functional.cross_entropy(net(x), y)
        loss.backward()
        opt.step()
        float(loss)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return sum(times) / len(times), max(threads, oracle.threads())


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the eager CPU module tree of
    oracle/cpu_path.py + the C restatements of selective_scan_ref / the SSD recurrence), all host threads.  Each step is a bounded
    sample of the workload: ONE fixed batch -- --cpu-batch, default 8 = BASELINE.json configs[0] -- so the number is reproducible
    from run to run and from N to N (round 1 picked the batch from a wall-clock heuristic)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = MODELS[args.model]
    cores = os.cpu_count() or 1
    b = args.cpu_batch
    t, threads = cpu_train_step_time(b, steps=args.steps, warmup=args.warmup, model=args.model)
    value = b / t
    sample = (f"{args.model} fp32 fwd+bwd+Adam on batch {b} of synthetic 3x224x224 per step "
              f"(PyTorch CPU ops + C/OpenMP restatement of the scan), {threads} threads")
    line = {"impl": "reference", "metric": cfg["metric"], "value": round(value, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t * 1e3, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "sample": sample, "cpu_batch": b},
            "cpu_baseline": {"value": round(value, 4), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                             "host_cores": cores},
            "e2e": {"value": round(value, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step computed, for comparing two builds output for output
# ------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 23      # elements kept of the flattened gradients: 32 MiB of float32


def restore_initial_state(net, opt, init_state):
    """Puts the model back to its seeded initial parameters and buffers and the optimizer back to a fresh state, in place (the
    captured step graph keeps reading the same tensors).  The step that --dump-outputs records starts from here, so its inputs are
    the same in every run: the backward kernels sum dB / dC / dA and the weight gradients with float atomics, in no fixed order,
    and Adam on the benchmark's one repeated batch turns those last-bit differences into large ones within a few steps."""
    import torch
    with torch.no_grad():
        for k, v in net.state_dict().items():
            v.copy_(init_state[k])
        for st in opt.state.values():           # Adam: step, exp_avg, exp_avg_sq
            for t in st.values():
                if torch.is_tensor(t):
                    t.zero_()


def dump_outputs(out_dir, loss, net):
    """Writes, as float32 .npy files, what the last timed step computed from the seeded model and batch:
      loss.npy     the loss the step returned, shape (1,)
      grads.npy    the parameters' gradients (zeros for a parameter that received none), flattened in named_parameters() order
      buffers.npy  the floating-point buffers (BatchNorm running statistics its forward updated), flattened in named_buffers() order
    Gradients larger than DUMP_SAMPLE elements keep the same DUMP_SAMPLE positions, drawn once from a fixed seed, so two runs of
    the same model are compared element for element."""
    import numpy as np
    import torch
    params = [p for _, p in net.named_parameters()]
    flat_g = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().float().reshape(-1) for p in params])
    if flat_g.numel() > DUMP_SAMPLE:
        keep = np.sort(np.random.default_rng(0).choice(flat_g.numel(), DUMP_SAMPLE, replace=False))
        flat_g = flat_g[torch.from_numpy(keep).to(flat_g.device)]
    bufs = [b.detach().float().reshape(-1) for _, b in net.named_buffers() if b.is_floating_point()]
    arrays = {"loss": loss.detach().float().reshape(1), "grads": flat_g,
              "buffers": torch.cat(bufs) if bufs else torch.zeros(0, device=flat_g.device)}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def run_cuda(args):
    import torch
    import torch.distributed as dist
    from medical_image_classification_b200 import _lib
    from medical_image_classification_b200.models import medmamba_t

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    _lib.load()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ddp = world > 1
    if ddp:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if not args.no_graph:  # NCCL collectives are captured into the step graph
            os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        dist.init_process_group(backend="nccl", device_id=dev)
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(1234 + rank)

    cfg = MODELS[args.model]
    cpu_base = None
    if rank == 0 and not args.no_cpu_baseline:
        # rank 0 times the CPU port at every N (before the other ranks' first collective: they wait at the barrier below)
        cb = args.cpu_batch if args.model == "medmamba_t" else min(args.cpu_batch, 2)
        t, threads = cpu_train_step_time(cb, steps=1, warmup=0, model=args.model)
        cpu_base = {"value": round(cb / t, 4), "unit": UNIT, "cores": threads, "kind": "port",
                    "sample": f"one fp32 {args.model} training step (fwd+bwd+Adam) on batch {cb} of synthetic "
                              f"3x224x224 (BASELINE.json configs[0] is batch 8); PyTorch CPU ops + C/OpenMP restatement of "
                              f"the scan; {t:.1f} s",
                    "host_cores": os.cpu_count()}

    from medical_image_classification_b200.train_step import TrainStep
    from medical_image_classification_b200 import models as _models
    _models.SS_Conv_SSM.overlap_branches = not args.no_overlap
    net = build_model(args.model).to(dev)
    use_graph = not args.no_graph
    step = TrainStep(net, lr=1e-4, autocast=torch.bfloat16, ddp=ddp, local_rank=local_rank, graph=use_graph,
                     bucket_cap_mb=args.bucket_mb, grad_bf16=args.grad_bf16, broadcast_buffers=args.broadcast_buffers,
                     ddp_impl=args.ddp_impl)
    model = step.model
    init_state = {k: v.detach().clone() for k, v in net.state_dict().items()} if args.dump_outputs else None
    B = args.batch
    x_dev = torch.randn(B, 3, 224, 224, device=dev)
    y_dev = torch.randint(0, NUM_CLASSES, (B,), device=dev)
    x_host = torch.randn(B, 3, 224, 224).pin_memory()
    y_host = torch.randint(0, NUM_CLASSES, (B,)).pin_memory()
    eager_step, barrier = step.eager, step.barrier

    prof = ScanProfiler() if args.model == "medmamba_t" else SsdProfiler()
    prof.install()
    step.warmup(x_dev, y_dev, n=max(args.warmup, 3))
    # ---- capture the whole step (forward, loss, backward, Adam) in one CUDA graph ----
    step.capture(x_dev, y_dev)
    graph, static_x, static_y, graph_note = step.graph, step.static_x, step.static_y, step.note
    run_step = step

    for _ in range(3):
        run_step(static_x if graph is not None else x_dev, static_y if graph is not None else y_dev)
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    xin, yin = (static_x, static_y) if graph is not None else (x_dev, y_dev)
    # ---- timed region 1: inputs resident in HBM ----
    launches0 = _lib.launches()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps - (init_state is not None)):
        run_step(xin, yin)
    e1.record()
    if init_state is not None:
        # the last timed step, timed on its own: it starts from the seeded initial state (restored outside the timing)
        restore_initial_state(net, step.opt, init_state)
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        loss = run_step(xin, yin)
        d1.record()
    barrier()
    launches = _lib.launches() - launches0
    ms = e0.elapsed_time(e1)
    if init_state is not None:
        ms += d0.elapsed_time(d1)
        if rank == 0:
            dump_outputs(args.dump_outputs, loss, net)   # before region 2 trains the model further
    # ---- timed region 2: end to end (pinned host input -> device, loss -> host) ----
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # Input pipeline of the public API path: every step's batch is copied from pinned host memory on a copy stream into one of
    # two device staging buffers (what a pin_memory DataLoader with prefetch does), so step i+1's host->device copy overlaps step
    # i's compute; the step then takes its batch from the staging buffer and the loss is read back to the host every step.
    copy_stream = torch.cuda.Stream(device=dev)
    stage_x = [torch.empty_like(x_dev), torch.empty_like(x_dev)]
    stage_y = [torch.empty_like(y_dev), torch.empty_like(y_dev)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            stage_x[i % 2].copy_(x_host, non_blocking=True)
            stage_y[i % 2].copy_(y_host, non_blocking=True)
            ready[i % 2].record(copy_stream)

    f0.record()
    last = 0.0
    copy_stream.wait_stream(torch.cuda.current_stream())
    prefetch(0)
    for i in range(args.steps):
        if i + 1 < args.steps:
            prefetch(i + 1)          # the buffer's previous reader (step i-1) finished: its loss was read back
        torch.cuda.current_stream().wait_event(ready[i % 2])
        if graph is None:
            last = eager_step(stage_x[i % 2], stage_y[i % 2]).item()
        else:
            last = run_step(stage_x[i % 2], stage_y[i % 2]).item()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    clocks = sampler.stop()
    # ---- per-launch CUDA-event timing of the scan kernels: the same K steps, launched eagerly so the
    #      events bracket each kernel on its stream (events cannot be read back from a graph replay) ----
    kernel_launches_per_step = None
    opt_e = torch.optim.Adam(model.parameters(), lr=1e-4, fused=True) if graph is not None else step.opt

    def eager_probe(x, y):
        opt_e.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = torch.nn.functional.cross_entropy(model(x).float(), y)
        loss.backward()
        return loss

    barrier()
    l0 = _lib.launches()
    prof.enabled = True
    _models.SS_Conv_SSM.overlap_branches = False   # single stream: each kernel's events bracket that kernel alone, not its co-runners
    for _ in range(args.steps):
        eager_probe(x_dev, y_dev)
    _models.SS_Conv_SSM.overlap_branches = not args.no_overlap
    prof.enabled = False
    barrier()
    kernel_launches_per_step = (_lib.launches() - l0) // args.steps
    if graph is not None:
        launches = kernel_launches_per_step * args.steps  # replays launch the captured kernels; count them from the eager twin

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if ddp:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    if rank == 0:
        peak, peak_src = peaks()
        roof, allscan = prof.summary(peak, peak_src, args.steps)
        total = B * world * args.steps
        line = {"metric": cfg["metric"], "value": round(total / (ms / 1e3), 2), "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic",
                "config": {"workload": cfg["workload"], "global_batch": B * world, "per_gpu_batch": B, "image": "3x224x224",
                           "parallelism": f"dp{world}", "optimizer": "Adam lr 1e-4 (fused)", "launch": graph_note,
                           "streams": ("conv branch of every block on a side stream, SS2D branch on the main stream (fork / join captured in the graph)"
                                       if not args.no_overlap else "single stream"),
                           "ddp": (None if not ddp else
                                   (f"FlatGradSync: one fp32 gradient buffer, {len(step.sync.slices)} chunked NCCL all-reduces (avg) of "
                                    f"{[round(b_ / 2**20, 1) for b_ in step.sync.chunk_bytes()]} MiB launched from accumulate-grad hooks on a side "
                                    f"stream, captured in the step graph") if step.sync is not None else
                                   (f"DistributedDataParallel: bucket_cap_mb {args.bucket_mb}, static_graph, gradient_as_bucket_view, "
                                    f"broadcast_buffers={args.broadcast_buffers}, {'bf16' if args.grad_bf16 else 'fp32'} gradient all-reduce")),
                           "scan_io": "fp32 (as the reference calls it), fp32 state",
                           "l2": "per-step activations (> 10 GB) exceed the 126 MB L2; no explicit flush"},
                "e2e": {"value": round(total / (ms_e2e / 1e3), 2), "unit": UNIT,
                        "h2d_bytes_per_step": x_host.numel() * 4 + y_host.numel() * 8, "d2h_bytes_per_step": 4,
                        "input_pipeline": "pinned host batch -> device staging buffer on a copy stream, one step ahead (double buffered)",
                        "ms_per_step": round(ms_e2e / args.steps, 3), "last_loss": round(last, 4)},
                "gpu_launches": launches, "roofline": roof,
                ("scan_fwd_bwd" if args.model == "medmamba_t" else "ssd_fwd_bwd"): allscan, "clocks": clocks}
        if cpu_base is not None:
            line["cpu_baseline"] = cpu_base
        print(json.dumps(line), flush=True)
    if ddp:
        # Leave without tearing NCCL down: ncclCommDestroy can block for minutes while captured step graphs still
        # reference the communicator (seen at N=2: the JSON line was out, the ranks never exited).  Every rank has
        # passed the final all-reduce of the timings, so nothing is in flight.
        try:
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="per-GPU batch (BASELINE config: 64)")
    ap.add_argument("--cpu-batch", type=int, default=REF_BATCH, help="batch of the CPU arm / cpu_baseline sample (BASELINE.json configs[0]: 8)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--model", default="medmamba_t", choices=sorted(MODELS), help="medmamba_t = BASELINE.json configs[1] (default), medssd = configs[2]")
    ap.add_argument("--no-overlap", action="store_true", help="run the blocks' convolution branch on the SS2D branch's stream (A/B of models.SS_Conv_SSM.overlap_branches)")
    ap.add_argument("--ddp-impl", default="flat", choices=["flat", "torch"],
                    help="N > 1: 'flat' = train_step.FlatGradSync (one gradient buffer, a few chunked all-reduces), 'torch' = DistributedDataParallel")
    ap.add_argument("--bucket-mb", type=int, default=8, help="DistributedDataParallel bucket size (--ddp-impl torch)")
    ap.add_argument("--grad-bf16", action="store_true", help="bf16-compressed gradient all-reduce (N > 1)")
    ap.add_argument("--broadcast-buffers", action="store_true",
                    help="re-enable DDP's per-step broadcast of rank 0's BatchNorm statistics (N > 1; see train_step.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, gradients and BatchNorm buffers of the last timed step as DIR/<name>.npy (float32); that step "
                         "starts from the seeded initial model and a fresh optimizer, so runs with the same arguments compare")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA training step computed: it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
