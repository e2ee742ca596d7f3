"""CPU: the `bench.py --impl reference` arm (the reference's CPU data flow timed on the host cores) prints ONE JSON line with
the keys the driver's contract names; the product arm refuses to run without a GPU instead of falling back."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-batch", "1"],
                         cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "MedMamba-T train images/sec @224" and d["unit"] == "images/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d, k
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["config"]["cpu_batch"] == 1          # --cpu-batch is honoured (round 1 picked the batch from a timing heuristic)
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and abs(cb["value"] - d["value"]) < 1e-6 * max(1.0, d["value"])
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0 and abs(e["value"] - d["value"]) < 1e-6 * max(1.0, d["value"])


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, "bench.py", "--steps", "1", "--warmup", "0", "--no-cpu-baseline"], cwd=ROOT, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode != 0                     # no silent CPU fallback
    assert not [l for l in out.stdout.splitlines() if l.startswith("{") and '"value"' in l]


def test_dump_outputs_writer_and_state_restore(tmp_path, monkeypatch):
    """CPU: bench.dump_outputs writes float32 loss / grads / buffers, sampling the gradients at the same seeded positions on every
    call; bench.restore_initial_state brings back the seeded weights and buffers and a fresh Adam state in place."""
    import numpy as np
    import torch
    import bench
    from medical_image_classification_b200.models import VSSM
    torch.manual_seed(0)
    net = VSSM(num_classes=6, depths=[1, 1], dims=[16, 32], drop_path_rate=0.0)
    init = {k: v.detach().clone() for k, v in net.state_dict().items()}
    ptrs = [p.data_ptr() for p in net.parameters()]
    opt = torch.optim.Adam(net.parameters(), lr=1e-2)
    for _ in range(2):
        for p in net.parameters():
            p.grad = torch.randn_like(p)
        opt.step()
    net.state_dict()[next(k for k in init if k.endswith("running_mean"))].add_(1.0)
    bench.restore_initial_state(net, opt, init)
    assert [p.data_ptr() for p in net.parameters()] == ptrs
    assert all(torch.equal(v, init[k]) for k, v in net.state_dict().items())
    assert all(not t.any() for st in opt.state.values() for t in st.values() if torch.is_tensor(t))

    params = list(net.parameters())
    params[0].grad = None                                        # a parameter without a gradient is dumped as zeros
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params]).numpy()
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.25), net)
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in ("loss", "grads", "buffers")}
    assert sorted(os.listdir(tmp_path / "a")) == ["buffers.npy", "grads.npy", "loss.npy"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss"].tolist() == [1.25] and a["grads"].shape == (1000,)
    assert a["buffers"].size == sum(b.numel() for b in net.buffers() if b.is_floating_point())
    for n, v in a.items():
        assert np.array_equal(v, np.load(tmp_path / "b" / f"{n}.npy")), n
    keep = np.sort(np.random.default_rng(0).choice(flat.size, 1000, replace=False))
    assert np.array_equal(a["grads"], flat[keep])
    monkeypatch.setattr(bench, "DUMP_SAMPLE", flat.size)         # at or under the limit: every element, in order
    bench.dump_outputs(str(tmp_path / "c"), torch.tensor(1.25), net)
    assert np.array_equal(np.load(tmp_path / "c" / "grads.npy"), flat)


def test_bench_rejects_meaningless_arguments():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, "bench.py", *extra], cwd=ROOT, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error" in out.stderr, extra


def test_reference_arm_medssd():
    """BASELINE.json configs[2]: the same arm for the SSD family (eager CPU tree + the from-definition SSD oracle)."""
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--model", "medssd", "--steps", "1", "--warmup", "0",
                          "--cpu-batch", "1"], cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.strip().splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["metric"] == "MedSSD train images/sec @224" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["config"]["cpu_batch"] == 1
