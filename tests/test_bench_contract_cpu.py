"""The bench.py output contract, checked on the committed result lines (profiles/r01_bench_*.json, profiles/r02_bench_*.json) and on
the helpers that do not need a GPU."""
import importlib.util
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(name):
    return json.loads(open(os.path.join(ROOT, "profiles", name)).read())


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_committed_gpu_lines_carry_every_contract_key():
    for name, n in (("r01_bench_1gpu.json", 1), ("r01_bench_2gpu.json", 2)):
        d = _load(name)
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                  "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
            assert k in d, (name, k)
        assert d["n_gpus"] == n and d["scaling"] == "weak" and d["higher_is_better"] is True
        assert "workload" in d["config"] and "model" not in d["config"]
        assert d["gpu_launches"] > 0
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
        r = d["roofline"]
        for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert k in r, (name, k)
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    one = _load("r01_bench_1gpu.json")
    assert one["cpu_baseline"]["kind"] == "port" and one["cpu_baseline"]["cores"] >= 1
    assert one["roofline"]["traffic"] is not None


def test_reference_arm_line():
    d = _load("r01_bench_reference_arm.json")
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]


def test_traffic_is_reported_only_for_the_captured_shape():
    b = _bench()
    t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    got, src = b.ncu_traffic({"attn_shape": t["attn_shape"]})
    assert got == t["kernels"]["attn_bwd"]["dram_bytes"] and "ncu_traffic.json" in src
    other = dict(t["attn_shape"], d=t["attn_shape"]["d"] * 2)
    assert b.ncu_traffic({"attn_shape": other}) == (None, None)


def test_dump_outputs_fits_the_budget_and_samples_the_same_rows(tmp_path):
    import numpy as np
    import torch

    b = _bench()
    whole = {"loss": torch.tensor(0.25), "grad.w": torch.randn(3000, 1024)}
    big = torch.randn(100_000, 256, dtype=torch.bfloat16)  # 102 MB as float32: must be row-sampled
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), whole, {"y": big})
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["grad.w.npy", "loss.npy", "y.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= b.DUMP_BYTES
    for f in files:
        a, c = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, c)
    y = np.load(tmp_path / "a" / "y.npy")
    assert 10_000 < y.shape[0] < big.shape[0] and y.shape[1] == 256
    assert np.array_equal(np.load(tmp_path / "a" / "grad.w.npy"), whole["grad.w"].numpy())


def test_round2_lines():
    one, two, strong = _load("r02_bench_1gpu.json"), _load("r02_bench_2gpu.json"), _load("r02_bench_2gpu_strong.json")
    for d, n, scaling in ((one, 1, "weak"), (two, 2, "weak"), (strong, 2, "strong")):
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                  "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"):
            assert k in d, k
        assert d["n_gpus"] == n and d["scaling"] == scaling and d["warmup"] >= 3
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
        assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    # the CPU arm of round 2 times the reference's own eager code (oracle/_ref recipe), not the port
    assert one["cpu_baseline"]["kind"] == "reference"
    # weak scaling keeps the per-GPU work: two GPUs process twice the sequences in (almost) the same step time
    assert two["config"]["global_batch"] == 2 * one["config"]["global_batch"]
    assert two["ms_per_step"] < 1.1 * one["ms_per_step"]
    # strong scaling keeps the global batch
    assert strong["config"]["global_batch"] == one["config"]["global_batch"]
    ref = _load("r02_bench_reference_arm.json")
    assert ref["impl"] == "reference" and ref["cpu_baseline"]["kind"] == "reference"
    assert ref["e2e"]["value"] == ref["value"] == ref["cpu_baseline"]["value"]
    for line in open(os.path.join(ROOT, "profiles", "r02_bench_research.json")):
        d = json.loads(line)
        assert d["unit"] == "sequences/s" and d["value"] > 0 and "research" in d["metric"]
