"""The committed bench lines (profiles/r02b_bench_n1.json = `python bench.py --steps 10 --warmup 3` on one B200, r02b_bench_n2.json =
the torchrun launch on two, r02_bench_reference_n1.json = `--impl reference`) carry every key of the driver's contract, with
consistent arithmetic: this pins the *shape* of what bench.py prints (values are whatever that box measured).  CPU only."""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
        "data", "config")


def _load(name):
    with open(os.path.join(ROOT, "profiles", name)) as fh:
        return json.load(fh)


def test_single_gpu_line_has_the_contract_keys_and_consistent_numbers():
    d = _load("r02b_bench_n1.json")
    for k in BASE + ("roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert k in d, k
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["metric"] in baseline["metric"] or baseline["metric"].startswith(d["metric"].split("/")[0])
    assert d["n_gpus"] == 1 and d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    samples = d["config"]["rays_per_step"] * d["config"]["samples_per_ray"]
    assert samples == 480 * 640 * 128
    assert abs(d["value"] - samples / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) <= 1e-9 and 0 < r["frac"] <= 1.0
    # the kernel cannot take longer than the step it is part of.  This line was printed when bench.py still timed the kernel in a
    # pass of its own after the timed region (58.47 against 58.41 ms: the power-capped clock had drifted between the two passes);
    # bench.py now takes both from the same iterations (kernel_ms_of_timed_steps, below)
    assert r["kernel_ms"] <= 1.002 * d["ms_per_step"]
    # the ncu traffic belongs to the sources this line was measured on
    traffic = _load("r02_render_traffic.json")
    assert traffic["src_sha16"] == d["src_sha16"] and r["traffic"] == traffic["dram_bytes_per_launch"]
    c = d["cpu_baseline"]
    assert set(("value", "unit", "cores", "kind", "sample")) <= set(c) and c["kind"] in ("reference", "port") and c["unit"] == d["unit"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["unit"] == d["unit"]
    assert e["value"] <= d["value"]                                  # host copies inside the timed region cannot make it faster
    assert d["gpu_launches"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    t = d["train_step"]
    assert "optimizer" in t and t["ms_per_step"] >= t["fwd_bwd_only"]["ms_per_step"]      # the optimizer step is inside the timed step
    g = t["cuda_graph_step"]["yaml_8x256x64"]
    assert g["graph_ms_per_step"] < g["eager_ms_per_step"]


def test_two_gpu_line_is_one_frame_strong_scaled():
    d1, d2 = _load("r02b_bench_n1.json"), _load("r02b_bench_n2.json")
    for k in BASE + ("roofline", "e2e", "gpu_launches", "clocks"):
        assert k in d2, k
    assert d2["n_gpus"] == 2 and d2["scaling"] == "strong" and d2["metric"] == d1["metric"] and d2["unit"] == d1["unit"]
    assert d2["config"]["rays_per_step"] == d1["config"]["rays_per_step"]          # the SAME frame, split across the ranks
    assert 1.5 < d1["ms_per_step"] / d2["ms_per_step"] < 2.5
    x = d2["train_step"]["exchange_vs_nccl_allreduce"]
    assert x["max_abs_diff"] == 0.0 and x["max_abs_value"] > 0            # the one-kernel NVLink exchange == the NCCL allreduce


def test_reference_arm_line():
    r, d = _load("r02_bench_reference_n1.json"), _load("r02b_bench_n1.json")
    for k in BASE + ("cpu_baseline", "e2e"):
        assert k in r, k
    assert r["impl"] == "reference" and r["metric"] == d["metric"] and r["unit"] == d["unit"] and r["higher_is_better"] is True
    assert r["cpu_baseline"]["kind"] == "reference" and r["cpu_baseline"]["value"] == r["value"]
    assert r["e2e"] == dict(value=r["value"], unit=r["unit"], h2d_bytes_per_step=0, d2h_bytes_per_step=0)


def test_kernel_time_comes_from_the_timed_iterations():
    import bench
    f = bench.kernel_ms_of_timed_steps
    assert f([9.0, 9.0, 9.0, 1.0, 2.0, 3.0], steps=3, warmup=3) == 2.0          # warm-up calls dropped
    assert f([5.0, 5.0, 1.0, 1.0, 2.0, 2.0], steps=2, warmup=1) == 3.0          # several launches per step are summed per step
    assert f([1.0, 2.0, 3.0], steps=2, warmup=2) is None and f([], 3, 1) is None and f([1.0, 2.0], 0, 2) is None


def test_dump_outputs_writes_float_arrays_and_samples_large_ones(tmp_path, monkeypatch):
    import numpy as np
    import pytest
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_WHOLE_BYTES", 4096)
    monkeypatch.setattr(bench, "DUMP_RAYS", 16)
    g = torch.Generator().manual_seed(0)
    out = dict(rgb=torch.rand(1, 100, 3, generator=g), alpha=torch.rand(1, 100, 32, generator=g).bfloat16(),
               density=torch.rand(1, 100, 32, 2, generator=g, dtype=torch.float64), idx=torch.tensor([3]), note="not an array")
    nbytes = bench.dump_outputs(str(tmp_path / "a"), out, 100)
    got = {p.stem: np.load(p) for p in (tmp_path / "a").iterdir()}
    assert sorted(got) == ["alpha", "density", "idx", "rgb", "sample_ray_idx"]
    assert nbytes == sum(a.nbytes for a in got.values())
    pick = got["sample_ray_idx"].astype(np.int64)
    assert len(pick) == 16 and len(set(pick)) == 16 and list(pick) == sorted(pick)
    assert got["rgb"].dtype == np.float32 and np.array_equal(got["rgb"], out["rgb"].numpy())              # small: whole
    assert got["alpha"].dtype == np.float32 and np.array_equal(got["alpha"], out["alpha"].float()[:, pick].numpy())
    assert got["density"].dtype == np.float64 and np.array_equal(got["density"], out["density"][:, pick].numpy())
    assert got["idx"].dtype == np.float64 and got["idx"].tolist() == [3.0]
    bench.dump_outputs(str(tmp_path / "b"), out, 100)                                                  # same arguments, same files
    assert all(np.array_equal(a, np.load(tmp_path / "b" / (k + ".npy"))) for k, a in got.items())
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 1024)
    with pytest.raises(ValueError, match="limit"):
        bench.dump_outputs(str(tmp_path / "c"), out, 100)
