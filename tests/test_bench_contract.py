"""The one-line JSON contract of bench.py, checked on the committed outputs of the last GPU run (profiles/): every key the driver
reads is present with the right type, for both arms.  (bench.py itself needs a B200; this guards the schema on CPU.)"""
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load(name):
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        pytest.skip(f"{name} not committed")
    return json.load(open(path))


BASE_KEYS = {"metric": str, "value": (int, float), "unit": str, "n_gpus": int, "steps": int, "warmup": int, "ms_per_step": (int, float),
             "higher_is_better": bool, "scaling": str, "dtype": str, "data": str, "config": dict, "e2e": dict, "gpu_launches": int,
             "cpu_baseline": dict}


def check_base(line):
    for k, t in BASE_KEYS.items():
        assert k in line, k
        assert isinstance(line[k], t), (k, type(line[k]))
    assert "vs_baseline" in line and line["vs_baseline"] is None          # BASELINE.md publishes no number for this metric
    assert "workload" in line["config"] and "model" not in line["config"]
    for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert k in line["e2e"], k
    for k in ("value", "unit", "cores", "kind", "sample"):
        assert k in line["cpu_baseline"], k
    assert line["cpu_baseline"]["kind"] in ("port", "reference")


@pytest.mark.parametrize("name", ["r01h_bench.json", "r01h_bench_dp4.json", "r02a_bench.json", "r02h_bench.json", "r02b_bench_dp4.json", "r02f_bench_dp4.json", "r02c_bench_dp8.json", "r02j_bench_dp2.json", "r02k_bench.json"])
def test_our_arm_line(name):
    line = load(name)
    if "dp" in name:
        line["cpu_baseline"] = load("r01h_bench.json")["cpu_baseline"]   # the CPU leg runs at N=1 only
    if name.startswith("r02"):
        # round 2: the reference's own request shapes, the multi-step loop and (N >= 2) the served mix + tensor parallelism are inside the contract
        assert "verbatim" in line["e2e"]["prompts"] and set(line["e2e"]["prompt_tokens_by_kind"]) <= {"analyze", "diagnose", "execute"}
        r = line["react"]
        assert r["conversations_with_final_answer"] == r["conversations"] and 0 < r["prefix_hit_rate"] < 1 and r["react_steps_per_sec"] > 0
        if line["n_gpus"] >= 2:
            assert "configs[2]" in line["config"]["workload"] and set(line["e2e"]["prompt_tokens_by_kind"]) == {"analyze", "diagnose", "execute"}
            assert line["router"]["completed"] == line["router"]["requests"] == line["n_gpus"] * 128
            if name >= "r02i":          # the serving block goes through the native front from r02i on
                assert line["router"]["front"] == "native" and line["router"]["errors"] == [] and line["router"]["rejected_429"] == 0
            tp = line["tp"]
            assert tp["parity"]["ok"] is True and tp["parity"]["t"] == line["n_gpus"] and tp["parity"]["max_dlogit"] < 2.5e-2
            assert tp["t"] == line["n_gpus"] and 0 < tp["roofline_frac_per_gpu"] < 1
    check_base(line)
    assert line["metric"] == "decode_tokens_per_sec" and line["unit"] == "tokens/s" and line["higher_is_better"] is True
    assert line["scaling"] == "weak" and line["dtype"] == "bf16" and line["warmup"] >= 3
    assert line["gpu_launches"] > 0
    assert abs(line["value"] - line["n_gpus"] * line["config"]["batch_per_gpu"] / (line["ms_per_step"] / 1e3)) / line["value"] < 1e-3
    # inputs larger than L2 between timed iterations, stated in config
    assert "l2" in line["config"]
    clk = line["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(clk) and not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(clk["reasons"]))
    e2e = line["e2e"]
    assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0 and e2e["value"] < line["value"]     # host copies inside, prefill included
    r = line["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3 and 0 < r["frac"] <= 1.0
    assert r["traffic"] is None or r["traffic"] >= 0.9 * r["algorithmic_bytes_per_launch"]


def test_dump_outputs_are_float_files_within_64mb(tmp_path):
    """--dump-outputs DIR: float32/float64 .npy files, at most 64 MB in all, the same logit columns on every run"""
    import sys
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(3)
    logits = rng.standard_normal((bench.BATCH, 128256), dtype=np.float32)
    r = {"last_ids": logits.argmax(1).astype(np.int32), "last_logits": logits}
    bench.dump_outputs(str(tmp_path / "a"), r)
    bench.dump_outputs(str(tmp_path / "b"), r)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files and all(f.endswith(".npy") for f in files)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
    ids, top = np.load(tmp_path / "a" / "decode_next_token_ids.npy"), np.load(tmp_path / "a" / "decode_next_token_logit.npy")
    assert np.array_equal(ids, r["last_ids"]) and np.array_equal(top, logits.max(1))
    cols = np.load(tmp_path / "a" / "decode_logits_sample_columns.npy").astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "decode_logits_sample.npy"), logits[:, cols])


@pytest.mark.parametrize("ref,ours_name", [("r01h_bench_reference_arm.json", "r01h_bench.json"), ("r02h_bench_reference_arm.json", "r02h_bench.json")])
def test_reference_arm_line(ref, ours_name):
    line = load(ref)
    check_base(line)
    ours = load(ours_name)
    assert line["impl"] == "reference" and line["gpu_launches"] == 0
    for k in ("metric", "unit", "higher_is_better"):
        assert line[k] == ours[k]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["value"] == line["value"]
