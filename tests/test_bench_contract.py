"""bench.py's output contract: the reference arm is RUN here (small tables, CPU: the oracle port is what that arm
times), and the committed B200 lines under profiles/ are checked for the keys the driver and the judge read."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def last_json_line(text):
    lines = [l for l in text.splitlines() if l.startswith("{")]
    assert lines, text[-2000:]
    return json.loads(lines[-1])


def test_reference_arm_runs_and_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--small", "--steps", "6",
                        "--warmup", "1", "--batch", "4096"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = last_json_line(r.stdout)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["steps"] == 6
    assert d["metric"] == "bpr_train_triples_per_sec" and d["unit"] == "triples/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_bench_refuses_what_it_cannot_do(extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "error:" in r.stderr, r.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: float32 arrays of what the last timed step computed, 64 MB at most.  The same arguments give the
    same inputs, so a second run writes the same arrays (to summation order)."""
    from tests.util import assert_close
    runs = [tmp_path / "a", tmp_path / "b"]
    for out in runs:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--small", "--steps", "3", "--warmup", "3",
                            "--preroll", "2", "--no-cpu", "--no-catalog", "--no-cfg5", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert last_json_line(r.stdout)["steps"] == 3
    names = sorted(p.name for p in runs[0].iterdir())
    assert names == ["Cat.npy", "G.npy", "P_sample.npy", "R_sample.npy", "scalars.npy"]
    assert sum(p.stat().st_size for p in runs[0].iterdir()) <= 64 << 20
    for n in names:
        a, b = np.load(runs[0] / n), np.load(runs[1] / n)
        assert a.dtype == np.float32 and np.isfinite(a).all(), n
        if n == "scalars.npy":
            np.testing.assert_allclose(b, a, rtol=1e-5, atol=0, err_msg=n)
        else:
            assert_close(b, a, what=n)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(ROOT, "profiles", "r02_bench_*gpu.json"))))
def test_round2_gpu_lines_carry_the_contract(path):
    d = last_json_line(open(path).read())
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["metric"] == "bpr_train_triples_per_sec" and d["scaling"] == "weak" and d["dtype"] == "f32"
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0 and "workload" in d["config"] and d["single_pass"] is True
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"])
    rf, rs = d["roofline"], d["roofline_step"]
    assert rf["bound"] == "hbm" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9 and 0.4 < rf["frac"] < 1.0
    assert rs["bound"] == "hbm" and 0.3 < rs["frac"] < 1.0
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["value"] != d["value"] and "dense feed" in e["feed"]
    # BASELINE configs[4]: 1:8 sampled negatives, Adagrad, bf16 tables -- on one GPU and row-sharded, fp32 tables beside it
    c5 = d["cfg5"]
    assert c5["value"] > 0 and c5["same_leg_fp32_tables"]["value"] > 0 and 0.9 < c5["speedup_vs_fp32_tables"] < 2.0
    assert c5["roofline"]["bound"] == "hbm" and c5["roofline_step"]["frac"] > 0
    if d["n_gpus"] == 1:
        assert c5["topk"]["ms"] > 0 and c5["topk_health"]["ms"] >= c5["topk"]["ms"] and c5["e2e"]["h2d_bytes_per_step"] > 0
        assert d["topk"]["ms"] < 5.0                                    # sampled evaluation: 7.57 ms at the start of round 2
    else:
        assert c5["table_dtype"] == "bf16" and c5["sampled_negatives_per_positive"] == 8 and c5["overflow_flag"] == 0
    if d["n_gpus"] == 1:
        assert d["ms_per_step"] < 1.35                                  # round 1: 1.659
        assert abs(sorted(e["runs"])[1] - e["value"]) < 1e-6 * e["value"]   # the MEDIAN of the three runs
        assert d["cpu_baseline"]["kind"] == "port" and d["cfg1"]["cpu_baseline"]["value"] > 0 and d["cfg1"]["gpu_e2e"]["value"] > 0
        c2, c4 = d["catalog_topk"]
        assert c2["fallback_rows"] == 0 and c2["train_steps_before"] >= 400     # the catalog leg runs AFTER the training legs
        assert c4["users"] == 1_000_000 and c4["recipes"] == 10_000_000 and c4["fallback_rows"] == 0   # cfg4 in full
    else:
        sc = d["self_check"]
        assert sc["ok"] is True and sc["loss_rel_err"] <= 1e-5 and max(sc["table_rel_err"].values()) <= 1e-4
        assert d["shard_phases_ms"] and d["unrouted"]["value"] > 0 and d["e2e_compact"]["value"] > d["e2e"]["value"]
        assert d["value"] > 0.7 * d["n_gpus"] * 184e6                    # weak scaling at constant per-GPU work >= 70 %
        if d["n_gpus"] == 8:
            assert d["cfg3"]["value"] > 0 and d["cfg3"]["local_rows"]["users"] == 12_500_000
            assert "cfg4 IN FULL" in d["catalog_topk"][1]["workload"]


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(ROOT, "profiles", "r01c_bench_*gpu.json"))))
def test_committed_gpu_lines_carry_the_contract(path):
    d = last_json_line(open(path).read())
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["metric"] == "bpr_train_triples_per_sec" and d["scaling"] == "weak" and d["dtype"] == "f32"
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0 and "workload" in d["config"]
    clk = d["clocks"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(clk)
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(clk["reasons"])
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert 0.5 < rf["frac"] < 1.0          # the user pass: ~86 % of the measured copy bandwidth
    e = d["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e) and e["h2d_bytes_per_step"] > 0
    assert e["value"] != d["value"]        # measured separately, host buffers inside the timed region
    if d["n_gpus"] == 1:
        assert rf["traffic"] and rf["traffic"] >= 0.9 * rf["alg_bytes_per_launch"]     # ncu DRAM bytes vs algorithmic
        cb = d["cpu_baseline"]
        assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0 and cb["sample"]
        assert d["topk"]["value"] > 0 and d["pointwise"]["value"] > 0 and len(d["catalog_topk"]) == 2
        for c in d["catalog_topk"]:
            assert c["roofline"]["bound"] == "tensor" and c["fallback_rows"] == 0
    else:
        assert d["shard_phases_ms"] and d["value"] > 0.7 * d["n_gpus"] * 158e6     # weak scaling >= 70 %
