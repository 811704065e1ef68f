"""bench.py's output contract (keys the driver parses), checked on the recorded B200 lines under profiles/ and on the CLI."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"metric": str, "value": (int, float), "unit": str, "n_gpus": int, "steps": int, "warmup": int,
            "ms_per_step": (int, float), "higher_is_better": bool, "scaling": str, "dtype": str, "data": str, "config": dict,
            "clocks": dict, "e2e": dict}


def _line(path):
    with open(os.path.join(ROOT, path)) as f:
        for l in f:
            if l.startswith("{"):
                return json.loads(l)
    raise AssertionError(f"no JSON line in {path}")


@pytest.mark.parametrize("path", ["profiles/r1_bench_ours_n1.json.log", "profiles/r1_bench_ddp_n2.json.log",
                                  "profiles/r1_bench_fp32_ours_n1.json", "profiles/r1_bench_reference_n1_final.json.log",
                                  "profiles/r2_bench_n1_final_TDS_NONE_1.json", "profiles/r2_bench_n2_bisect_TDS_PDL_0.json",
                                  "profiles/r2_final2_ours_n8.json", "profiles/r2_final_ours_n8.json", "profiles/r2_final_ref_n8.json",
                                  "profiles/r2_bench_reference_n1_modes.json"])
def test_recorded_bench_lines_follow_the_contract(path):
    d = _line(path)
    for k, t in REQUIRED.items():
        assert k in d and isinstance(d[k], t), (k, d.get(k))
    assert "vs_baseline" in d
    assert d["metric"] == "gpt2_train_tokens_per_sec" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["warmup"] >= 3
    assert {"model", "global_batch", "seq_len", "parallelism"} <= set(d["config"])
    assert d["config"]["model"] == "gpt2-small" and d["config"]["seq_len"] == 1024
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    tokens = d["config"]["global_batch"] * d["config"]["seq_len"]
    assert d["value"] == pytest.approx(tokens / (d["ms_per_step"] * 1e-3), rel=1e-6)     # whole-job tokens/s
    if d.get("impl") == "ours":
        assert d["e2e"]["value"] <= d["value"] * 1.02      # e2e adds the copies (the host-bound reference arm varies +-8 % run to run)
        assert d["gpu_launches"] > 0 and d["launches_per_step"] > 100


def test_round2_lines_carry_modes_and_comm_check():
    """Round 2 additions: both arms report the same `config` block; the multi-GPU line of our arm carries `comm_check`
    (collectives vs NCCL + bit-identical replicas) and, by default, the `modes` block with the other BASELINE.json configs."""
    ours, ref = _line("profiles/r2_final_ours_n8.json"), _line("profiles/r2_final_ref_n8.json")
    assert ours["config"] == ref["config"] and ours["impl"] == "ours" and ref["impl"] == "reference"
    assert ours["comm_check"]["ok"] is True and ours["comm_check"]["replicas_bit_identical"] is True
    assert {c["size"] for c in ours["comm_check"]["cases"]} == {"3KB", "2.4MB", "77MB"}
    assert set(ours["modes"]) == {"zero1-medium", "zero2-large", "zero3-xl"}
    for m in ours["modes"].values():
        assert m["ms_per_step"] > 0 and m["value"] > 0 and m["peak_hbm_bytes"] > 0 and "exposed_comm_ms_per_step" in m
    assert ours["value"] / ref["value"] > 10          # the ratio the tables in BASELINE.md quote
    final = _line("profiles/r2_final2_ours_n8.json")
    assert final["n_gpus"] == 8 and final["comm_check"]["ok"] is True and final["value"] > ours["value"]


def test_bench_cli_parses_on_cpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dtype", "--mode", "--dump-outputs"):
        assert flag in r.stdout


def test_dump_outputs_writes_float32_sampled_reproducible_arrays(tmp_path, monkeypatch):
    """bench.dump_outputs: loss + every parameter + its fp32 master as float32 .npy, long arrays cut to the per-array share
    of the budget at name-seeded positions, so two dumps of the same state are identical."""
    import importlib.util
    import numpy as np
    import torch
    import tiny_deepspeed_b200 as tds
    from tiny_deepspeed_b200.models.gpt2 import GPT2Model, gpt2_config

    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    monkeypatch.setattr(bench, "DUMP_BUDGET", 20000)
    torch.manual_seed(0)
    model = GPT2Model(gpt2_config("tiny")).to(torch.bfloat16)
    opt = tds.AdamW(model.named_parameters(), lr=1e-3)
    names = bench.dump_outputs(str(tmp_path / "a"), torch.tensor(2.5), opt)
    assert bench.dump_outputs(str(tmp_path / "b"), torch.tensor(2.5), opt) == names
    params = dict(model.named_parameters())
    assert names[0] == "loss"
    assert sorted(names[1:]) == sorted([f"param.{n}" for n in params] + [f"master.{n}" for n in params])
    keep = min(1000, 20000 // len(names))
    total = 0
    for n in names:
        a, b = np.load(tmp_path / "a" / f"{n}.npy"), np.load(tmp_path / "b" / f"{n}.npy")
        assert a.dtype == np.float32 and a.ndim == 1 and np.array_equal(a, b), n
        total += a.size
        if n == "loss":
            assert a.tolist() == [2.5]
            continue
        src = params[n.split(".", 1)[1]].detach().float().reshape(-1).numpy()
        assert a.size == min(src.size, keep), n
        if src.size <= keep:
            assert np.array_equal(a, src), n
        else:
            assert np.isin(a, src).all(), n
    assert total <= 20000
