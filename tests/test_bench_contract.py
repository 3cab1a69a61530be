"""CPU checks of bench.py's contract pieces that need no GPU: the algorithmic FLOP counts the roofline uses (SURVEY 8d), the
reference arm's JSON line (run here on a tiny configuration), and the arguments the driver passes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

# SURVEY 8(d) table: algorithmic FLOP / sample (2 MAC, MLPs only)
SURVEY_FLOPS = {"cfg1_toy": 2113536, "cfg2_power": 5365760, "cfg3_miniboone": 23633920, "cfg4_hepmass": 89128960,
                "cfg5_bsds300": 183336960}


@pytest.mark.parametrize("name", list(SURVEY_FLOPS))
def test_flops_per_sample_match_survey(name):
    assert bench.flops_per_sample(bench.CONFIGS[name]) == SURVEY_FLOPS[name]


def test_peaks_have_the_keys_the_roofline_uses():
    pk = bench.peaks()
    assert set(pk) >= {"bf16_burst", "bf16_sustained", "hbm", "source"}
    assert pk["bf16_burst"] >= pk["bf16_sustained"] > 0 and pk["hbm"] > 0


def test_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` is the CPU arm (oracle port on the host threads): one JSON line with the base contract's keys,
    impl = reference, a cpu_baseline describing the run and an e2e object that repeats the line's own value."""
    env = dict(os.environ, OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cfg1_toy",
                          "--steps", "1", "--warmup", "1", "--batch", "256"], capture_output=True, text=True, env=env,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0
    staged = os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "models", "boosted_flow.py"))
    assert d["cpu_baseline"]["kind"] == ("reference" if staged else "port") and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_port_fallback():
    """Without the staged reference (or with --port) the arm times the oracle's torch-CPU port and says so."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--port", "--config", "cfg1_toy",
                          "--steps", "1", "--warmup", "1", "--batch", "256"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0


def test_staged_reference_matches_its_source():
    if not os.path.isdir("/root/reference"):
        pytest.skip("the reference tree only exists in the build container")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "baseline", "vendor_reference.py"), "--check"], capture_output=True,
                         text=True)
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref")):
        pytest.skip("baseline/_ref not staged yet (python __graft_entry__.py build stages it)")
    assert out.returncode == 0, out.stdout + out.stderr


def test_dump_outputs_writes_float32_rows(tmp_path):
    import numpy as np
    import torch
    G, w = torch.randn(1000), torch.rand(1000)
    bench.dump_outputs(str(tmp_path / "d"), {"mixture_log_density": G, "boosting_weights": w})
    for name, t in (("mixture_log_density", G), ("boosting_weights", w)):
        a = np.load(tmp_path / "d" / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy())


def test_dump_outputs_samples_the_same_rows_under_the_byte_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    G = torch.arange(5000, dtype=torch.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"mixture_log_density": G, "boosting_weights": -G})
    a = np.load(tmp_path / "a" / "mixture_log_density.npy")
    assert a.shape == (500,) and np.all(np.diff(a) > 0)                   # 4000 bytes / 8 bytes per row, in row order
    assert np.array_equal(np.load(tmp_path / "a" / "boosting_weights.npy"), -a)
    assert np.array_equal(np.load(tmp_path / "b" / "mixture_log_density.npy"), a)


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and out.stdout == ""


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path(tmp_path):
    """Two runs with the same arguments time exactly --steps steps and dump the same G_ll and weights of the last one."""
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "cfg1_toy", "--batch", "4096", "--rows", "16384",
                              "--steps", "5", "--warmup", "3", "--no-cpu", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
        assert d["steps"] == 5 and d["value"] > 0
        dumps.append({n: np.load(tmp_path / run / (n + ".npy")) for n in ("mixture_log_density", "boosting_weights")})
    for n, v in dumps[0].items():
        assert v.dtype == np.float32 and v.shape == (4096,) and np.isfinite(v).all(), n
        np.testing.assert_allclose(dumps[1][n], v, rtol=1e-6, atol=0)
    assert abs(float(dumps[0]["boosting_weights"].astype(np.float64).sum()) - 1.0) < 1e-4


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, env=env, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""
