"""Sampling-direction throughput at the cfg5 shape (BSDS300: Glow, D = 63, K = 10, h = 1024), batch 65 536, one component:
gbnf_component_inverse in f16fast and f16 (CTA-pair kernel, coupling_tc3.cuh with INV = 1) and in fp32 (CUDA-core inverse
kernel), next to gbnf_component_forward of the same component in f16fast (the same GEMMs in the forward direction).

    python tools/sample_bench.py OUT_DIR

Writes OUT_DIR/sample_bench_cfg5.json (rows/s per arm, the card's name, power limit and maximum SM clock) and prints it.
Timing: CUDA events around back-to-back calls after a warm-up, at least 1 s of timed work per arm; the f16fast inverse and
forward arms alternate over three rounds so that their ratio comes with its spread.  The z / x batch (16.5 MB) and one
component's packed weights (~21 MB) both fit in the 126 MB L2, so every arm runs L2-resident after its first call."""
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import torch  # noqa: E402

import bench  # noqa: E402
import gbnf_b200  # noqa: E402

B = 65536
MIN_SECONDS = 1.0


def timed(fn, min_s=MIN_SECONDS):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n, s = max(5, math.ceil(min_s / (e0.elapsed_time(e1) / 1e3))), 0.0
    while s < min_s:          # the calibration call can be slower than the steady state: repeat until the window is long enough
        if s > 0.0:
            n = math.ceil(1.1 * n * min_s / s)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3
    return {"rows_per_s": n * B / s, "calls": n, "seconds": s, "ms_per_call": 1e3 * s / n}


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    power, clock = (v.strip() for v in q.stdout.strip().split(","))
    return {"device": torch.cuda.get_device_name(index), "power_limit": power, "clocks_max_sm": clock}


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    out_dir = sys.argv[1]
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench.py measures the GPU kernels: no CUDA device")
    dev = torch.device("cuda", 0)
    cfg = bench.CONFIGS["cfg5_bsds300"]
    D = cfg["D"]
    # the benchmark's model recipe: product constructors under seed 1, ActNorm initialised from 4096 data rows
    torch.manual_seed(1)
    model = gbnf_b200.BoostedFlow(bench.make_args(cfg, dev), gemm_mode="f16fast").to(dev)
    x = torch.randn((B, D), device=dev, generator=torch.Generator(device=dev).manual_seed(1234))
    model.train()
    with torch.no_grad():
        for c in range(cfg["C"]):
            model(x=x[:4096], components=c)
    model.eval()
    for p in model.parameters():
        p.requires_grad_(False)
    c = 0
    z = torch.randn((B, D), device=dev, generator=torch.Generator(device=dev).manual_seed(99))

    res = {"config": "cfg5_bsds300", "shape": dict(kind="glow", D=D, K=cfg["K"], h=cfg["h"]), "rows": B, "component": c,
           "unit": "rows/s (one component)"}
    res.update(card(0))

    model.gemm_mode = "f16fast"
    assert model.info()["pipelined"] == 2, model.info()
    rounds = []
    for _ in range(3):
        inv = timed(lambda: model.component_inverse(z, c))
        fwd = timed(lambda: model.component_forward(x, c))
        rounds.append({"inverse": inv["rows_per_s"], "forward": fwd["rows_per_s"], "inverse_over_forward": inv["rows_per_s"] / fwd["rows_per_s"]})
    res["f16fast_rounds"] = rounds
    zf, _ = model.component_forward(x, c)
    xr, _ = model.component_inverse(zf, c)
    res["f16fast_round_trip_max_abs_err"] = float((xr - x).abs().max())
    x_f16fast, _ = model.component_inverse(z, c)

    model.gemm_mode = "f16"
    assert model.info()["pipelined"] == 2, model.info()
    res["f16_inverse"] = timed(lambda: model.component_inverse(z, c))
    x_f16, _ = model.component_inverse(z, c)

    model.gemm_mode = "fp32"
    res["fp32_inverse"] = timed(lambda: model.component_inverse(z, c))
    x_fp32, _ = model.component_inverse(z, c)
    model.check_status()
    model.release()

    best = max(rounds, key=lambda r: r["inverse"])
    res["summary"] = {
        "f16fast_inverse_rows_per_s": [r["inverse"] for r in rounds],
        "f16fast_forward_rows_per_s": [r["forward"] for r in rounds],
        "f16fast_inverse_over_forward": [r["inverse_over_forward"] for r in rounds],
        "f16_inverse_rows_per_s": res["f16_inverse"]["rows_per_s"],
        "fp32_inverse_rows_per_s": res["fp32_inverse"]["rows_per_s"],
        "f16fast_inverse_over_fp32_inverse": best["inverse"] / res["fp32_inverse"]["rows_per_s"],
        "f16_inverse_over_fp32_inverse": res["f16_inverse"]["rows_per_s"] / res["fp32_inverse"]["rows_per_s"],
        "max_abs_diff_f16fast_vs_fp32_inverse": float((x_f16fast - x_fp32).abs().max()),
        "max_abs_diff_f16_vs_fp32_inverse": float((x_f16 - x_fp32).abs().max()),
    }
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "sample_bench_cfg5.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
