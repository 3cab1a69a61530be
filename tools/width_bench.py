"""Throughput of hidden widths the f16 tensor-core kernels serve by zero padding, next to the padded width itself and to the
fp32 CUDA-core path: the fused mixture log-density (gbnf_fused_eval, every component of the model) in samples/s.

    python tools/width_bench.py OUT_DIR

Groups (f16fast unless named):
  glow_d43_c8_k5      h = 215 (padded to 256) vs h = 256 vs fp32 at h = 215   (upstream's getting-started h = 5 x 43)
  glow_d43_c8_k5_h430 h = 430 (padded to 512) vs h = 512
  glow_d63_c8_k10     h = 630 (padded to 1024, CTA-pair kernel) vs h = 1024
  realnvp_d63_c8_k10  h = 1024 on the CTA-pair kernel vs fp32
TFLOP/s is stated from the TRUE h (the algorithmic work of bench.flops_per_sample) with the padded FLOPs next to it.  Writes
OUT_DIR/width_bench.json (with the card's name, power limit and maximum SM clock) and prints it.  Timing: CUDA events around
back-to-back calls after a warm-up, at least 1 s of timed work per arm; the arms of a group alternate over three rounds (fp32
arms: one round) so that their ratio comes with its spread.  The 65 536-row batch is 11 - 17 MB, so it stays L2-resident."""
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
GLOW43 = dict(kind="glow", D=43, C=8, K=5, bn=False, toy=False, rho="decreasing")
GLOW63 = dict(kind="glow", D=63, C=8, K=10, bn=False, toy=False, rho="decreasing")
RNVP63 = dict(kind="realnvp", D=63, C=8, K=10, bn=False, toy=False, rho="decreasing")
GROUPS = {   # name -> [(arm, shape, h, gemm_mode)]
    "glow_d43_c8_k5": [("h215_f16fast", GLOW43, 215, "f16fast"), ("h256_f16fast", GLOW43, 256, "f16fast"),
                       ("h215_fp32", GLOW43, 215, "fp32")],
    "glow_d43_c8_k5_h430": [("h430_f16fast", GLOW43, 430, "f16fast"), ("h512_f16fast", GLOW43, 512, "f16fast")],
    "glow_d63_c8_k10": [("h630_f16fast", GLOW63, 630, "f16fast"), ("h1024_f16fast", GLOW63, 1024, "f16fast")],
    "realnvp_d63_c8_k10": [("h1024_f16fast", RNVP63, 1024, "f16fast"), ("h1024_fp32", RNVP63, 1024, "fp32")],
}


def padded(h):
    """The width the f16 tensor-core kernels run (gbnf_api.cu plan_layout, depth 1)."""
    if h % 64 and h <= 512:
        return -(-h // 128) * 128
    return 1024 if 512 < h <= 1024 else h


def timed(fn, min_s=MIN_SECONDS):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n, s = max(3, math.ceil(min_s / (e0.elapsed_time(e1) / 1e3))), 0.0
    while s < min_s:
        if s > 0.0:
            n = math.ceil(1.1 * n * min_s / s)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        s = e0.elapsed_time(e1) / 1e3
    return n * B / s


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    power, clock = (v.strip() for v in q.stdout.strip().split(","))
    return {"device": torch.cuda.get_device_name(index), "power_limit": power, "clocks_max_sm": clock}


def make_model(shape, h, mode, dev, x):
    cfg = dict(shape, h=h)
    torch.manual_seed(1)           # the benchmark's recipe: product constructors under seed 1, ActNorm / BatchNorm from data rows
    model = gbnf_b200.BoostedFlow(bench.make_args(cfg, dev), gemm_mode=mode).to(dev)
    model.train()
    with torch.no_grad():
        for c in range(cfg["C"]):
            model(x=x[:4096], components=c)
    model.eval()
    for p in model.parameters():
        p.requires_grad_(False)
    return model, cfg


def main():
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    out_dir = sys.argv[1]
    if not torch.cuda.is_available():
        raise SystemExit("width_bench.py measures the GPU kernels: no CUDA device")
    dev = torch.device("cuda", 0)
    res = {"rows": B, "unit": "samples/s (fused mixture log-density over all C components)"}
    res.update(card(0))
    for name, arms in GROUPS.items():
        x = torch.randn((B, arms[0][1]["D"]), device=dev, generator=torch.Generator(device=dev).manual_seed(1234))
        models = [make_model(shape, h, mode, dev, x) for _, shape, h, mode in arms]
        rates = {arm: [] for arm, *_ in arms}
        for rnd in range(3):
            for (arm, _, _, mode), (model, cfg) in zip(arms, models):
                if mode == "fp32" and rnd > 0:
                    continue
                rates[arm].append(timed(lambda: model.mixture_log_density(x, cfg["C"])))
        group = {}
        for (arm, _, h, mode), (model, cfg) in zip(arms, models):
            model.check_status()
            inf = model.info()
            hp = padded(h) if mode != "fp32" else h
            fl_true, fl_pad = bench.flops_per_sample(cfg), bench.flops_per_sample(dict(cfg, h=hp))
            best = max(rates[arm])
            group[arm] = {"h": h, "h_run": hp, "gemm_mode": mode, "kernel": {0: "serial/fp32", 1: "pipelined", 2: "cta_pair"}[inf["pipelined"]],
                          "two_chain": inf["two_chain"], "samples_per_s": rates[arm], "tflops_true_h": best * fl_true / 1e12,
                          "tflops_padded": best * fl_pad / 1e12, "flops_per_sample_true_h": fl_true, "flops_per_sample_padded": fl_pad}
        G0 = models[0][0].mixture_log_density(x[:4096], models[0][1]["C"])
        for (arm, *_), (model, cfg) in zip(arms[1:], models[1:]):
            if cfg["h"] == models[0][1]["h"]:   # same model in another GEMM mode: how far apart are the results
                group[arm]["max_abs_diff_G_vs_first_arm"] = float((model.mixture_log_density(x[:4096], cfg["C"]) - G0).abs().max())
        for model, _ in models:
            model.release()
        res[name] = group
        print(name, json.dumps(group), flush=True)
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "width_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
