"""Mixture sampling throughput: BoostedFlow.sample() -- one gbnf_mixture_inverse call, one coupling launch over every component's
rows -- against the per-component loop it replaced (C + 1 host synchronisations, a gather, an inverse launch and a scatter per
component), at n = 65 536 samples of cfg3 (pipelined kernel), cfg5 (CTA-pair kernel) and cfg2 (RealNVP, pipelined kernel), in the
f16fast and f16 modes.  The two arms alternate within one process over several rounds; both are checked to give the same bits
first.  The card's name and power limit are recorded with the numbers.

    python tools/mixture_sample_bench.py [--n 65536] [--rounds 3] [--iters 10] [--out file.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CONFIGS = {
    "cfg3_miniboone": dict(kind="glow", D=43, C=8, K=5, h=512, batch_norm=False),
    "cfg5_bsds300": dict(kind="glow", D=63, C=8, K=10, h=1024, batch_norm=False),
    "cfg2_power": dict(kind="realnvp", D=6, C=4, K=5, h=256, batch_norm=True),
}


def per_component_sample(model, u, z):
    """sample() as it was before gbnf_mixture_inverse: one inverse launch per component present in the batch."""
    import torch
    comp = model.assign_components(u)
    x = torch.empty_like(z)
    for c in torch.unique(comp).tolist():
        rows = torch.nonzero(comp == c, as_tuple=False).squeeze(1)
        x[rows] = model.component_inverse(z[rows].contiguous(), int(c))[0]
    return x, comp


def seconds_per_call(fn, iters):
    import torch
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / 1e3 / iters


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["max_sm_clock_mhz"] = float(q[0]), float(q[1])
    except Exception as e:   # the numbers still stand; say why the card's limits are missing
        out["power_limit_w"] = None
        out["query_error"] = str(e)
    return out


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--n", type=int, default=65536)
    p.add_argument("--rounds", type=int, default=3)
    p.add_argument("--iters", type=int, default=10)
    p.add_argument("--configs", default=",".join(CONFIGS))
    p.add_argument("--modes", default="f16fast,f16")
    p.add_argument("--out", default=None)
    a = p.parse_args()
    import torch
    from helpers import build_model
    from oracle import gbnf_oracle as orc
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    res = {"n": a.n, "rounds": a.rounds, "iters_per_round": a.iters, "card": card(), "results": []}
    for name in a.configs.split(","):
        cfg = CONFIGS[name]
        md = orc.make_synthetic_model(cfg["kind"], cfg["D"], cfg["C"], cfg["K"], cfg["h"], seed=1, batch_norm=cfg["batch_norm"],
                                      init_rows=2048)
        for mode in a.modes.split(","):
            model = build_model(md, "cuda", gemm_mode=mode)
            try:
                model.component, model.all_trained = cfg["C"] - 1, True
                g = torch.Generator(device="cuda").manual_seed(1)
                u = torch.rand(a.n, dtype=torch.float64, device="cuda", generator=g)
                z = torch.randn((a.n, cfg["D"]), device="cuda", generator=g)
                x_new, c_new = model.sample(a.n, u=u, z=z)
                x_old, c_old = per_component_sample(model, u, z)
                same = bool(torch.equal(x_new, x_old) and torch.equal(c_new, c_old))
                fused, loop = [], []
                for _ in range(a.rounds):
                    fused.append(a.n / seconds_per_call(lambda: model.sample(a.n, u=u, z=z), a.iters))
                    loop.append(a.n / seconds_per_call(lambda: per_component_sample(model, u, z), a.iters))
                model.check_status()
                row = {"config": name, "mode": mode, "kernel": "CTA pair" if model.info()["pipelined"] == 2 else "pipelined",
                       "bitwise_equal": same, "fused_rows_per_s": fused, "loop_rows_per_s": loop,
                       "speedup_median": sorted(f / l for f, l in zip(fused, loop))[len(fused) // 2]}
                print(json.dumps(row), flush=True)
                res["results"].append(row)
            finally:
                model.release()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
