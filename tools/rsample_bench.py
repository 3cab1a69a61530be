"""Sampling with gradients: BoostedFlow.rsample forward + backward through the fused inverse backward (gbnf_mixture_inverse +
gbnf_mixture_inverse_backward) against the autograd fallback (each component's rows through inverse_autograd), for cfg3 (Glow
D 43, K 5, h 512, C 8) and cfg2's RealNVP shape without BatchNorm (D 6, K 5, h 256, C 4: the fused backward serves RealNVP only
without BatchNorm), at n = 512, 4096 and 65 536 samples, with only the newest component trained and with all components
trained.  The loss is a reverse-KL-style sum over x and ldj.  The two arms alternate within one process over several rounds;
the median of each arm is reported.  The card's name and power limit are recorded with the numbers.

    python tools/rsample_bench.py [--rounds 5] [--iters 5] [--out file.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

CONFIGS = {
    "cfg3_miniboone": dict(kind="glow", D=43, C=8, K=5, h=512),
    "cfg2_power_no_bn": dict(kind="realnvp", D=6, C=4, K=5, h=256),
}


def step(model, n, z, comp):
    x, ldj, _ = model.rsample(n, z=z, comp=comp)
    (0.5 * (x * x).sum() - ldj.sum()).backward()


def main():
    p = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    p.add_argument("--ns", default="512,4096,65536")
    p.add_argument("--rounds", type=int, default=5)
    p.add_argument("--iters", type=int, default=5)
    p.add_argument("--mode", default="f16fast")
    p.add_argument("--out", default=None)
    a = p.parse_args()
    import torch
    from helpers import build_model
    from oracle import gbnf_oracle as orc
    from mixture_sample_bench import card, seconds_per_call
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    res = {"mode": a.mode, "rounds": a.rounds, "iters_per_round": a.iters, "card": card(), "results": []}
    for name, cfg in CONFIGS.items():
        md = orc.make_synthetic_model(cfg["kind"], cfg["D"], cfg["C"], cfg["K"], cfg["h"], seed=1, init_rows=2048)
        model = build_model(md, "cuda", gemm_mode=a.mode)
        try:
            model.component, model.all_trained = cfg["C"] - 1, True
            for trained in ("newest", "all"):
                for c, f in enumerate(model.flows):
                    for q in f.parameters():
                        q.requires_grad_(trained == "all" or c == cfg["C"] - 1)
                for n in map(int, a.ns.split(",")):
                    g = torch.Generator(device="cuda").manual_seed(n)
                    u = torch.rand(n, dtype=torch.float64, device="cuda", generator=g)
                    z = torch.randn((n, cfg["D"]), device="cuda", generator=g)
                    comp = model.assign_components(u)
                    arms = {"fused": [], "fallback": []}
                    for r in range(a.rounds + 1):            # round 0 warms both arms up
                        for arm in ("fused", "fallback"):
                            model.fused_backward = arm == "fused"
                            t = seconds_per_call(lambda: step(model, n, z, comp), a.iters)
                            if r:
                                arms[arm].append(t)
                    model.fused_backward = True
                    model.check_status()
                    med = {k: sorted(v)[len(v) // 2] for k, v in arms.items()}
                    row = {"config": name, "trained": trained, "n": n, "fused_s": arms["fused"], "fallback_s": arms["fallback"],
                           "fused_median_ms": med["fused"] * 1e3, "fallback_median_ms": med["fallback"] * 1e3,
                           "speedup_median": med["fallback"] / med["fused"]}
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
