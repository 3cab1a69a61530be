#!/usr/bin/env python
"""One TRAINING step of the boosted objective (density_experiment.py:359-374: compute_kl_pq_loss -> backward -> clip -> optimizer
step) on cfg3's architecture, component C-1 being trained: this library (fixed mixture + weights + resampling kernels, new
component forward and backward through gbnf_component_backward) against the same host code with the new component on torch
autograd, and against the UNMODIFIED reference moved to the same GPU.  --depth sets coupling_network_depth (cfg3 itself has
depth 1); the reference arm builds depth-1 networks only, so at any other depth its column is null and the JSON says why.
Prints one JSON line with the card's name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "baseline"))
import bench  # noqa: E402
import gbnf_b200  # noqa: E402


def time_steps(step, n, warm=5):
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def ours(cfg, dev, batch, fused, mode, n, depth):
    torch.manual_seed(1)
    a = bench.make_args(cfg, dev)
    a.coupling_network_depth = depth
    a.fused_backward = fused
    model = gbnf_b200.BoostedFlow(a, gemm_mode=mode).to(dev)
    x = torch.randn((batch, cfg["D"]), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    model.train()
    with torch.no_grad():
        for c in range(cfg["C"]):
            model(x=x, components=c)
    C = cfg["C"]
    model.component, model.all_trained = C - 1, False
    for i, f in enumerate(model.flows):
        for p in f.parameters():
            p.requires_grad_(i == C - 1)
    opt = torch.optim.Adam(list(model.flows[C - 1].parameters()), lr=1e-4)
    assert model._fused_backward_ok(x) == fused, "the fused arm must train through gbnf_component_backward"
    largs = argparse.Namespace(flow="boosted")
    gen = torch.Generator(device=dev).manual_seed(3)

    def step():
        opt.zero_grad(set_to_none=True)
        losses = gbnf_b200.compute_kl_pq_loss(model, x, largs, generator=gen)
        losses["nll"].backward()
        torch.nn.utils.clip_grad_norm_(model.flows[C - 1].parameters(), 5.0)
        opt.step()
    ms = time_steps(step, n)
    model.release()
    return ms


def reference(cfg, dev, batch, n):
    import ref_harness as rh
    if not rh.available():
        return None
    ref = rh.load()
    import types
    for name in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    import density_experiment as de
    x = torch.randn((batch, cfg["D"]), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    model, args = rh.build_model(ref, cfg, dev, x)
    model.train()
    C = cfg["C"]
    model.component, model.all_trained = C - 1, False
    for n_, p in model.named_parameters():
        p.requires_grad_(n_.startswith(f"flows.{C - 1}."))
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        losses = de.compute_kl_pq_loss(model, x, args)
        losses["nll"].backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 5.0)
        opt.step()
    return time_steps(step, n)


def card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(index), "power_limit": q.stdout.strip()}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--config", default="cfg3_miniboone")
    p.add_argument("--batches", default="512,4096")
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--mode", default="f16fast")
    p.add_argument("--depth", type=int, default=1, help="coupling_network_depth of every coupling network (0 .. 4)")
    a = p.parse_args()
    cfg = bench.CONFIGS[a.config]
    dev = torch.device("cuda", 0)
    out = {"what": f"one training step of component {cfg['C'] - 1} of {a.config} (fixed mixture of {cfg['C'] - 1} components + weights + resampling + "
                   "new-component forward/backward + clip + Adam)", "mode": a.mode, "coupling_network_depth": a.depth,
           **card(0), "rows": []}
    if a.depth != 1:
        out["reference_note"] = ("null: baseline/ref_harness builds the reference with coupling_network_depth 1 only, so the reference "
                                 f"arm has no depth-{a.depth} model")
    for b in [int(v) for v in a.batches.split(",")]:
        row = {"batch": b,
               "library_fused_backward_ms": ours(cfg, dev, b, True, a.mode, a.steps, a.depth),
               "library_torch_autograd_new_component_ms": ours(cfg, dev, b, False, a.mode, a.steps, a.depth),
               "reference_eager_same_gpu_ms": reference(cfg, dev, b, a.steps) if a.depth == 1 else None}
        row["samples_per_s_fused"] = b / (row["library_fused_backward_ms"] * 1e-3)
        out["rows"].append(row)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
