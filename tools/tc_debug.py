"""GPU-side diagnostic for the tensor-core path: smallest fixtures, per-component error vs the oracle."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch
from helpers import build_model, golden_model
from oracle import gbnf_oracle as orc
from tests.golden import store

names = sys.argv[1:] or ["glow_d43", "realnvp_d6_bn", "glow_d6_additive_relu", "realnvp_d5_mixed", "toy_d2"]
for mode in ("f16", "f16fast"):
    for name in names:
        g = store.load(name)
        md = golden_model(g)
        model = build_model(md, "cuda", gemm_mode=mode)
        x = torch.from_numpy(g["x"]).cuda()
        lq = model.component_log_density(x).cpu().numpy()
        torch.cuda.synchronize()
        ref = g["logq64"]
        rel = np.abs(lq - ref) / np.abs(ref)
        print(f"[{mode}] {name}: max rel err per component {rel.max(0)}  info={model.info()}")
        if not np.isfinite(lq).all() or rel.max() > 1e-3:
            z, ldj = model.component_forward(x, 0)
            print("  row0 lq", lq[0], "ref", ref[0])
            print("  z[0,:8]", z[0, :8].cpu().numpy(), "ref", g["z64"][0][0, :8])
            print("  ldj[:4]", ldj[:4].cpu().numpy(), "ref", g["ldj64"][0][:4])
        model.release()
print("TC DEBUG DONE")
