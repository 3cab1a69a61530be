"""Fixed mixture with an ODD number of components (what the training loop evaluates for component index 7, 5, 3) on the cfg3 shape:
the default handle (two-chain kernel on the even part + single-chain kernel on the last component where the cost model puts the
even part on two chains, one single-chain launch otherwise) vs the single-chain kernel on all of them (GBNF_TC4=0).
usage: python tools/odd_count_bench.py [--rows 65536]"""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import bench, gbnf_b200

p = argparse.ArgumentParser()
p.add_argument("--rows", type=int, default=65536, help="batch rows (the training loop's default batch is 512)")
rows = p.parse_args().rows
cfg = bench.CONFIGS["cfg3_miniboone"]
dev = torch.device("cuda", 0)
power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                       text=True).stdout.strip()
out = {"device": torch.cuda.get_device_name(dev), "power_limit": power, "rows": rows}
iters = max(100, min(2000, 100 * 65536 // rows))
for tag, env in (("default", None), ("single_chain", "0")):
    if env is None:
        os.environ.pop("GBNF_TC4", None)
    else:
        os.environ["GBNF_TC4"] = env
    torch.manual_seed(1)
    model = gbnf_b200.BoostedFlow(bench.make_args(cfg, dev), gemm_mode="f16fast").to(dev)
    x = torch.randn((max(rows, 4096), cfg["D"]), device=dev)
    model.train()
    with torch.no_grad():
        for c in range(cfg["C"]):
            model(x=x[:4096], components=c)
    model.eval()
    for p_ in model.parameters():
        p_.requires_grad_(False)
    model.pack_all()
    x = x[:rows].contiguous()
    for n in (7, 5, 3):
        for _ in range(20):
            model.mixture_log_density(x, n)
        torch.cuda.synchronize()
        l0 = model.info()["launches"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            model.mixture_log_density(x, n)
        e1.record(); torch.cuda.synchronize()
        out[f"{tag}.n{n}.ms"] = round(e0.elapsed_time(e1) / iters, 4)
        out[f"{tag}.n{n}.launches"] = (model.info()["launches"] - l0) // iters
    model.release()
print(json.dumps(out))
