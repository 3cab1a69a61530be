#!/usr/bin/env python
"""Benchmark of the boosted-mixture density path (BASELINE.json metric: boosted mixture log-density samples/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg3_miniboone] [--mode f16|fp32]
                    [--dump-outputs DIR]

A "step" is ONE pass of the hot path over ONE eval batch (default 65 536 rows) of synthetic N(0,1) rows:
fused per-component log q_c + rho-weighted logsumexp (one kernel) followed by the boosting weights.  Rows are
resident in HBM for `value` (the resident set, 2^20 rows, is larger than L2 and the batches rotate through it);
`e2e` runs the same step through the public Python API from pinned HOST buffers with the H2D / D2H copies inside
the timed region.  Multi-GPU = batch-parallel weak scaling: every rank evaluates its own batch, the boosting
weights use the global softmax (three scalar all-reduces over NCCL); `--parallel component` shards the components
instead (every rank sees the batch, one all-gather of [B, C/G] log q per step, strong scaling).  One JSON line on
stdout (rank 0).  `--dump-outputs DIR` also writes what the last timed step returned (rank 0), so that two builds run with
the same arguments, hence on the same seeded model and rows, can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree (it may be read-only)

CONFIGS = {   # BASELINE.json "configs" / SURVEY 8(d)
    "cfg1_toy": dict(kind="realnvp", D=2, C=8, K=1, h=256, bn=False, toy=True, rho="uniform"),
    "cfg2_power": dict(kind="realnvp", D=6, C=4, K=5, h=256, bn=True, toy=False, rho="decreasing"),
    "cfg3_miniboone": dict(kind="glow", D=43, C=8, K=5, h=512, bn=False, toy=False, rho="decreasing"),
    "cfg4_hepmass": dict(kind="glow", D=21, C=16, K=10, h=512, bn=False, toy=False, rho="decreasing"),
    "cfg5_bsds300": dict(kind="glow", D=63, C=8, K=10, h=1024, bn=False, toy=False, rho="decreasing"),
}
METRIC = "boosted_mixture_logdensity_samples_per_sec"
UNIT = "samples/s"
DUMP_BYTES = 60 << 20      # --dump-outputs: at most 64 MB in all, .npy headers included


def dump_outputs(out_dir, outputs):
    """Writes each per-row output as out_dir/<name>.npy (float32).  When the rows would exceed DUMP_BYTES, every output keeps
    the same fixed, seeded sample of rows (in row order), so files of two runs with the same arguments still line up."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outputs.items()}
    rows = len(next(iter(arrays.values())))
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if rows * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(rows, DUMP_BYTES // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def flops_per_sample(cfg, depth=1):
    """Algorithmic FLOPs (2*MAC, coupling MLPs only), SURVEY 8(d)."""
    D, h, K, C = cfg["D"], cfg["h"], cfg["K"], cfg["C"]
    h0, h1 = D // 2, D - D // 2
    if cfg["kind"] == "glow":
        step = 2 * (h0 * h + depth * h * h + h * 2 * h1)
        return step * K * C
    total = 0
    for c in range(C):
        for k in range(K):
            i, o = (h1, h0) if (k + c) % 2 else (h0, h1)
            total += 2 * 2 * (i * h + depth * h * h + h * o)
    return total


def make_args(cfg, device):
    import torch
    return argparse.Namespace(
        flow="boosted", boosted=True, density_evaluation=True, device=torch.device(device), cuda=device != "cpu",
        component_type=cfg["kind"], num_components=cfg["C"], num_flows=cfg["K"], z_size=cfg["D"], input_size=[cfg["D"]],
        h_size=cfg["h"], rho_init=cfg["rho"], coupling_network="tanh", coupling_network_depth=1, batch_norm=cfg["bn"],
        flow_permutation="shuffle", flow_coupling="affine", actnorm_scale=1.0, LU_decomposed=True, num_blocks=1,
        num_dequant_blocks=0, learn_top=False, y_classes=1, y_condition=False, sample_size=16, save_results=False,
        batch_size=100, rho_iters=0, toy_base=cfg["toy"])


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_burst": d["bf16_tflops"], "bf16_sustained": d["bf16_tflops_sustained"], "hbm": d["hbm_gbs"],
                "source": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines, self.proc = [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        for ts, ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 8 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


def cpu_port_throughput(cfg_name, rows, repeats=1):
    """The oracle (numpy port of the reference algorithm) on the host cores: C component log q + mixture + weights."""
    import numpy as np
    from oracle import gbnf_oracle as orc
    try:
        from threadpoolctl import threadpool_info
        threads = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        threads = os.cpu_count()
    cfg = CONFIGS[cfg_name]
    md = orc.make_synthetic_model(cfg["kind"], cfg["D"], cfg["C"], cfg["K"], cfg["h"], seed=1, batch_norm=cfg["bn"],
                                  rho_init=cfg["rho"], toy_base=cfg["toy"], init_rows=2048)
    import torch
    torch.set_num_threads(os.cpu_count())
    threads = torch.get_num_threads()
    tm = orc.to_torch_model(md)
    x = torch.from_numpy(np.random.default_rng(1234).standard_normal((rows, cfg["D"])).astype(np.float32))

    def one(xb):
        with torch.no_grad():
            return orc.torch_density_step(tm, xb)
    one(x[: min(rows, 2048)])   # warm-up (thread pool, page faults)
    best = float("inf")
    for _ in range(repeats):
        t = time.perf_counter()
        for s in range(0, rows, 8192):
            one(x[s:s + 8192])
        best = min(best, time.perf_counter() - t)
    return rows / best, threads, best


def _ref_harness():
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import ref_harness
    return ref_harness


def cpu_baseline_leg(a):
    """`cpu_baseline` of our arm's line: ~10-30 s of the reference's CPU path on the host cores (rank 0, N = 1)."""
    rh = _ref_harness()
    if rh.available():
        import torch
        ref = rh.load()
        cfg = CONFIGS[a.config]
        torch.set_num_threads(os.cpu_count())
        g = torch.Generator().manual_seed(1234)
        x_init = torch.randn((4096, cfg["D"]), generator=g)
        model, args = rh.build_model(ref, cfg, "cpu", x_init)
        rows = min(a.batch, 65536)
        x = torch.randn((rows, cfg["D"]), generator=g)
        rh.density_step(ref, model, x[:4096], args, toy=cfg["toy"])           # warm-up
        t = time.perf_counter()
        n = 0
        while n == 0 or (time.perf_counter() - t < 10.0 and n < 8):
            rh.density_step(ref, model, x, args, toy=cfg["toy"])
            n += 1
        secs = time.perf_counter() - t
        return {"value": rows * n / secs, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "reference",
                "sample": f"{n} x {rows} rows of {a.config}, unmodified reference (baseline/_ref) on torch CPU, {secs:.1f} s"}
    v, threads, secs = cpu_port_throughput(a.config, a.cpu_rows)
    return {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{a.cpu_rows} rows of {a.config} in 8192-row batches, {secs:.1f} s"}


def run_reference_unmodified(a):
    """--impl reference, preferred form: the UNMODIFIED reference (baseline/_ref, staged by baseline/vendor_reference.py) on the
    host cores -- models.boosted_flow.BoostedFlow + the driver lines density_experiment.py:561-571 / :627-641 replayed by
    baseline/ref_harness.density_step -- all host threads, same configuration and batch as our arm."""
    import torch
    rh = _ref_harness()
    ref = rh.load()
    cfg = CONFIGS[a.config]
    torch.set_num_threads(os.cpu_count())
    threads = torch.get_num_threads()
    g = torch.Generator().manual_seed(1234)
    x_init = torch.randn((4096, cfg["D"]), generator=g)
    model, args = rh.build_model(ref, cfg, "cpu", x_init)
    rows = a.batch
    x = torch.randn((rows, cfg["D"]), generator=g)
    # bounded sample: one probe step decides how many rows a step may take so that W + K steps end within ~3 minutes
    t = time.perf_counter()
    rh.density_step(ref, model, x[:8192], args, toy=cfg["toy"])
    rate = min(rows, 8192) / (time.perf_counter() - t)
    budget_rows = rate * 180.0 / (a.steps + a.warmup)
    while rows > 1024 and rows > budget_rows:
        rows //= 2
    xb = x[:rows].contiguous()
    for _ in range(a.warmup):
        rh.density_step(ref, model, xb, args, toy=cfg["toy"])
    t0 = time.perf_counter()
    for _ in range(a.steps):
        G, w = rh.density_step(ref, model, xb, args, toy=cfg["toy"])
    dt = time.perf_counter() - t0
    val = rows * a.steps / dt
    sample = (f"{rows} rows/step of {a.config}: unmodified reference BoostedFlow (baseline/_ref) + density_experiment.py:561-571,"
              f"627-641, torch {torch.__version__} CPU, eval mode, no_grad")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "batch": rows, "same_config": rows == a.batch,
                   "note": "unmodified reference modules from baseline/_ref on the host cores"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def gpu_torch_baseline(a, device, steps=5, warmup=2):
    """The unmodified reference moved to the SAME B200 (`.cuda()`, stock eager PyTorch: ATen kernels + cuBLAS), same
    configuration and batch, timed with CUDA events: the honest library-GPU baseline (SURVEY 2 / 8d)."""
    import torch
    rh = _ref_harness()
    if not rh.available():
        return {"value": None, "unavailable": "baseline/_ref is not staged (run baseline/vendor_reference.py where /root/reference exists)"}
    ref = rh.load()
    cfg = CONFIGS[a.config]
    g = torch.Generator(device=device).manual_seed(1234)
    x = torch.randn((a.batch, cfg["D"]), device=device, generator=g)
    model, args = rh.build_model(ref, cfg, device, x[:4096])
    for _ in range(warmup):
        rh.density_step(ref, model, x, args, toy=cfg["toy"])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        rh.density_step(ref, model, x, args, toy=cfg["toy"])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del model
    torch.cuda.empty_cache()
    return {"value": a.batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "dtype": "f32 (TF32 off: torch default)",
            "what": f"unmodified reference BoostedFlow.cuda() + density_experiment.py:561-571,627-641, eager torch {torch.__version__}, batch {a.batch}"}


def run_reference(a):
    """--impl reference: the reference's own CPU implementation of the path on all host threads.  With baseline/_ref staged this
    is the UNMODIFIED reference (run_reference_unmodified); otherwise the oracle's torch-CPU port stands in (kind = "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not a.port and _ref_harness().available():
        return run_reference_unmodified(a)
    cfg = CONFIGS[a.config]
    rows_per_step = min(a.batch, 8192)
    import numpy as np
    from oracle import gbnf_oracle as orc
    try:
        from threadpoolctl import threadpool_info
        threads = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        threads = os.cpu_count()
    md = orc.make_synthetic_model(cfg["kind"], cfg["D"], cfg["C"], cfg["K"], cfg["h"], seed=1, batch_norm=cfg["bn"],
                                  rho_init=cfg["rho"], toy_base=cfg["toy"], init_rows=2048)
    import torch
    torch.set_num_threads(os.cpu_count())
    threads = torch.get_num_threads()
    tm = orc.to_torch_model(md)
    x = torch.from_numpy(np.random.default_rng(1234).standard_normal((rows_per_step * 4, cfg["D"])).astype(np.float32))

    def step(i):
        xb = x[(i % 4) * rows_per_step:(i % 4 + 1) * rows_per_step]
        with torch.no_grad():
            return orc.torch_density_step(tm, xb)
    for i in range(a.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(a.steps):
        step(i)
    dt = time.perf_counter() - t0
    val = rows_per_step * a.steps / dt
    sample = f"{rows_per_step} rows/step of {a.config} (same model shape, same functions: C log q + mixture + weights)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a), "batch": rows_per_step, "note": "CPU port of the reference algorithm executed "
                   "with the reference's own backend (PyTorch CPU ops, all host threads); the Python reference tree itself "
                   "does not travel to the GPU box"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def workload_name(a):
    c = CONFIGS[a.config]
    return (f"{a.config}: boosted {c['kind']} C={c['C']} K={c['K']} h={c['h']} D={c['D']}, fused log q_c + logsumexp "
            f"mixture + boosting weights, eval batch {a.batch}")


def run_ours(a):
    import torch
    import torch.distributed as dist
    import gbnf_b200
    from gbnf_b200 import dist as gd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep stdout to the one JSON line unless the caller asks for more
        dist.init_process_group("nccl", device_id=device)
    cfg = CONFIGS[a.config]
    C, D = cfg["C"], cfg["D"]

    # ---- model: random-init weights of the named architecture (product constructors, seed 1) -------------------
    torch.manual_seed(1)
    model = gbnf_b200.BoostedFlow(make_args(cfg, device), gemm_mode=a.mode).to(device)
    comp_par = (a.parallel == "component" and world > 1)
    if comp_par and C % world != 0:
        raise SystemExit(f"--parallel component needs C % world == 0 (C = {C}, world = {world})")
    # batch-parallel: every rank owns different rows; component-parallel: every rank sees the SAME rows (SURVEY 8e)
    gen = torch.Generator(device=device).manual_seed(1234 + (0 if comp_par else rank))
    x_all = torch.randn((a.rows, D), device=device, generator=gen)
    model.train()
    with torch.no_grad():   # ActNorm data-dependent init from the first 4096 rows (density_experiment.py:346-356)
        for c in range(C):
            model(x=x_all[:4096], components=c)
    model.eval()
    for p in model.parameters():
        p.requires_grad_(False)
    model.component, model.all_trained = C - 1, False
    model.pack_all()
    peer = world > 1 and not a.nccl
    ops = gd.KernelOps(model, peer=peer)
    if peer:    # library-owned peer-memory exchange over NVLink (gbnf_comm_*): no NCCL call inside a step
        gd.init_peer_exchange(model, a.batch)
    nb = a.rows // a.batch
    batches = [x_all[i * a.batch:(i + 1) * a.batch] for i in range(nb)]

    def step(xb, ev=None):
        if ev: ev[0].record()
        if comp_par:    # rank g: log q of components [g C/G, (g+1) C/G) -> all-gather [B, C/G] -> local mixture kernel
            G = gd.mixture_component_parallel(ops, xb, C)
        else:
            G = model.mixture_log_density(xb, C)
        if ev: ev[1].record()
        if world > 1 and not comp_par:
            w = gd.boosting_weights_batch_parallel(ops, G, "density")
        else:           # component-parallel: every rank holds the whole batch's G_ll, weights are computed redundantly
            w = model.boosting_weights(G)
        if ev: ev[2].record()
        return G, w

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- N > 1: the sharded result must equal the single-GPU kernel path BEFORE anything is timed --------------------------
    parity = None
    if world > 1:
        xb = batches[0]
        if comp_par:     # every rank holds the same rows: component-parallel mixture vs the fused single-GPU launch
            G_cp = gd.mixture_component_parallel(ops, xb[:8192].contiguous(), C)
            G_1 = model.mixture_log_density(xb[:8192].contiguous(), C)
            err = float(((G_cp - G_1).abs() / G_1.abs().clamp_min(1e-30)).max())
            ok = err < 2e-6
            parity = {"what": "component-parallel G_ll (all-gather + mixture kernel) vs the fused single-GPU launch, 8192 rows",
                      "max_rel_err": err, "tol": 2e-6}
        else:            # global-softmax weights of the row shards vs the single-GPU weight kernels on the gathered G_ll
            G_loc = model.mixture_log_density(xb, C)
            w_loc = gd.boosting_weights_batch_parallel(ops, G_loc, "density")
            G_all = torch.empty(world * a.batch, device=device)
            dist.all_gather_into_tensor(G_all, G_loc)
            w_one = model.boosting_weights(G_all)[rank * a.batch:(rank + 1) * a.batch]
            err = float(((w_loc - w_one).abs() / w_one.abs().clamp_min(1e-30)).max())
            ok = err < 5e-6
            parity = {"what": f"batch-parallel boosting weights ({world} shards x {a.batch} rows, global softmax) vs the "
                              "single-GPU weight kernels on the all-gathered G_ll", "max_rel_err": err, "tol": 5e-6}
        flag = torch.tensor([0 if ok else 1], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        errt = torch.tensor([err], device=device)
        dist.all_reduce(errt, op=dist.ReduceOp.MAX)
        parity["max_rel_err"] = errt.item()
        parity["passed"] = flag.item() == 0
        if not parity["passed"]:
            raise SystemExit(f"multi-GPU parity check FAILED: {parity}")

    # ---- `value`: inputs resident in HBM ----------------------------------------------------------------------
    sampler = ClockSampler(local)
    sampler.start()
    for i in range(a.warmup):
        step(batches[i % nb])
    sync()
    launches0 = model.info()["launches"]
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.steps)]
    t_wall0 = time.time()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(a.steps):
        last = step(batches[(a.warmup + i) % nb], evs[i])
    end.record()
    sync()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = model.info()["launches"] - launches0
    ms_total = torch.tensor([start.elapsed_time(end)], device=device)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_total = ms_total.item()
    k_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / a.steps          # fused coupling+mixture kernel
    w_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / a.steps          # boosting-weight kernels
    job_rows = a.batch if comp_par else world * a.batch     # rows the whole job finishes per step
    value = job_rows * a.steps / (ms_total * 1e-3)

    # ---- `e2e`: host buffers in, host result out, copies inside the timed region -------------------------------
    n_host = min(nb, 4)
    host_x = torch.empty((n_host, a.batch, D), dtype=torch.float32).pin_memory()
    for i in range(n_host):
        host_x[i].copy_(batches[i])
    host_G = torch.empty(a.batch, dtype=torch.float32).pin_memory()
    host_w = torch.empty(a.batch, dtype=torch.float32).pin_memory()
    dev_x = [torch.empty((a.batch, D), device=device) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def e2e_loop(n):
        main = torch.cuda.current_stream(device)
        with torch.cuda.stream(copy_stream):
            dev_x[0].copy_(host_x[0], non_blocking=True); ready[0].record(copy_stream)
        for i in range(n):
            cur, nxt = i & 1, (i + 1) & 1
            if i + 1 < n:   # prefetch the next batch on the copy stream while this one computes
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(consumed[nxt])
                    dev_x[nxt].copy_(host_x[(i + 1) % n_host], non_blocking=True); ready[nxt].record(copy_stream)
            main.wait_event(ready[cur])
            G, w = step(dev_x[cur])
            consumed[cur].record(main)
            host_G.copy_(G, non_blocking=True); host_w.copy_(w, non_blocking=True)
        torch.cuda.synchronize()
        return float(host_G[0]) + float(host_w[0])     # the host really reads the result

    e2e_loop(max(3, a.warmup))
    sync()
    t0 = time.perf_counter()
    s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s2.record()
    e2e_loop(a.steps)
    e2.record()
    sync()
    e2e_ms = torch.tensor([max(s2.elapsed_time(e2), 0.0)], device=device)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = job_rows * a.steps / (e2e_ms.item() * 1e-3)

    if peer:
        gd.shutdown_peer_exchange(model)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"mixture_log_density": last[0], "boosting_weights": last[1]})
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel --------------------------------------------------------------------
    pk = peaks()
    fl = flops_per_sample(cfg) * a.batch / (world if comp_par else 1)    # per GPU (component-parallel: C / world components)
    long_run = ms_total > 1000.0
    peak = pk["bf16_sustained"] if long_run else pk["bf16_burst"]
    achieved = fl / (k_ms * 1e-3) / 1e12
    # DRAM bytes per launch of the dominant kernel cannot be read from inside the process (no CUPTI here): they come from the
    # committed `ncu --set full` capture of this exact command (profiles/traffic.json names the capture per configuration)
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic = tj.get(f"{a.config}:{a.mode}:{a.batch}")
        src = tj.get("_source")
        traffic_src = src.get(f"{a.config}:{a.mode}:{a.batch}") if isinstance(src, dict) else src
    inf = model.info()
    kname = ("coupling_fp32_kernel" if a.mode == "fp32" else "coupling_tc5_kernel (interleaved s / t networks, tcgen05)" if inf.get("two_chain") == 2 else
             "coupling_tc4_kernel (two-chain, tcgen05)" if inf.get("two_chain") == 1 else
             "coupling_tc3_kernel (CTA pair, tcgen05)" if inf["pipelined"] == 2 else "coupling_tc2_kernel (pipelined, tcgen05)" if inf["pipelined"] == 1
             else "coupling_tc_kernel (serial, tcgen05)")
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "strong" if comp_par else "weak",
        "vs_baseline": None,
        "dtype": "f32" if a.mode == "fp32" else "f16 operands / f32 accumulate", "data": "synthetic",
        "config": {"workload": workload_name(a), "batch": a.batch, "rows_resident_per_gpu": a.rows, "gemm_mode": a.mode,
                   "l2": f"resident rows {a.rows * D * 4 / 1e6:.0f} MB per GPU > 126 MB L2; batches rotate through them",
                   "parallelism": (f"component-parallel x{world} ({C // world} of {C} components per GPU, every GPU sees all "
                                   f"{a.batch} rows of a step; log q [B, C/G] " + ("stored by the coupling epilogue into every rank's gather buffer over NVLink peer memory" if peer else "all-gathered with NCCL") + ")" if comp_par else
                                   f"batch-parallel x{world} (weak: {a.batch} rows per GPU per step" + ("" if world == 1 else "; global softmax via " + ("the library's peer-memory exchange" if peer else "three NCCL scalar all-reduces")) + ")")},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": "coupling (C/G components) + all-gather + mixture" if comp_par else "fused coupling+mixture", "kernel_name": kname,
                     "kernel_ms": k_ms, "weights_ms": w_ms,
                     "flops_per_sample": flops_per_sample(cfg),
                     "peak_kind": ("sustained" if long_run else "burst") + " bf16, " + pk["source"]},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": a.batch * D * 4, "d2h_bytes_per_step": a.batch * 8},
        "gpu_launches": launches,
    }
    if parity is not None:
        out["parity_check"] = parity
    if world == 1 and not a.no_cpu:
        out["cpu_baseline"] = cpu_baseline_leg(a)
        out["gpu_torch_baseline"] = gpu_torch_baseline(a, device)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", default="cfg3_miniboone", choices=list(CONFIGS))
    p.add_argument("--mode", default=os.environ.get("GBNF_BENCH_MODE", "f16fast"), choices=["f16", "f16fast", "fp32"])
    p.add_argument("--batch", type=int, default=65536)
    p.add_argument("--parallel", default="batch", choices=["batch", "component"],
                   help="N > 1: shard rows (default, weak scaling) or components (strong scaling, cfg4's layout)")
    p.add_argument("--rows", type=int, default=1 << 20)
    p.add_argument("--cpu-rows", type=int, default=524288)
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--nccl", action="store_true", help="N > 1: torch.distributed collectives between the staged kernels instead of "
                   "the library's peer-memory exchange (A/B measurements)")
    p.add_argument("--port", action="store_true", help="--impl reference: time the oracle's torch-CPU port even when baseline/_ref exists")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the G_ll and boosting weights of the last timed step to DIR/<name>.npy")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs needs --impl ours")
    a.warmup = max(a.warmup, 3)
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
