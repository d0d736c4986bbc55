#!/usr/bin/env python
"""bench.py — DPSVI.update examples/sec on the BASELINE.json workloads.

Default workload (config.workload = "c2", BASELINE.json configs[1]): synthetic logistic regression,
N = 10M records x d = 1024 float32 (41 GB resident in HBM, >> L2), Poisson sampling q = 0.01
(max_batch_size = the 0.99 Poisson quantile = 100736), hand-written mean-field guide, Adam(1e-3),
C = 1, dp_scale = 1.  Other workloads: c1 (N=10k d=8), c3 (Gaussian N=50M d=256, subsample
B=500k), c4 (GMM K=64 d=128 N=20M, Poisson), c5 (VAE 784-400-20, B=4096: tcgen05 clipped-sum GEMMs).

A "step" = `get_batch(i, state)` (sampler kernels) followed by `DPSVI.update(state, *batch,
mask=mask)` (fused gather / per-example gradient / clip / sum kernel(s) + (NCCL all-reduce at N > 1)
+ reduce / ChaCha noise / rescale / Adam kernel).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2] [--dump-outputs DIR]

`--dump-outputs DIR` writes, after the timed steps, what the headline path handed its caller after its last step
(parameters, optimizer moments, state key, that step's loss and example count) as DIR/<name>.npy.  The data set and
every key are derived from fixed seeds, so two builds run with the same arguments can be compared array by array.

N > 1 is launched by torchrun (one rank per GPU, NCCL); the batch is sharded over the ranks
(strong scaling: the global batch is fixed by the config).  `--impl reference` times the CPU
oracle port of the same step on the host cores (the reference itself needs jax/numpyro/
jax-chacha-prng, none of which can be installed here — see DESIGN.md).
"""
import argparse
import gc
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c1": dict(N=10_000, d=8, q=0.02, family="logreg", C=1.0, sampler="poisson"),
    "c2": dict(N=10_000_000, d=1024, q=0.01, family="logreg", C=1.0, sampler="poisson"),
    "c3": dict(N=50_000_000, d=256, q=0.01, family="gauss", C=1.0, sampler="subsample"),
    "c4": dict(N=20_000_000, d=128, q=0.01, family="gmm", C=20.0, sampler="poisson", K=64),
    "c5": dict(N=60_000, d=784, q=4096 / 60_000, family="vae", C=10.0, sampler="subsample", batch=4096,
               hidden=400, z=20),
}
# SURVEY.md 8(d): algorithmic HBM bytes per example of the dominant kernel
ALGO_BYTES_PER_EXAMPLE = {"c1": 4 * (8 + 1), "c2": 4 * (1024 + 1), "c3": 4 * 256, "c4": 4 * 128}
# launches of OUR kernels per step: sampler (Poisson: select + compact; Feistel: 1) + step kernel(s) + finalize;
# matches the ncu launch list profiles/r1_c2_launches_v7.csv (4 per C2 step)
LAUNCHES = {"poisson": 2, "subsample": 1, "logreg": 2, "gauss": 2, "gmm": 2, "vae": 14}   # vae: 2 split + prep x + prep mid + 7 GEMMs + 2 thin-layer MMA + loss (13) + finalize


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def ncu_traffic(workload):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(workload)
    return None


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the benchmark runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def batch_size_of(cfg):
    if cfg["sampler"] == "poisson":
        import scipy.stats
        return int(scipy.stats.poisson(cfg["N"] * cfg["q"]).ppf(.99))
    return cfg.get("batch", int(cfg["N"] * cfg["q"]))


def workload_config(name, cfg):
    b = batch_size_of(cfg)
    sampler = (f"Poisson q={cfg['q']} max_batch_size={b}" if cfg["sampler"] == "poisson"
               else f"subsample without replacement batch={b}")
    model = (f"VAE {cfg['d']}-{cfg['hidden']}-{cfg['z']}" if cfg["family"] == "vae" else
             f"GMM K={cfg['K']} d={cfg['d']}" if cfg["family"] == "gmm" else f"{cfg['family']} d={cfg['d']}")
    data_mb = cfg["N"] * cfg["d"] * 4 / 1e6
    if data_mb > 126:
        l2 = (f"inputs larger than L2: the {data_mb:.0f} MB data set stays in HBM and every step gathers a fresh random "
              "batch of rows from it")
    else:
        l2 = (f"the {data_mb:.2f} MB data set is L2-resident by construction (BASELINE configs[0], the reference's "
              "CPU-runnable case): a latency / parity configuration, not a roofline one; no L2 flush")
    return {"workload": f"{name}: synthetic {model} N={cfg['N']} {sampler}", "l2_policy": l2,
            "optimizer": "Adam(1e-3)", "clipping_threshold": cfg["C"], "dp_scale": 1.0}


# ------------------------------------------------------------------------------------------------
# CPU arm — the cpu_baseline leg and `--impl reference`
# ------------------------------------------------------------------------------------------------
# Rows of the data set the CPU arm keeps in host memory (same d, q, sampler, clip, optimizer as the workload;
# examples/s does not depend on N except through the Poisson selector draw, which is part of the step and scales
# with it: SURVEY.md section 8d).  The batch follows from q: c2 at 1 M rows = Poisson(1e4) batches, max 10 233.
CPU_ROWS = {"c1": 10_000, "c2": 1_000_000, "c3": 1_000_000, "c4": 5_000, "c5": 60_000}
CPU_BATCH = {"c5": 256}        # the autodiff port materialises [B, P] per-example gradients: 4096 x 652 824 x 4 B = 10.7 GB


def cpu_port_setup(name, cfg, threads):
    """-> (step(i, state) -> (state, n_valid), state, description).  A step = get_batch(i) (oracle sampler + masked
    gather, oracle/minibatch.py) + DPSVI.update (oracle/svi.py: Threefry keys and guide noise in numpy,
    torch.func vmap(grad), clip, mean, ChaCha noise, Adam) — the same work as one step of the B200 arm."""
    import torch
    from oracle import chacha, families, minibatch as omb, svi as osvi
    torch.set_num_threads(threads)
    d, q = cfg["d"], cfg["q"]
    N = min(cfg["N"], CPU_ROWS[name])
    rs = np.random.default_rng(123)
    if cfg["family"] == "logreg":
        fam = families.LogisticRegression(d, N)
        data = (rs.standard_normal((N, d), dtype=np.float32), (rs.random(N) < .5).astype(np.int32))
    elif cfg["family"] == "gauss":
        fam = families.GaussianMean(d, N)
        data = ((1 + .1 * rs.standard_normal((N, d), dtype=np.float32)),)
    elif cfg["family"] == "gmm":
        from oracle import gmm as ogmm
        fam = ogmm.GaussianMixture(cfg["K"], d, N)
        data = ((3 * rs.standard_normal((N, d), dtype=np.float32)),)
    else:
        from oracle import vae as ovae
        fam = ovae.VAE(d, cfg["hidden"], cfg["z"], N)
        data = ((rs.random((N, 28, 28), dtype=np.float32) < .3).astype(np.float32),)
    if cfg["sampler"] == "poisson":
        init, get = omb.poisson_batchify_data(data, q, .99)
        sampler = f"Poisson q={q}"
    else:
        B = CPU_BATCH.get(name, max(1, int(round(N * q))))
        init, get = omb.subsample_batchify_data(data, batch_size=B, return_mask=True)
        sampler = f"subsample batch={B}"
    key, k_init, k_fetch = chacha.split(chacha.PRNGKey(0), 3)
    _, bstate = init(k_fetch)
    batch, mask = get(0, bstate)
    s = osvi.DPSVI(fam, None, osvi.Adam(1e-3), None, cfg["C"], 1.0)
    state = s.init(k_init, *batch)

    def step(i, state):
        batch, mask = get(i, bstate)
        state, _ = s.update(state, *batch, mask=mask)
        return state, int(np.sum(mask))

    desc = (f"oracle port (numpy ChaCha / Threefry / sampler + gather, torch.func vmap(grad), clip, noise, Adam) on "
            f"{N} rows x d={d}, {sampler}, padded batch {len(mask)}: each step = get_batch + DPSVI.update")
    return step, state, desc


def cpu_run(name, cfg, steps, warmup, threads):
    step, state, desc = cpu_port_setup(name, cfg, threads)
    for i in range(warmup):
        state, _ = step(i, state)
    n = 0
    t0 = time.perf_counter()
    for i in range(steps):
        state, nv = step(warmup + i, state)
        n += nv
    dt = time.perf_counter() - t0
    return n / dt, dt / steps * 1e3, desc


def run_reference(args, cfg):
    """`--impl reference`: the reference's CPU implementation of the path on the host cores.  The real d3p (jax +
    numpyro + jax-chacha-prng) when importable (baseline/run_reference.py, kind = "reference"), else the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    from baseline import run_reference as rr
    ok, why = rr.available()
    kind = "port"
    if ok and cfg["family"] == "logreg":
        r = rr.time_update(cfg, args.steps, args.warmup, min(cfg["N"], CPU_ROWS[args.workload]))
        value, ms, kind = r["value"], r["ms_per_step"], "reference"
        desc = (f"the reference itself (d3p from {why}, {r['versions']}): jitted get_batch + DPSVI.update on "
                f"{min(cfg['N'], CPU_ROWS[args.workload])} rows x d={cfg['d']}, padded batch {r['max_batch_size']}")
    else:
        value, ms, desc = cpu_run(args.workload, cfg, args.steps, args.warmup, threads)
        desc += f"; the reference's JAX path is unavailable here ({why})"
    line = {
        "impl": "reference", "metric": "DPSVI.update examples/sec", "value": value, "unit": "examples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, cfg),
        "cpu_baseline": {"value": value, "unit": "examples/s", "cores": threads, "kind": kind, "sample": desc},
        "e2e": {"value": value, "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def make_dataset(cfg, device):
    """Synthetic data of the named shape, generated on the device with the build's own ChaCha
    kernels (reproducible without JAX)."""
    import torch
    import d3p_b200.random as rng
    N, d = cfg["N"], cfg["d"]
    kx, kw, ky = rng.split(rng.PRNGKey(123), 3)
    if cfg["family"] == "vae":      # uniform [0,1] "pixels", Bernoulli-binarised (examples/vae.py:156-168)
        X = (rng.uniform(kx, (N, 28, 28)) < rng.uniform(kw, (N, 28, 28))).to(torch.float32)
        return (X,)
    X = rng.normal(kx, (N, d))
    if cfg["family"] == "gmm":      # K-component diagonal mixture: means ~ N(0, 10^2), unit scales
        centers = rng.normal(kw, (cfg["K"], d)) * 10.0
        z = rng.randint(ky, (N,), 0, cfg["K"]).to(torch.int64)
        for lo in range(0, N, 1 << 20):     # in place, chunked: no second copy of the data set
            X[lo:lo + (1 << 20)] += centers[z[lo:lo + (1 << 20)]]
        return (X,)
    if cfg["family"] == "gauss":    # x ~ N(1, 0.1^2)  (simple_gaussian_posterior.py:62-65,105)
        X.mul_(0.1).add_(1.0)
        return (X,)
    w = rng.normal(kw, (d + 1,))    # y ~ Bernoulli(sigmoid(X w* + b*))  (logistic_regression.py:88-104)
    logits = torch.mv(X, w[:d]) + w[d]
    y = (rng.uniform(ky, (N,)) < torch.sigmoid(logits)).to(torch.int32)
    return (X, y)


def make_family(cfg):
    from d3p_b200 import models
    if cfg["family"] == "logreg":
        return models.LogisticRegression(cfg["d"])
    if cfg["family"] == "gauss":
        return models.GaussianMean(cfg["d"])
    if cfg["family"] == "gmm":
        return models.GaussianMixture(cfg["K"], cfg["d"])
    return models.VAE(cfg["d"], cfg["hidden"], cfg["z"])


DUMP_LIMIT_BYTES = 64 << 20


def output_arrays(svi, state, loss, n_examples):
    """Host copies of what a caller of DPSVI.update / run_epoch holds after a step: the constrained parameters, the
    optimizer's moments, the state key (uint32 words, exact in float64), the step's loss and its example count."""
    import re
    import torch

    def host(x):
        a = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
        return a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    out = {"param_" + re.sub(r"[^0-9A-Za-z_]+", "_", k): host(v) for k, v in svi.get_params(state).items()}
    os_ = state.optim_state
    out.update({f"optim_{k}": host(v) for k, v in (("m", os_.m), ("v", os_.v)) if v is not None})
    out["rng_key"] = host(state.rng_key)
    out["loss"] = host(loss).reshape(1)
    out["n_examples"] = host(n_examples).astype(np.float64).reshape(1)
    return out


def write_outputs(path, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


class LibEvents:
    """CUDA events owned by libd3p_b200 (recorded inside the C call around the dominant kernels)."""

    def __init__(self, n):
        from d3p_b200 import _native as _n
        self._n = _n
        self.arr = (C.c_void_p * n)()
        for i in range(n):
            e = C.c_void_p()
            _n.check(_n.lib().d3p_event_create(C.byref(e)))
            self.arr[i] = e.value

    def elapsed(self, i, j):
        ms = C.c_float()
        self._n.check(self._n.lib().d3p_event_elapsed_ms(C.c_void_p(self.arr[i]), C.c_void_p(self.arr[j]), C.byref(ms)))
        return ms.value


def ncu_side_run(workload, elements_per_example):
    """Measures, in THIS bench invocation, the instruction count and issue activity of the dominant step kernel: one
    launch of a child `bench.py --ncu-child` under `ncu --metrics ...` (outside every timed region; a number printed by
    the child under the profiler is never a bench value).  -> dict or None when ncu is not on the box / fails."""
    import shutil
    import subprocess
    ncu = shutil.which("ncu") or ("/usr/local/cuda/bin/ncu" if os.path.exists("/usr/local/cuda/bin/ncu") else None)
    if ncu is None:
        return None
    metrics = "smsp__inst_executed.sum,smsp__issue_active.avg.pct_of_peak_sustained_active,gpu__time_duration.sum"
    # child launch order of the step kernel: 3 warm-up steps, then 2 timed steps: skip 4 = the second timed step
    cmd = [ncu, "--metrics", metrics, "--clock-control", "none", "-k", "regex:meanfield_step", "-s", "4", "-c", "1", "--csv",
           sys.executable, os.path.abspath(__file__), "--workload", workload, "--steps", "2", "--warmup", "3", "--no-e2e",
           "--no-cpu-baseline", "--no-other-workloads", "--ncu-child"]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
    except Exception:
        return None
    vals, child = {}, None
    for ln in r.stdout.splitlines():
        if ln.startswith("{") and "per_step_examples" in ln:
            child = json.loads(ln)
        parts = [p.strip('"') for p in ln.split('","')]
        for m in metrics.split(","):
            if m in parts:
                try:
                    vals[m] = float(parts[-1].replace(",", ""))
                except ValueError:
                    pass
    if child is None or "smsp__inst_executed.sum" not in vals:
        return None
    examples = child["per_step_examples"][1]
    return {"warp_instr_per_launch": vals["smsp__inst_executed.sum"], "examples_in_launch": examples,
            "warp_instr_per_element": vals["smsp__inst_executed.sum"] * 32.0 / (examples * elements_per_example),
            "issue_active_pct": vals.get("smsp__issue_active.avg.pct_of_peak_sustained_active"),
            "kernel_us_under_ncu": vals.get("gpu__time_duration.sum", 0.0) / 1e3,
            "how": "ncu --metrics smsp__inst_executed.sum,smsp__issue_active... -k regex:meanfield_step -s 4 -c 1 on a "
                   "child run of this script (same workload, 5 steps), launched by this bench run"}


def quick_workload(name, steps, warmup, device):
    """A short device-resident run of another BASELINE workload through DPSVI.run_epoch (same kernels, same step
    definition as the headline), so that the driver's default run also records C3 and C5.  -> dict for `workloads`."""
    import torch
    import d3p_b200.random as rng
    from d3p_b200 import minibatch as mb, models, optimizers, svi as dsvi
    cfg = dict(WORKLOADS[name])
    dataset = make_dataset(cfg, device)
    fam = make_family(cfg)
    svi = dsvi.DPSVI(fam.model, fam.guide, optimizers.Adam(1e-3), models.Trace_ELBO(), cfg["C"], 1.0, num_obs_total=cfg["N"])
    svi.donate_state = True
    if cfg["sampler"] == "poisson":
        init, get_batch = mb.poisson_batchify_data(dataset, cfg["q"], .99)
    else:
        init, get_batch = mb.subsample_batchify_data(dataset, batch_size=batch_size_of(cfg), return_mask=True)
    key, k_init, k_fetch = rng.split(rng.PRNGKey(0), 3)
    _, bstate = init(k_fetch)
    batch, mask = get_batch(0, bstate)
    state = svi.init(k_init, *batch)
    state, _ = svi.run_epoch(state, get_batch, bstate, max(warmup, 3), first_step=0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    state, stats = svi.run_epoch(state, get_batch, bstate, steps, first_step=16)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if not bool(torch.isfinite(stats[:, 0]).all()):
        raise RuntimeError(f"workload {name} produced a non-finite loss")
    out = {"value": float(stats[:, 1].sum().item()) / (ms * 1e-3), "unit": "examples/s", "ms_per_step": ms / steps,
           "steps": steps, "config": workload_config(name, cfg), "driver": "DPSVI.run_epoch"}
    if name in ALGO_BYTES_PER_EXAMPLE:
        out["algorithmic_gbs_whole_step"] = ALGO_BYTES_PER_EXAMPLE[name] * out["value"] / 1e9
    del dataset, state, svi
    torch.cuda.empty_cache()
    return out


def run_b200(args, cfg):
    import torch
    import torch.distributed as dist
    import d3p_b200.random as rng
    from d3p_b200 import minibatch as mb, models, optimizers, parallel, svi as dsvi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    N, q = cfg["N"], cfg["q"]
    is_vae = cfg["family"] == "vae"
    # N > 1, outside the timed region: the sharded path (p2p update + run_epoch, logreg and VAE) must reproduce the
    # unsharded one on small problems before anything is measured (d3p_b200/selfcheck.py); a mismatch is fatal
    parity = None
    if world > 1:
        from d3p_b200 import selfcheck
        parity = selfcheck.sharded_parity_check(device)
        if not parity["ok"]:
            raise RuntimeError(f"sharded-vs-unsharded parity check failed: {json.dumps(parity)}")
    dataset = make_dataset(cfg, device)
    fam = make_family(cfg)
    svi = dsvi.DPSVI(fam.model, fam.guide, optimizers.Adam(1e-3), models.Trace_ELBO(), cfg["C"], 1.0,
                     num_obs_total=N)
    svi.donate_state = True
    if world > 1:
        parallel.shard_dpsvi(svi, rank, world, backend=args.collective)
        args.collective = "p2p" if svi.peer_window is not None else "nccl"     # what "auto" resolved to
    if cfg["sampler"] == "poisson":
        init, get_batch = mb.poisson_batchify_data(dataset, q, .99)
    else:
        init, get_batch = mb.subsample_batchify_data(dataset, batch_size=batch_size_of(cfg), return_mask=True)
    key = rng.PRNGKey(0)
    key, k_init, k_fetch = rng.split(key, 3)
    _, bstate = init(k_fetch)
    batch, mask = get_batch(0, bstate)
    max_b = len(batch[0])
    state = svi.init(k_init, *batch)

    kernel_events = []

    def hook(tag):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        kernel_events.append(ev)

    def one_step(i, state):
        batch, mask = get_batch(i, bstate)
        state, loss = svi.update(state, *batch, mask=mask)
        nv = batch[0].num_valid
        return state, loss, (nv if nv is not None else max_b)

    def sync_all():
        # garbage of the set-up phase (parity check, data generation) is collected here, outside the timed regions: a
        # collection that runs finalisers with CUDA calls in the middle of a timed loop is a multi-millisecond host stall
        gc.collect()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        # fail loudly: a peer-memory exchange that timed out poisons the step (NaN) and is counted; no bench value
        # may come out of such a run
        if svi.peer_window is not None:
            svi.peer_window.check(synchronize=False)

    # the headline is the C-side epoch driver where there is one for the family and collective (row f2 below), else the
    # interpreter-driven loop
    headline_epoch = cfg["family"] in ("logreg", "gauss", "vae") and (world == 1 or args.collective == "p2p")
    outputs = None
    sync_all()        # ranks finish generating 41 GB of data at different times: align them before the first exchange
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(args.warmup):
        state, loss, _ = one_step(i, state)
    sync_all()
    svi.event_hook = hook
    lib_events = None
    gemm_ms = []
    if is_vae:
        lib_events = LibEvents(2)
        fam.profile_events = lib_events.arr
    counts = []
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin.record()
    for i in range(args.steps):
        state, loss, nv = one_step(args.warmup + i, state)
        counts.append(nv)
    t_end.record()
    sync_all()
    if args.dump_outputs and not headline_epoch:
        outputs = output_arrays(svi, state, loss, counts[-1])
    svi.event_hook = None
    if args.ncu_child:      # profiled child of ncu_side_run: report which launch held how many examples, nothing else
        print(json.dumps({"per_step_examples": [int(c) if isinstance(c, int) else int(c.reshape(()).item()) for c in counts]}))
        return
    elapsed_ms = t_begin.elapsed_time(t_end)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    n_examples = int(sum(int(c) if isinstance(c, int) else int(c.reshape(()).item()) for c in counts))
    value = n_examples / (elapsed_ms * 1e-3)
    kern_ms = [kernel_events[2 * i].elapsed_time(kernel_events[2 * i + 1]) for i in range(len(kernel_events) // 2)]
    kern_ms_avg = float(np.mean(kern_ms))
    if not np.isfinite(float(loss)):
        raise RuntimeError("bench produced a non-finite loss")
    if is_vae:
        # time the clipped-sum GEMMs live: a few more steps, reading the library's events after each
        for i in range(min(args.steps, 20)):
            state, loss, _ = one_step(args.warmup + args.steps + i, state)
            gemm_ms.append(lib_events.elapsed(0, 1))
        fam.profile_events = None

    # ---- the same K steps through the C-side epoch driver (row f2): no interpreter between launches ----
    epoch_line = None
    if headline_epoch:
        base = args.warmup + args.steps + 32
        state, _ = svi.run_epoch(state, get_batch, bstate, max(args.warmup, 3), first_step=base)
        sync_all()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        state, ep_stats = svi.run_epoch(state, get_batch, bstate, args.steps, first_step=base + 8)
        p1.record()
        sync_all()
        if args.dump_outputs:
            outputs = output_arrays(svi, state, ep_stats[-1, 0], ep_stats[-1, 1])
        ep_ms = p0.elapsed_time(p1)
        if world > 1:
            t = torch.tensor([ep_ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ep_ms = float(t.item())
        epoch_line = {"value": float(ep_stats[:, 1].sum().item()) / (ep_ms * 1e-3), "unit": "examples/s",
                      "ms_per_step": ep_ms / args.steps,
                      "note": "DPSVI.run_epoch: the fori_loop(get_batch -> update) of the examples driven by "
                              + ("d3p_dpsvi_run_epoch_vae" if is_vae else "d3p_dpsvi_run_epoch_meanfield")
                              + " (same kernels, host work in C)"}

    clocks = sampler.stop()

    # ---- end to end through the public API with HOST buffers (rank-local shard at N > 1) -----------
    e2e = None
    if args.e2e:
        # N > 1 (mean-field families): every rank keeps and uploads only the rows of its own position
        # range (minibatch.LocalRows), so the H2D traffic is split over the GPUs' PCIe links
        local = world > 1 and cfg["family"] in ("logreg", "gauss")
        pb, pe = parallel.position_range(max_b, rank, world) if local else (0, max_b)
        dev_batch = [b.tensor()[pb:pe] for b in batch]
        host = [torch.empty(t_.shape, dtype=t_.dtype).pin_memory() for t_ in dev_batch]
        for h, src in zip(host, dev_batch):
            h.copy_(src)
        host_mask = torch.empty(mask[pb:pe].shape, dtype=torch.bool).pin_memory()
        host_mask.copy_(mask[pb:pe])
        n_valid_host = int(mask.sum().item())

        def wrap(t_):
            return mb.LocalRows(t_, pb, max_b) if local else t_
        dev_bufs = [[torch.empty_like(h, device=device) for h in host] + [torch.empty_like(host_mask, device=device)]
                    for _ in range(2)]
        loss_host = torch.empty(args.steps + args.warmup, dtype=torch.float32).pin_memory()
        copy_stream = torch.cuda.Stream()
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        h2d_bytes = sum(h.numel() * h.element_size() for h in host) + host_mask.numel()

        def e2e_loop(n_steps, state, base):
            main = torch.cuda.current_stream()
            for i in range(n_steps):
                slot = i & 1
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(consumed[slot])
                    for dst, src in zip(dev_bufs[slot], host + [host_mask]):
                        dst.copy_(src, non_blocking=True)
                    ready[slot].record(copy_stream)
                main.wait_event(ready[slot])
                state, loss = svi.update(state, *[wrap(t_) for t_ in dev_bufs[slot][:-1]], mask=wrap(dev_bufs[slot][-1]))
                consumed[slot].record(main)
                loss_host[base + i:base + i + 1].copy_(loss.reshape(1), non_blocking=True)
            return state

        for ev in consumed:
            ev.record()
        state = e2e_loop(args.warmup, state, 0)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        state = e2e_loop(args.steps, state, args.warmup)
        e1.record()
        sync_all()
        e_ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([e_ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e_ms = float(t.item())
        if world > 1:
            t = torch.tensor([float(h2d_bytes)], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            h2d_bytes = int(t.item())
        e2e = {"value": n_valid_host * args.steps / (e_ms * 1e-3), "unit": "examples/s",
               "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 4 * world,
               "note": "DPSVI.update(state, *batch, mask) with the batch in pinned HOST memory: "
                       "H2D copy of the padded batch + update + loss read-back every step (double-buffered)"
                       + ("; each rank uploads the rows of its own position range, bytes are summed over ranks"
                          if local else "")}

    ncu_side_run_result = None
    if (rank == 0 and world == 1 and args.ncu_side_run and not args.ncu_child and cfg["family"] in ("logreg", "gauss")
            and cfg["d"] >= 256):
        ncu_side_run_result = ncu_side_run(args.workload, cfg["d"] + (1 if cfg["family"] == "logreg" else 0))
    if rank == 0:
        peaks, peak_kind = measured_peaks()
        step_ms = elapsed_ms / args.steps
        per_rank_examples = (n_examples / args.steps) / world
        if is_vae:
            D, H, Zd = cfg["d"], cfg["hidden"], cfg["z"]
            # SURVEY 8(d): the clipped-sum GEMMs dW1, dW5 (+ the thin dW2|dW3, dW4), which run as one concurrent group
            flops = 2.0 * (2.0 * D * H + 3.0 * H * Zd) * per_rank_examples
            g_ms = float(np.mean(gemm_ms))
            achieved = flops / (g_ms * 1e-3) / 1e12
            # TF32 dense = half the bf16 rate; the group is timed inside the running step => the sustained figure
            peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]) / 2.0
            roofline = {"bound": "tensor", "kernel": "tc_gemm_kernel<MN,MN,*,EpiGrad> x4 (dW1, dW5, dW2|dW3, dW4 clipped sums, "
                                                     "concurrent on forked streams: one wave of CTAs)",
                        "achieved": achieved, "peak": peak,
                        "peak_kind": peak_kind + " sustained bf16 GEMM / 2 (no measured TF32 figure)", "unit": "TFLOP/s",
                        "frac": achieved / peak, "traffic": ncu_traffic(args.workload), "kernel_ms": g_ms,
                        "kernel_share_of_step": g_ms / step_ms,
                        "executed_tflops": 3.0 * achieved,
                        "note": "algorithmic FLOPs = 2*(2*784*400 + 3*400*20) per example; the kernels execute 3x that "
                                "(3xTF32 split for fp32 parity), see executed_tflops; kernel_ms = CUDA events around "
                                "the concurrent group",
                        "step_kernels_ms": kern_ms_avg}
        else:
            algo_bytes = ALGO_BYTES_PER_EXAMPLE[args.workload] * per_rank_examples
            achieved = algo_bytes / (kern_ms_avg * 1e-3) / 1e9
            kname = ("gmm_step_kernel" if cfg["family"] == "gmm" else
                     "meanfield_step_vec_kernel" if cfg["d"] >= 256 else "meanfield_step_kernel")
            roofline = {"bound": "hbm", "kernel": kname,
                        "achieved": achieved, "peak": peaks["hbm_gbs"], "peak_kind": peak_kind, "unit": "GB/s",
                        "frac": achieved / peaks["hbm_gbs"], "traffic": ncu_traffic(args.workload),
                        "kernel_ms": kern_ms_avg, "kernel_share_of_step": kern_ms_avg / step_ms,
                        "note": ("ALU-bound by the reference's semantics: ~16 k guide variates (8 k gamma rejection "
                                 "samples at ~10 Threefry calls each) per 512-byte row, DESIGN.md section 6"
                                 if cfg["family"] == "gmm" else
                                 "issue-bound, not HBM-bound: one Threefry-2x32-20 normal per data float "
                                 "(~84 warp-instructions per element, measured by this run under issue_slots when "
                                 "the ncu side run is on; DESIGN.md section 5)")}
            if kname == "meanfield_step_vec_kernel" and world == 1 and args.ncu_side_run and clocks.get("sm_mhz"):
                # the bound that does apply: issue slots.  The instruction count per element is MEASURED by this run
                # (ncu side run of a child process, see ncu_side_run); the slots offered are SMs x 4 schedulers x
                # measured SM clock x the kernel time measured above with CUDA events (not the profiler's).
                epe = cfg["d"] + (1 if cfg["family"] == "logreg" else 0)
                side = ncu_side_run_result
                if side is not None:
                    elems = per_rank_examples * epe
                    slots = 148 * 4 * clocks["sm_mhz"] * 1e6 * kern_ms_avg * 1e-3
                    roofline["issue_slots"] = dict(side, frac_of_issue_slots=(side["warp_instr_per_element"] * elems / 32) / slots,
                                                   min_instr_per_element_at_70pct_hbm=31)
                else:
                    roofline["issue_slots"] = {"unavailable": "ncu side run failed or ncu is not on this box"}
        line = {
            "metric": "DPSVI.update examples/sec", "value": value, "unit": "examples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args.workload, cfg),
            "clocks": clocks,
            "gpu_launches": (LAUNCHES[cfg["sampler"]] + LAUNCHES[cfg["family"]] +
                             (1 if world > 1 and args.collective == "nccl" else 0)) * args.steps,
            "roofline": roofline,
            "examples_per_step": n_examples / args.steps, "max_batch_size": max_b,
        }
        if e2e is not None:
            line["e2e"] = e2e
        line["driver"] = "python loop: get_batch(i, state) + DPSVI.update per step"
        if world > 1:
            line["parity_check"] = parity
            line["peer_timeouts"] = 0 if svi.peer_window is None else svi.peer_window.timeouts()
            line["collective"] = ("clipped sums exchanged inside the finalize kernel over NVLink peer memory"
                                            if args.collective == "p2p" else "reduce kernel + ncclAllReduce(P + 2 floats)")
        if epoch_line is not None:
            # headline = the same K steps through DPSVI.run_epoch (the examples' fori_loop, driven from C);
            # the interpreter-driven loop above stays as `stepwise` and provides the per-kernel event timings
            line["stepwise"] = {"value": value, "ms_per_step": step_ms}
            line["value"], line["ms_per_step"] = epoch_line["value"], epoch_line["ms_per_step"]
            line["driver"] = ("DPSVI.run_epoch: get_batch + update for all K steps inside "
                                        + ("d3p_dpsvi_run_epoch_vae" if is_vae else "d3p_dpsvi_run_epoch_meanfield"))
            line["roofline"]["kernel_share_of_step"] = line["roofline"]["kernel_ms"] / epoch_line["ms_per_step"]
        if world == 1 and args.workload == "c2" and args.other_workloads:
            # the default run also records the other single-GPU roofline workloads (short runs, outside the headline)
            del dataset, batch
            svi._ws = svi._epoch_ws = None
            torch.cuda.empty_cache()
            line["workloads"] = {w: quick_workload(w, min(args.steps, 50), args.warmup, device) for w in ("c3", "c5")}
        if world == 1 and args.cpu_baseline:
            threads = os.cpu_count() or 1
            v, ms, desc = cpu_run(args.workload, cfg, 4, 1, threads)
            line["cpu_baseline"] = {"value": v, "unit": "examples/s", "cores": threads, "kind": "port",
                                    "sample": "4 steps: " + desc}
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--collective", default="auto", choices=["auto", "p2p", "nccl"],
                    help="N > 1: exchange the clipped sums inside the finalize kernel over NVLink peer memory (p2p) "
                         "or with a reduce kernel + ncclAllReduce (nccl)")
    ap.add_argument("--rows", type=int, default=None, help="override N (development only)")
    ap.add_argument("--no-e2e", dest="e2e", action="store_false")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-ncu-side-run", dest="ncu_side_run", action="store_false",
                    help="skip the ncu child run that measures instructions per element of the step kernel")
    ap.add_argument("--ncu-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-other-workloads", dest="other_workloads", action="store_false",
                    help="default (c2, N = 1) run only: skip the short c3 / c5 runs reported under `workloads`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the headline path computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the B200 path computed: use it with --impl b200")
    args.warmup = max(args.warmup, 3)
    cfg = dict(WORKLOADS[args.workload])
    if args.rows:
        cfg["N"] = args.rows
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_b200(args, cfg)


if __name__ == "__main__":
    main()
