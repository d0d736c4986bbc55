#!/usr/bin/env python
"""Where the time of one DP-SVI step of a user model (models.AutoDiagonalNormalModel) goes, next to the fused family.

Workloads: logistic regression at d = 1024 written as a user model (the same model as the fused
``LogisticRegression(1024, guide="auto")``), and a Poisson regression with float counts at the same size, which has no
fused kernel.  Batches are C2-sized Poisson batches (q * N = 100 000 expected examples).

Reports, per workload:
  * CUDA-event times of the phases of ``update``: the guide draw (d3p_autodiag_draw_f32), the torch potential and
    its autograd, the step entry point (d3p_dpsvi_step_autodiag) and the finalize (d3p_perturb_finalize_p2p_f32);
  * per-kernel device times from torch.profiler, in a separate run;
  * examples/s of ``update`` over fresh batches, and for the logistic regression the same for the fused family.
The device name and power limit are read in the same run.

    python scripts/autodiag_step_times.py --out autodiag_step_times.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import d3p_b200.random as rng                                                          # noqa: E402
from d3p_b200 import _native as _n, minibatch as mb, models, optimizers, svi as dsvi  # noqa: E402


def logreg_ll(lat, X, y):
    z = (X * lat["w"]).sum(-1) + lat["intercept"]
    return -(torch.clamp(z, min=0) + torch.log1p(torch.exp(-torch.abs(z))) - z * y.to(z.dtype))


def poisson_ll(lat, X, y):
    eta = (X * lat["w"]).sum(-1) + lat["b"]
    return y * eta - torch.exp(eta) - torch.lgamma(y + 1)


def device_info():
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return out


def timed(fn, reps):
    """Mean ms of fn() over reps calls, CUDA events around the whole loop (after one warm-up call)."""
    fn()
    b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    b.record()
    for _ in range(reps):
        fn()
    e.record()
    e.synchronize()
    return b.elapsed_time(e) / reps


def phases(fam, s, st, batch, mask, reps):
    """Times of the phases of one update on a fixed batch."""
    B = int(batch[0].shape[0])
    N = s._num_obs_total()
    desc = fam.desc(N)
    params = _n.ptr(st.optim_state.flat)
    key = np.ascontiguousarray(rng.convert_to_jax_rng_key(rng.PRNGKey(1)), dtype=np.uint32)
    kp = key.ctypes.data_as(C.POINTER(C.c_uint32))
    rows = fam._rows(batch, 0, B)
    theta, eps = fam._draw(desc, params, kp, B, 0, B)
    U, h = fam.potential_and_grad(theta, rows, N)
    mask_t, _ = s._mask_arg(mask, B)
    num_valid = batch[0].num_valid if isinstance(batch[0], mb.BatchView) else None
    n_part = C.c_uint32(0)
    need = _n.lib().d3p_autodiag_workspace_bytes(C.byref(desc), B, C.byref(n_part))
    ws = s._workspace(need)

    def step():
        _n.check(_n.lib().d3p_dpsvi_step_autodiag(
            C.byref(desc), params, _n.ptr(eps), _n.ptr(h), fam.latent_dim, _n.ptr(U), _n.ptr(mask_t), _n.ptr(num_valid),
            B, 0, B, float(st.observation_scale), float(s._clipping_threshold), None, None, None, _n.ptr(ws), need,
            _n.stream_ptr()), "step")

    ctx = s._update_launch_step(st, batch, mask)
    out = {"batch_rows": B, "n_partials": n_part.value,
           "draw_ms": timed(lambda: fam._draw(desc, params, kp, B, 0, B), reps),
           "potential_and_autograd_ms": timed(lambda: fam.potential_and_grad(theta, rows, N), reps),
           "step_ms": timed(step, reps),
           "finalize_ms": timed(lambda: s._update_finalize(ctx), reps),
           "update_same_batch_ms": timed(lambda: s.update(st, *batch, mask=mask), reps)}
    return out


def kernel_times(s, st, batch, mask, reps):
    """Per-kernel mean device time (us) of `update` on a fixed batch, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    s.update(st, *batch, mask=mask)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            s.update(st, *batch, mask=mask)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            out[ev.key[:120]] = {"count": ev.count, "mean_us": t / ev.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["mean_us"] * kv[1]["count"]))


def examples_per_s(s, st, get, bst, steps):
    """examples/s of update over `steps` fresh Poisson batches (host clock around work ending in a synchronise)."""
    import time
    batches = [get(i, bst) for i in range(steps + 2)]
    n = sum(int(b[0][0].num_valid.item()) for b in batches[2:])
    for b, m in batches[:2]:
        st, _ = s.update(st, *b, mask=m)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b, m in batches[2:]:
        st, _ = s.update(st, *b, mask=m)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"steps": steps, "examples": n, "seconds": dt, "examples_per_s": n / dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--N", type=int, default=1_000_000)
    ap.add_argument("--q", type=float, default=0.1)
    ap.add_argument("--d", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    N, d, q = a.N, a.d, a.q
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    X = torch.randn((N, d), device=dev, generator=g) / d ** 0.5
    w = torch.randn(d, device=dev, generator=g)
    y_bin = (torch.rand(N, device=dev, generator=g) < torch.sigmoid(X @ w)).to(torch.int32)
    y_cnt = torch.poisson(torch.exp(0.5 * (X @ w)).clamp(max=50.), generator=g)
    result = {"config": dict(N=N, d=d, q=q, expected_batch=N * q, reps=a.reps, steps=a.steps), **device_info()}
    workloads = {
        "logreg_user": (lambda: models.AutoDiagonalNormalModel([("w", (d,)), ("intercept", ())], logreg_ll), (X, y_bin)),
        "logreg_fused": (lambda: models.LogisticRegression(d, guide="auto"), (X, y_bin)),
        "poisson_user": (lambda: models.AutoDiagonalNormalModel([("w", (d,)), ("b", ())], poisson_ll), (X, y_cnt)),
    }
    for name, (make, data) in workloads.items():
        fam = make()
        s = dsvi.DPSVI(fam.model, fam.guide, optimizers.Adam(1e-3), models.Trace_ELBO(), 1.0, 1.0, num_obs_total=N)
        init, get = mb.poisson_batchify_data(data, q, .99)
        _, bst = init(rng.PRNGKey(4))
        batch, mask = get(0, bst)
        st = s.init(rng.PRNGKey(2), *batch)
        r = {}
        if isinstance(fam, models.AutoDiagonalNormalModel):
            r["phases"] = phases(fam, s, st, batch, mask, a.reps)
            r["kernels"] = kernel_times(s, st, batch, mask, 5)
        r["update"] = examples_per_s(s, st, get, bst, a.steps)
        result[name] = r
        print(name, json.dumps(r.get("phases", {})), json.dumps(r["update"]), flush=True)
        del s, st, fam
        torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
