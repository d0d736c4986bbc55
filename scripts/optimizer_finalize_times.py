#!/usr/bin/env python
"""Finalize-kernel time per optimizer kind (reduce + noise + rescale + optimizer step, d3p_perturb_finalize_f32).

Two shapes: C2 (P = 2 050, 296 partial rows: finalize_kernel) and C5 (P = 652 824, 4 partial rows:
finalize_quad_kernel).  Each kind is timed with CUDA events around `--launches` back-to-back launches on the same
buffers after `--warmup` launches; the kinds are interleaved over `--rounds` rounds and the median round is reported
(us per launch).  The working set (partial rows, x, m, v) of both shapes fits in the 126 MB L2, so these are
L2-resident times, as in the training loop where the step kernel has just written the partial rows.

    python scripts/optimizer_finalize_times.py [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"c2": (2050, 296, [1024, 1024, 1, 1]), "c5": (652824, 4, None)}


def _leaves(P, lens):
    from d3p_b200 import _native as _n
    import d3p_b200.random as rng
    if lens is None:                    # the C5 VAE (784-400-20): 10 leaves in pytree order
        D, H, Z = 784, 400, 20
        lens = [Z * H, H, H * D, D, D * H, H, H * Z, Z, H * Z, Z]
    assert sum(lens) == P, (sum(lens), P)
    lt = _n.LeafTable()
    lt.n_leaves = len(lens)
    keys = rng.split(rng.PRNGKey(3), len(lens))
    off = 0
    for l, n in enumerate(lens):
        lt.leaf_off[l], lt.leaf_len[l] = off, n
        for i in range(16):
            lt.site_state[l][i] = int(np.asarray(keys[l], np.uint32).reshape(16)[i])
        off += n
    return lt


def _optims():
    from d3p_b200 import optimizers as o
    sched = o.exponential_decay(1e-3, 1000, 0.5)
    return [("sgd", o.SGD(1e-3)), ("adam", o.Adam(1e-3)), ("momentum", o.Momentum(1e-3, 0.9)),
            ("adagrad", o.Adagrad(1e-3)), ("rmsprop", o.RMSProp(1e-3)), ("rmsprop_momentum", o.RMSPropMomentum(1e-3)),
            ("clipped_adam", o.ClippedAdam(1e-3)), ("adam+exponential_decay", o.Adam(sched)),
            ("rmsprop_momentum+exponential_decay", o.RMSPropMomentum(sched))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from d3p_b200 import _native as _n
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lib = _n.lib()
    dev = torch.device("cuda", 0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = "nvidia-smi unavailable"
    result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi, "launches": args.launches,
              "rounds": args.rounds, "us_per_launch": {}}
    stream = _n.stream_ptr()
    for shape, (P, n_part, lens) in SHAPES.items():
        lt = _leaves(P, lens)
        g = torch.Generator(device=dev).manual_seed(0)
        part = torch.randn(n_part, P + 2, device=dev, generator=g) * 0.01
        part[:, P + 1] = 0
        part[0, P + 1] = 256
        times = {name: [] for name, _ in _optims()}
        for _ in range(args.rounds):
            for name, opt in _optims():
                x = torch.randn(P, device=dev, generator=g)
                m, v = torch.zeros(P, device=dev), torch.zeros(P, device=dev)
                od = opt.desc(0)

                def launch():
                    _n.check(lib.d3p_perturb_finalize_f32(_n.ptr(part), n_part, P, 512, C.byref(lt), 1.0, 1.0, 1.0, 1,
                                                          None, C.byref(od), _n.ptr(x), _n.ptr(m), _n.ptr(v), None,
                                                          None, stream), name)
                for _ in range(args.warmup):
                    launch()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.launches):
                    launch()
                e1.record()
                e1.synchronize()
                times[name].append(e0.elapsed_time(e1) * 1e3 / args.launches)
        result["us_per_launch"][f"{shape} (P={P}, rows={n_part})"] = {
            k: {"median": round(float(np.median(t)), 3), "min": round(float(np.min(t)), 3),
                "max": round(float(np.max(t)), 3)} for k, t in times.items()}
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
