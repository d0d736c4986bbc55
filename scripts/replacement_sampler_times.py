#!/usr/bin/env python
"""What drawing with-replacement minibatches on the device costs, before and after the one-launch randint.

"before" is the path the library took for ``subsample_batchify_data(with_replacement=True)`` until the one-launch
kernel existed: ``randint`` ran its rejection loop from the host (one ``d3p_chacha_randint_round`` launch and one
4-byte device->host read per round, then ``d3p_randint_finish``), and ``run_epoch`` stepped through
``get_batch`` + ``update`` in Python because the batchifier had no C-side description.  The script restates that
loop (``randint_per_round``) and wraps it in a batchifier without a ``spec``, so both arms run in the same process on
the same data.  "after" is ``rng.randint`` (``d3p_chacha_randint``) and ``run_epoch`` through the C epoch driver.

Reports:
  * ms per ``randint`` call at B = 100 736, N = 10 M (CUDA events around `reps` calls, ending in a synchronise);
  * ms per step of ``run_epoch`` at a C1-sized problem (logistic regression d = 8, N = 10 k, B = 200) and a C3-sized
    one (Gaussian mean d = 256, B = 500 000 of N = 50 M), host clock around calls that end in a synchronise, the arms
    alternated `repeats` times; the parameters of both arms are compared bit for bit.
The device name and power limit are read in the same run.

    python scripts/replacement_sampler_times.py --out profiles/replacement_sampler_times_b200.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import d3p_b200.random as rng                                                   # noqa: E402
from d3p_b200 import _native as _n, minibatch as mb, models, optimizers, svi as dsvi  # noqa: E402


def device_info():
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["power_limit_and_max_sm_clock"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"not read: {e}"
    return out


def randint_per_round(key, n, minval, maxval):
    """int32 randint as the host-driven round loop (the "before" arm); same values as rng.randint."""
    lib = _n.lib()
    delta = (maxval - 1 - minval) & 0xFFFFFFFF
    log_po2 = min(int(np.float32(np.log2(np.float32(delta))) + np.float32(1)) if delta > 0 else 0, 32)
    bitmask = ((1 << log_po2) - 1) & 0xFFFFFFFF
    vals = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    pending = torch.zeros(1, dtype=torch.int32, device="cuda")
    first, rounds = 1, 0
    while True:
        ks = rng.split(key, 2)
        key, round_key = ks[0], ks[1]
        a, p = _n.u32(round_key.reshape(16))
        _n.check(lib.d3p_chacha_randint_round(p, 32, bitmask, delta, first, _n.ptr(vals), n, _n.ptr(pending),
                                              _n.stream_ptr()), "randint_round")
        first, rounds = 0, rounds + 1
        if int(pending.item()) == 0:
            break
    out = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    _n.check(lib.d3p_randint_finish(_n.ptr(vals), int(minval), 32, _n.ptr(out), n, _n.stream_ptr()), "randint_finish")
    randint_per_round.rounds = rounds
    return out[:n]


def per_round_batchifier(dataset, batch_size):
    """subsample_batchify_data(with_replacement=True) as it was: per-round randint and no spec."""
    init, _ = mb.subsample_batchify_data(dataset, batch_size=batch_size, with_replacement=True)
    data = tuple(mb._to_device(a) for a in dataset)
    N = len(data[0])

    def get_batch(i, state):
        idx = randint_per_round(rng.fold_in(state, i), batch_size, 0, N)
        return tuple(mb.BatchView(a, idx) for a in data)

    return init, get_batch


def randint_times(reps):
    n, N = 100_736, 10_000_000
    key = rng.PRNGKey(3)
    assert torch.equal(rng.randint(key, (n,), 0, N), randint_per_round(key, n, 0, N))
    out = {"B": n, "N": N, "reps": reps, "rounds_of_the_per_round_loop": []}
    for name, fn in (("per_round_loop", lambda k: randint_per_round(k, n, 0, N)),
                     ("one_launch", lambda k: rng.randint(k, (n,), 0, N))):
        keys = [rng.fold_in(key, i) for i in range(reps + 1)]
        fn(keys[0])
        b, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        rounds = []
        b.record()
        for k in keys[1:]:
            fn(k)
            if name == "per_round_loop":
                rounds.append(randint_per_round.rounds)
        e.record()
        e.synchronize()
        out[name + "_ms"] = b.elapsed_time(e) / reps
        if rounds:
            out["rounds_of_the_per_round_loop"] = [int(min(rounds)), float(np.mean(rounds)), int(max(rounds))]
    return out


def epoch_times(name, fam, data, B, steps, warmup, repeats):
    N = len(data[0])
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.Adam(1e-3), models.Trace_ELBO(), 1.0, 1.0, num_obs_total=N)
    init_c, get_c = mb.subsample_batchify_data(data, batch_size=B, with_replacement=True)
    _, get_p = per_round_batchifier(data, B)
    _, bst = init_c(rng.PRNGKey(4))
    st0 = s.init(rng.PRNGKey(2), *get_c(0, bst))
    arms = {"before_stepwise_per_round": get_p, "after_c_driver": get_c}
    res = {"N": N, "B": B, "steps": steps, "warmup_steps": warmup, "repeats": repeats}
    finals = {}
    for arm, get in arms.items():                       # warm-up: modules, workspaces, the epoch plan
        s.run_epoch(st0, get, bst, warmup)
    torch.cuda.synchronize()
    for r in range(repeats):
        for arm, get in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            st, _ = s.run_epoch(st0, get, bst, steps, first_step=warmup)
            torch.cuda.synchronize()
            res.setdefault(arm + "_ms_per_step", []).append((time.perf_counter() - t0) * 1e3 / steps)
            finals[arm] = st.optim_state.flat.clone()
    res["parameters_bit_identical"] = bool(torch.equal(*finals.values()))
    for arm in arms:
        v = res[arm + "_ms_per_step"]
        res[arm + "_ms_per_step_median"] = float(np.median(v))
    print(name, json.dumps(res), flush=True)
    del s
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--c3-records", type=int, default=50_000_000)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    result = {**device_info(), "timing": "randint: CUDA events; run_epoch: host clock around calls ending in a "
                                         "synchronise. C3's data set (51 GB) is far larger than L2."}
    result["randint"] = randint_times(a.reps)
    print("randint", json.dumps(result["randint"]), flush=True)
    g = torch.Generator(device=dev).manual_seed(0)
    N, d = 10_000, 8
    X = torch.randn((N, d), device=dev, generator=g)
    y = (torch.rand(N, device=dev, generator=g) < torch.sigmoid(X @ torch.randn(d, device=dev, generator=g))).to(torch.int32)
    result["c1_logreg"] = epoch_times("c1_logreg", models.LogisticRegression(d), (X, y), 200, a.steps, a.warmup,
                                      a.repeats)
    del X, y
    N, d = a.c3_records, 256
    X = torch.empty((N, d), device=dev).normal_(1.0, 0.1, generator=g)
    result["c3_gauss"] = epoch_times("c3_gauss", models.GaussianMean(d), (X,), 500_000, a.steps, a.warmup, a.repeats)
    del X
    torch.cuda.empty_cache()
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
