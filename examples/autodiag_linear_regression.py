#!/usr/bin/env python
"""A model of your own on d3p_b200: Bayesian linear regression with an unknown noise scale, trained under an
AutoDiagonalNormal guide with DP-SVI.  The workflow is d3p's: the noise scale from the privacy accountant, Poisson
batches for training, ``DPSVI.run_epoch`` per epoch and ``evaluate`` on held-out split batches.

The model is given as two torch functions of the latents, ``log_likelihood(latents, X, y) -> [B]`` and (here the
default) ``log_prior``, one value per example.  The noise scale is constrained (sigma > 0), so the model samples the
unconstrained ``log_sigma``: its N(0, 1) prior is the density of log_sigma under sigma ~ LogNormal(0, 1), Jacobian
included.  Needs a B200 (no CPU fallback).

    python examples/autodiag_linear_regression.py --num-epochs 20 --epsilon 1.0
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import d3p_b200.random as rng_suite                                                    # noqa: E402
from d3p_b200 import models, optimizers                                                # noqa: E402
from d3p_b200.dputil import approximate_sigma_remove_relation                          # noqa: E402
from d3p_b200.minibatch import poisson_batchify_data, split_batchify_data              # noqa: E402
from d3p_b200.svi import DPSVI                                                         # noqa: E402


def log_likelihood(latents, X, y):
    """y_i ~ N(x_i . w + b, exp(log_sigma))."""
    mean = (X * latents["w"]).sum(-1) + latents["b"]
    log_sigma = latents["log_sigma"]
    z = (y - mean) * torch.exp(-log_sigma)
    return -0.5 * z * z - log_sigma - 0.5 * math.log(2 * math.pi)


def create_toy_data(N, w_true, b_true, sigma_true, seed=0):
    rs = np.random.RandomState(seed)
    X = rs.randn(2 * N, len(w_true)).astype(np.float32)
    y = (X @ w_true + b_true + sigma_true * rs.randn(2 * N)).astype(np.float32)
    dev = torch.device("cuda", torch.cuda.current_device())
    X, y = torch.tensor(X, device=dev), torch.tensor(y, device=dev)
    return (X[:N], y[:N]), (X[N:], y[N:])


def main(args):
    w_true, b_true, sigma_true = np.array([1.5, -1.0, 0.5], np.float32), 0.5, 0.5
    train_data, test_data = create_toy_data(args.num_samples, w_true, b_true, sigma_true)
    d = len(w_true)
    fam = models.AutoDiagonalNormalModel([("w", (d,)), ("b", ()), ("log_sigma", ())], log_likelihood)

    q = args.batch_size / args.num_samples
    train_init, train_fetch = poisson_batchify_data(train_data, q, max_batch_size=.99, rng_suite=rng_suite)
    test_init, test_fetch = split_batchify_data(test_data, batch_size=args.batch_size, rng_suite=rng_suite)

    dpsvi_rng = rng_suite.PRNGKey(0)
    dpsvi_rng, svi_init_rng, data_fetch_rng = rng_suite.split(dpsvi_rng, 3)
    num_iter_per_epoch, batchifier_state = train_init(rng_key=data_fetch_rng)
    delta = 1 / args.num_samples ** 2
    num_iter = num_iter_per_epoch * args.num_epochs
    dp_scale, _, _ = approximate_sigma_remove_relation(args.epsilon, delta=delta, q=q, num_iter=num_iter)

    svi = DPSVI(fam.model, fam.guide, optimizers.Adam(args.learning_rate), models.Trace_ELBO(), dp_scale=dp_scale,
                clipping_threshold=args.clip, num_obs_total=args.num_samples, rng_suite=rng_suite)
    svi_state = svi.init(svi_init_rng, *train_fetch(0, batchifier_state)[0])

    for i in range(args.num_epochs):
        dpsvi_rng, data_fetch_rng = rng_suite.split(dpsvi_rng, 2)
        num_batches, batchifier_state = train_init(rng_key=data_fetch_rng)
        svi_state, stats = svi.run_epoch(svi_state, train_fetch, batchifier_state, num_batches)
        num_test, test_state = test_init(rng_key=data_fetch_rng)
        test_loss = float(svi.evaluate_epoch(svi_state, test_fetch, test_state, num_test).sum()) / (
            args.num_samples * num_test)
        print(f"epoch {i}: train loss {float(stats[:, 0].sum()) / (args.num_samples * num_batches):.4f}, "
              f"test loss {test_loss:.4f}")

    loc = svi.get_params(svi_state)["auto_loc"].cpu().numpy()
    out = dict(w_loc=loc[:d].tolist(), w_true=w_true.tolist(), b=float(loc[d]), b_true=b_true,
               sigma=float(np.exp(loc[d + 1])), sigma_true=sigma_true, dp_scale=dp_scale, test_loss=test_loss,
               epsilon=svi.get_epsilon(delta, q, num_iter=num_iter))
    print(json.dumps(out))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f)
    return out


def parse(argv=None):
    p = argparse.ArgumentParser(description="DP-SVI linear regression with a learned noise scale on d3p_b200")
    p.add_argument("-e", "--epsilon", default=1., type=float)
    p.add_argument("-n", "--num-epochs", default=20, type=int)
    p.add_argument("-lr", "--learning-rate", default=1e-2, type=float)
    p.add_argument("--batch-size", default=200, type=int)
    p.add_argument("--clip", default=5., type=float)
    p.add_argument("-N", "--num-samples", default=20000, type=int)
    p.add_argument("--json", default=None, help="also write the learned parameters to this JSON file")
    return p.parse_args(argv)


if __name__ == "__main__":
    main(parse())
