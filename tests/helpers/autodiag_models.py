"""User models of the AutoDiagonalNormalModel tests: torch log densities ``(latents, *batch) -> [B]`` with
``latents[site]`` of shape [B, *shape].  The same functions feed d3p_b200.models.AutoDiagonalNormalModel (float32 on
the device) and oracle.families.AutoDiagonalNormalModel (float64 autodiff, one example at a time under vmap)."""
import math

import torch

LOG_SQRT_2PI = math.log(math.sqrt(2 * math.pi))


def normal_lp(x, loc, scale):
    scale = torch.as_tensor(scale, dtype=x.dtype, device=x.device)
    z = (x - loc) / scale
    return -0.5 * z * z - torch.log(scale) - LOG_SQRT_2PI


def logreg_ll(lat, X, y):
    """examples/logistic_regression.py: y ~ Bernoulli(logits = X w + intercept)."""
    z = (X * lat["w"]).sum(-1) + lat["intercept"]
    return -(torch.clamp(z, min=0) + torch.log1p(torch.exp(-torch.abs(z))) - z * y.to(z.dtype))


def gauss_ll(lat, X):
    """examples/simple_gaussian_posterior.py: x ~ N(mu, 0.1) per dimension."""
    return normal_lp(X, lat["mu"], 0.1).sum(-1)


def unit_gauss_ll(lat, X):
    """tests/test_dpsvi.py:65-70 (GenericNormalMean): x ~ N(mu, 1)."""
    return normal_lp(X, lat["mu"], 1.0).sum(-1)


def linreg_ll(lat, X, y):
    """y ~ N(X w + b, sigma) with sigma = exp(log_sigma); the default N(0, 1) prior on log_sigma is the density of
    log_sigma under sigma ~ LogNormal(0, 1), Jacobian included."""
    mean = (X * lat["w"]).sum(-1) + lat["b"]
    return normal_lp(y, mean, torch.exp(lat["log_sigma"]))


def poisson_ll(lat, X, y):
    """y ~ Poisson(exp(X w + b)) with float counts."""
    eta = (X * lat["w"]).sum(-1) + lat["b"]
    return y * eta - torch.exp(eta) - torch.lgamma(y + 1)


def softmax_ll(lat, X, y):
    """y ~ Categorical(logits = W x + b) with W of shape [K, d]: a matrix-shaped site."""
    logits = (lat["W"] * X.unsqueeze(-2)).sum(-1) + lat["b"]
    K = logits.shape[-1]
    onehot = (torch.arange(K, device=logits.device) == y.unsqueeze(-1).to(torch.int64)).to(logits.dtype)
    return (torch.log_softmax(logits, -1) * onehot).sum(-1)


def nan_at_zero_gauss_ll(lat, X):
    """gauss_ll times |x|_1 / |x|_1: the same value on every record, NaN (value and gradient) on an all-zero row."""
    r = X.abs().sum(-1)
    return gauss_ll(lat, X) * (r / r)


# name -> (sites(d), log_likelihood, batch kind)
MODELS = {
    "linreg": (lambda d: [("w", (d,)), ("b", ()), ("log_sigma", ())], linreg_ll, "real"),
    "poisson": (lambda d: [("w", (d,)), ("b", ())], poisson_ll, "count"),
    "softmax": (lambda d: [("W", (3, d)), ("b", (3,))], softmax_ll, "class3"),
    "generic_normal_mean": (lambda d: [("mu", (d,))], unit_gauss_ll, "x_only"),
}
