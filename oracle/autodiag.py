"""Oracle: a user model with real-valued latents under an AutoDiagonalNormal guide.  TEST INFRASTRUCTURE ONLY.

The counterpart of ``d3p_b200.models.AutoDiagonalNormalModel``: the caller's torch log densities on the mean-field
machinery of ``oracle/families.py`` (joint ``_auto_latent`` site, softplus link, numpyro's seed-handler plumbing), so
float64 autodiff of the same functions is the reference for the CUDA path.
"""
import numpy as np

from .families import _MeanFieldFamily, normal_log_prob, softplus_inv


class AutoDiagonalNormalModel(_MeanFieldFamily):
    """``d3p_b200.models.AutoDiagonalNormalModel``: the caller's ``log_likelihood(latents, *batch) -> [B]`` and
    ``log_prior(latents) -> [B]`` (``latents``: site -> [B, *shape]; default prior N(0, 1) per element) under an
    AutoDiagonalNormal guide.  The oracle hands them one example at a time (B = 1, or the whole batch with one shared
    draw in ``DPSVI.evaluate``), so autodiff of the same functions in float64 is the reference."""
    link = "softplus"
    joint_site = True

    def __init__(self, sites, log_likelihood, num_obs_total, log_prior=None, init_scale=0.1):
        self.site_shapes = [(name, tuple(shape)) for name, shape in sites]
        self.sites = [(name, int(np.prod(shape)) if len(shape) else 1) for name, shape in self.site_shapes]
        self.num_obs_total = float(num_obs_total)
        self._log_lik, self._log_prior, self.init_scale = log_likelihood, log_prior, float(init_scale)

    def init_params(self, auto_loc=None):
        D = self.latent_dim()
        loc = np.zeros(D, np.float32) if auto_loc is None else np.asarray(auto_loc, np.float32)
        return {"auto_loc": loc, "auto_scale": np.full(D, softplus_inv(self.init_scale), np.float32)}

    def loc_scale(self, p):
        return {"_auto_latent": (p["auto_loc"], self.scale_of(p["auto_scale"]))}

    def _batched(self, lat, n):
        return {name: lat[name].reshape((1,) + shape).expand((n,) + shape) for name, shape in self.site_shapes}

    def log_prior(self, lat):
        if self._log_prior is None:
            return sum(normal_log_prob(v, 0., 1.).sum() for v in lat.values())
        return self._log_prior(self._batched(lat, 1)).sum()

    def log_lik(self, lat, *args):
        return self._log_lik(self._batched(lat, args[0].shape[0]), *args).sum()
