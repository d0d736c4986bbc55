"""``DPSVI.evaluate`` (``d3p/svi.py:436-449``) on the device: numpyro's ``SVI.evaluate`` draws one guide
sample for the whole batch from ``split(rng_key)[1]`` and returns ``Trace_ELBO.loss`` with the plate scale
``N / B``.  ``d3p_elbo_evaluate_meanfield`` / ``_vae`` / ``_gmm``: the four fused model families;
``AutoDiagonalNormalModel`` draws with ``d3p_autodiag_draw_f32`` and evaluates its likelihood in torch."""
import ctypes as C

import numpy as np
import torch

from . import _native as _n
from .models import AutoDiagonalNormalModel


def _threefry_split_second(key):
    """jax.random.split(key, 2)[1] on the host (two Threefry calls; same arithmetic as common.cuh)."""
    k0, k1 = int(key[0]), int(key[1])
    M = 0xFFFFFFFF
    ks = (k0, k1, k0 ^ k1 ^ 0x1BD11BDA)
    rot = ((13, 15, 26, 6), (17, 29, 16, 24))

    def tf(c0, c1):
        x0, x1 = (c0 + ks[0]) & M, (c1 + ks[1]) & M
        for r in range(5):
            for s in rot[r % 2]:
                x0 = (x0 + x1) & M
                x1 = ((x1 << s) | (x1 >> (32 - s))) & M
                x1 ^= x0
            x0 = (x0 + ks[(r + 1) % 3]) & M
            x1 = (x1 + ks[(r + 2) % 3] + r + 1) & M
        return x0, x1

    a = tf(0, 2)
    b = tf(1, 3)
    return np.array([a[1], b[1]], dtype=np.uint32)


def evaluate_elbo(svi, svi_state, jax_key, args):
    fam = svi.family
    # the reference's evaluate has no mask: a Poisson batch enters with its padding rows zero-filled
    # (d3p/minibatch.py:126-131), so those are materialised rather than read through the index list
    from .minibatch import BatchView
    args = tuple(a.tensor() if (isinstance(a, BatchView) and a.num_valid is not None) else a for a in args)
    key = _threefry_split_second(np.asarray(jax_key, dtype=np.uint32).reshape(2))    # SVI.evaluate: _, rng_key_eval
    if isinstance(fam, AutoDiagonalNormalModel):            # the likelihood is torch code: it takes the arrays as given
        loss = torch.empty(1, dtype=torch.float32, device=torch.device("cuda", torch.cuda.current_device()))
        fam._evaluate(svi, fam.desc(svi._num_obs_total()), svi_state.optim_state.flat, args,
                      key.ctypes.data_as(C.POINTER(C.c_uint32)), loss)
        return loss[0]
    b = svi._resolve_args(args)
    if b.local_rows is not None:
        raise NotImplementedError("DPSVI.evaluate takes whole batches (LocalRows are a sharded-update input)")
    desc = fam.desc(svi._num_obs_total())
    loss = torch.empty(1, dtype=torch.float32, device=b.x.device)
    fam._evaluate(svi, desc, _n.ptr(svi_state.optim_state.flat), b, key.ctypes.data_as(C.POINTER(C.c_uint32)), loss)
    return loss[0]
