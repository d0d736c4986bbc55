#!/usr/bin/env python
"""The REAL reference (DPBayes/d3p + jax + numpyro + jax-chacha-prng), where it can be imported.

Two jobs, both guarded by ``available()``:

* ``time_update(cfg, ...)``  — the reference's own ``DPSVI.update`` (with its batchifier's ``get_batch``) under
  ``jax.jit`` on the host CPU, ``block_until_ready`` around the timed loop; ``bench.py --impl reference`` prefers it
  over the oracle port (``cpu_baseline.kind = "reference"``).
* ``dump_golden(path)``      — outputs of the reference on fixed seeds (``tests/golden/make_reference_golden.py``
  writes ``tests/golden/reference_v1.npz``): ChaCha key plumbing (``PRNGKey/split/fold_in/random_bits/uniform/normal/
  randint/convert_to_jax_rng_key``), Feistel and Poisson indices, per-example Threefry keys and guide normals, jax
  gamma draws, 3-step ``DPSVI.update`` trajectories per model family, and 3-step logistic-regression trajectories with
  numpyro's other optimizers and a scheduled Adam (``OPTIM_CASES``, keys ``optraj_*``).
  ``tests/test_reference_golden.py`` (and ``tests/test_reference_optimizers.py`` for the ``optraj_*`` keys) holds the
  oracle and the CUDA path to that file: this is the one command that turns "parity unpinned" (the key-derivation rule
  of jax-chacha-prng, numpyro's seed plumbing, jax's gamma sampler: DESIGN.md section 8) into a pinned statement.

Neither jax nor numpyro nor jax-chacha-prng is in this image or its wheelhouse (``setup.py:46-49`` of the reference
pins them), so here ``available()`` is False and nothing below the guard has ever run in this container; the writer
side is exercised through the same ``dump()`` with the oracle as the implementation (``OracleImpl``), which checks
the file format and the consumer, not the reference.

The reference is looked up in ``baseline/_ref`` (a pip --target install, git-ignored).
"""
import importlib.util
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIRS = [os.path.join(ROOT, "baseline", "_ref")]
NEEDED = ("jax", "numpyro", "chacha")

SEEDS = (0, 1, 123, (1 << 40) + 5)

# Optimizer cases of the short logistic-regression trajectories under the ``optraj_*`` keys: numpyro.optim class name,
# positional and keyword arguments.  A step size given as (schedule name, args) is that schedule of
# jax.example_libraries.optimizers (the oracle side: oracle/optim.py, same names).
OPTIM_CASES = {
    "momentum": ("Momentum", (1e-3, 0.9), {}),
    "adagrad": ("Adagrad", (1e-2,), {"momentum": 0.8}),
    "rmsprop": ("RMSProp", (1e-3,), {"gamma": 0.8}),
    "rmsprop_momentum": ("RMSPropMomentum", (1e-3,), {"gamma": 0.8, "momentum": 0.7}),
    "clipped_adam": ("ClippedAdam", (1e-3,), {"clip_norm": 10.0}),
    "adam_exponential_decay": ("Adam", (("exponential_decay", (1e-3, 2, 0.5)),), {}),
}


def make_optim(spec, optim_module, schedule_module):
    """An optimizer of ``OPTIM_CASES`` from ``optim_module`` (numpyro.optim or oracle.optim), its schedule (if any)
    from ``schedule_module`` (jax.example_libraries.optimizers or oracle.optim)."""
    cls, args, kwargs = spec
    if args and isinstance(args[0], tuple):
        name, sargs = args[0]
        args = (getattr(schedule_module, name)(*sargs),) + tuple(args[1:])
    return getattr(optim_module, cls)(*args, **kwargs)
FOLD_DATA = (0, 1, 7, 1 << 31)


def available():
    """-> (ok, reason)"""
    missing = [m for m in NEEDED if importlib.util.find_spec(m) is None]
    if missing:
        return False, "not importable: " + ", ".join(missing) + " (reference pins: setup.py:46-49)"
    for d in REF_DIRS:
        if os.path.isdir(os.path.join(d, "d3p")):
            return True, d
    return False, "no d3p package under " + " or ".join(REF_DIRS)


def _import_reference():
    ok, where = available()
    if not ok:
        raise RuntimeError("reference unavailable: " + where)
    for p in (where, os.path.join(where, "examples")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.setdefault("JAX_PLATFORMS", "cpu")
    import d3p  # noqa: F401
    return where


# ----------------------------------------------------------------------------------------------------------------------
# Implementations behind dump(): the real reference, and the oracle (format / consumer check only)
# ----------------------------------------------------------------------------------------------------------------------
class ReferenceImpl:
    """Thin adapter: every method calls the reference's public API (d3p.random, d3p.util, d3p.minibatch, d3p.svi) or
    jax.random / numpyro exactly as d3p's own code does; results come back as numpy arrays."""
    name = "reference"

    def __init__(self):
        self.where = _import_reference()
        import jax
        import jax.numpy as jnp
        import numpyro
        import d3p.minibatch
        import d3p.random
        import d3p.svi
        import d3p.util
        self.jax, self.jnp, self.numpyro = jax, jnp, numpyro
        self.rng, self.util, self.mb, self.svi = d3p.random, d3p.util, d3p.minibatch, d3p.svi
        self.versions = {"jax": jax.__version__, "numpyro": numpyro.__version__,
                         "chacha": getattr(__import__("chacha"), "__version__", "?")}

    # rng suite (d3p/random/__init__.py:28-155)
    def PRNGKey(self, seed): return np.asarray(self.rng.PRNGKey(seed))
    def split(self, key, n): return np.asarray(self.rng.split(self.jnp.asarray(key), n))
    def fold_in(self, key, data): return np.asarray(self.rng.fold_in(self.jnp.asarray(key), data))
    def random_bits(self, key, width, shape): return np.asarray(self.rng.random_bits(self.jnp.asarray(key), width, shape))
    def uniform(self, key, shape, lo=0., hi=1.):
        return np.asarray(self.rng.uniform(self.jnp.asarray(key), shape, self.jnp.float32, lo, hi))
    def normal(self, key, shape): return np.asarray(self.rng.normal(self.jnp.asarray(key), shape, self.jnp.float32))
    def randint(self, key, shape, lo, hi): return np.asarray(self.rng.randint(self.jnp.asarray(key), shape, lo, hi))
    def convert_to_jax_rng_key(self, key): return np.asarray(self.rng.convert_to_jax_rng_key(self.jnp.asarray(key)))

    # samplers (d3p/util.py:216-301, d3p/minibatch.py:29-39)
    def sample_indices(self, key, capacity, n):
        return np.asarray(self.util.sample_from_array(self.jnp.asarray(key), self.jnp.arange(capacity), n, 0,
                                                      rng_suite=self.rng))

    def poisson_sample_idxs(self, key, q, N, cutoff):
        idxs, num = self.mb.poisson_sample_idxs(self.jnp.asarray(key), q, N, self.rng, cutoff_size=cutoff)
        return np.asarray(idxs), int(num)

    # jax.random pieces the per-example path uses (d3p/svi.py:290; numpyro seed handler; Dirichlet / InverseGamma)
    def threefry_split(self, key2, n): return np.asarray(self.jax.random.split(self.jnp.asarray(key2, self.jnp.uint32), n))
    def threefry_normal(self, key2, n):
        return np.asarray(self.jax.random.normal(self.jnp.asarray(key2, self.jnp.uint32), (n,), self.jnp.float32))
    def threefry_gamma(self, key2, alpha):
        return np.asarray(self.jax.random.gamma(self.jnp.asarray(key2, self.jnp.uint32), self.jnp.asarray(alpha)))

    # DPSVI trajectories -----------------------------------------------------------------------------------------
    def _family(self, fam):
        """-> (model, guide, static kwargs, clipping threshold) taken from the reference's example files."""
        if fam == "logreg":
            import logistic_regression as ex
            return ex.model, ex.guide, {}, 1.0
        if fam == "gauss":
            import simple_gaussian_posterior as ex
            return ex.model, ex.guide, {"d": None}, 1.0
        if fam == "gmm":
            import gaussian_mixture_model as ex
            return ex.model, ex.guide, {}, 20.0
        if fam == "vae":
            import vae as ex
            return ex.model, ex.guide, {}, 10.0
        raise ValueError(fam)

    def trajectory(self, fam, data, mask, steps, seed, N, optim=None, **shape):
        """3 masked ``DPSVI.update`` steps from ``svi.init`` on a fixed batch.  Returns the flat initial parameters
        (jax pytree leaf order of the unconstrained param dict), and per step: loss, flat parameters, rng key.
        ``optim``: an ``OPTIM_CASES`` entry (default: Adam(1e-3), as the examples)."""
        import jax.example_libraries.optimizers as schedules
        import numpyro.optim as optimizers
        from numpyro.handlers import scale
        from numpyro.infer import Trace_ELBO
        jnp, jax = self.jnp, self.jax
        model, guide, kw, clip = self._family(fam)
        if fam == "gauss":
            kw = {"d": data[0].shape[1]}
        if fam == "gmm":
            K = shape["K"]
            m0, g0 = model, guide
            model = lambda obs, **k: m0(K, obs, **k)          # noqa: E731   (examples/gaussian_mixture_model.py:186-193)
            guide = lambda obs, **k: g0(K, obs, **k)          # noqa: E731
        if fam == "vae":
            model, guide = scale(model, scale=1 / N), scale(guide, scale=1 / N)       # examples/vae.py:193-194
            kw = {"z_dim": shape["z_dim"], "hidden_dim": shape["hidden_dim"]}
        opt = optimizers.Adam(1e-3) if optim is None else make_optim(optim, optimizers, schedules)
        svi = self.svi.DPSVI(model, guide, opt, Trace_ELBO(), dp_scale=1.0, clipping_threshold=clip,
                             num_obs_total=N, rng_suite=self.rng, **kw)
        batch = tuple(jnp.asarray(a) for a in data)
        state = svi.init(self.rng.PRNGKey(seed), *batch)
        leaves0, treedef = jax.tree_util.tree_flatten(svi.optim.get_params(state.optim_state))
        out = {"p0": [np.asarray(l) for l in leaves0], "treedef": str(treedef),
               "observation_scale": float(state.observation_scale), "clip": clip, "loss": [], "params": [], "rng_key": []}
        upd = jax.jit(lambda s, m: svi.update(s, *batch, mask=m))
        for _ in range(steps):
            state, loss = upd(state, jnp.asarray(mask))
            out["loss"].append(float(loss))
            out["params"].append([np.asarray(l) for l in jax.tree_util.tree_leaves(svi.optim.get_params(state.optim_state))])
            out["rng_key"].append(np.asarray(state.rng_key))
        return out


class OracleImpl:
    """The repo's own CPU oracle behind the same interface: used to test the writer / file format / consumer, never as
    a reference (the file it writes is marked ``impl = "oracle"`` and the consumer refuses to call it a pin)."""
    name = "oracle"
    versions = {}

    def __init__(self):
        if ROOT not in sys.path:
            sys.path.insert(0, ROOT)
        from oracle import chacha, gamma, minibatch, threefry
        self.c, self.g, self.m, self.t = chacha, gamma, minibatch, threefry

    def PRNGKey(self, seed): return self.c.PRNGKey(seed)
    def split(self, key, n): return self.c.split(key, n)
    def fold_in(self, key, data): return self.c.fold_in(key, data)
    def random_bits(self, key, width, shape): return self.c.random_bits(key, width, shape)
    def uniform(self, key, shape, lo=0., hi=1.): return self.c.uniform(key, shape, minval=lo, maxval=hi)
    def normal(self, key, shape): return self.c.normal(key, shape)
    def randint(self, key, shape, lo, hi): return self.c.randint(key, shape, lo, hi)
    def convert_to_jax_rng_key(self, key): return self.c.convert_to_jax_rng_key(key)
    def sample_indices(self, key, capacity, n): return self.m.sample_indices(key, capacity, n)
    def poisson_sample_idxs(self, key, q, N, cutoff): return self.m.poisson_sample_idxs(key, q, N, cutoff_size=cutoff)
    def threefry_split(self, key2, n): return self.t.split(np.asarray(key2, np.uint32), n)
    def threefry_normal(self, key2, n): return self.t.normal(np.asarray(key2, np.uint32), (n,))
    def threefry_gamma(self, key2, alpha): return self.g.gamma(np.asarray(key2, np.uint32), np.asarray(alpha, np.float32))

    def trajectory(self, fam, data, mask, steps, seed, N, optim=None, **shape):
        from oracle import families, gmm, optim as ooptim, svi, vae
        if fam == "logreg":
            f, clip = families.LogisticRegression(data[0].shape[1], N), 1.0
        elif fam == "gauss":
            f, clip = families.GaussianMean(data[0].shape[1], N), 1.0
        elif fam == "gmm":
            f, clip = gmm.GaussianMixture(shape["K"], data[0].shape[1], N), 20.0
        else:
            f, clip = vae.VAE(int(np.prod(data[0].shape[1:])), shape["hidden_dim"], shape["z_dim"], N), 10.0
        opt = svi.Adam(1e-3) if optim is None else make_optim(optim, ooptim, ooptim)
        s = svi.DPSVI(f, None, opt, None, clip, 1.0)
        p0 = f.init_params(0, 0.05) if fam == "vae" else f.init_params()
        st = s.init(self.c.PRNGKey(seed), *data, params=p0)
        order = f.flat_param_order()
        out = {"p0": [np.asarray(p0[k]) for k in order], "treedef": ",".join(order),
               "observation_scale": float(st.observation_scale), "clip": clip, "loss": [], "params": [], "rng_key": []}
        for _ in range(steps):
            st, loss = s.update(st, *data, mask=mask)
            out["loss"].append(float(loss))
            out["params"].append([np.asarray(s.get_params(st)[k]) for k in order])
            out["rng_key"].append(np.asarray(st.rng_key))
        return out


# ----------------------------------------------------------------------------------------------------------------------
def trajectory_inputs(fam):
    """Fixed inputs of the trajectory cases (numpy only, so that writer and consumer build identical arrays)."""
    rs = np.random.RandomState({"logreg": 1, "gauss": 2, "gmm": 3, "vae": 4}[fam])
    if fam == "logreg":
        B, d = 33, 8
        data = (rs.randn(B, d).astype(np.float32), (rs.rand(B) < .5).astype(np.int32))
        return data, np.arange(B) < B - 4, 10000, {}
    if fam == "gauss":
        B, d = 29, 6
        return ((1 + .1 * rs.randn(B, d)).astype(np.float32),), np.arange(B) < B - 3, 10000, {}
    if fam == "gmm":
        B, d, K = 12, 2, 3
        return ((rs.randn(B, d) * 2).astype(np.float32),), np.arange(B) != 5, 500, {"K": K}
    B = 10
    return ((rs.rand(B, 6, 6) < .4).astype(np.float32),), np.arange(B) != 2, 1000, {"z_dim": 4, "hidden_dim": 24}


def dump(impl, path, families=("logreg", "gauss", "gmm", "vae")):
    out = {"impl": np.array(impl.name), "versions": np.array(repr(impl.versions))}
    for seed in SEEDS:
        k = impl.PRNGKey(seed)
        out[f"prngkey_{seed}"] = k
        for n in (2, 3, 5):
            out[f"split_{seed}_{n}"] = impl.split(k, n)
        for dta in FOLD_DATA:
            out[f"fold_in_{seed}_{dta}"] = impl.fold_in(k, dta)
    out["prngkey_bytes"] = impl.PRNGKey(bytes(range(1, 21)))
    k = impl.PRNGKey(123)
    child = impl.split(impl.fold_in(k, 3), 2)[1]                       # a chain, as DPSVI + a batchifier build it
    out["chain_child"] = child
    for w in (8, 16, 32, 64):
        out[f"random_bits_{w}"] = impl.random_bits(child, w, (37,))
    out["random_bits_2d"] = impl.random_bits(child, 32, (10, 3))
    out["uniform_64"] = impl.uniform(child, (64,))
    out["uniform_lohi"] = impl.uniform(child, (64,), -3.0, 5.0)
    out["normal_1000"] = impl.normal(child, (1000,))
    out["randint_1000"] = impl.randint(child, (1000,), 0, 1000)
    out["randint_pow2"] = impl.randint(child, (100,), 8, 8 + 1024)
    jk = impl.convert_to_jax_rng_key(child)
    out["jax_key"] = jk
    for cap, n in ((10_000, 200), (100, 100), (60_000, 128), (1_000_003, 977)):
        out[f"feistel_{cap}_{n}"] = impl.sample_indices(child, cap, n)
    for q, N, cutoff in ((0.02, 10_000, 234), (0.3, 105, 60), (0.3, 105, 20), (0.0, 50, 10)):
        idxs, num = impl.poisson_sample_idxs(child, q, N, cutoff)
        out[f"poisson_idx_{q}_{N}_{cutoff}"], out[f"poisson_num_{q}_{N}_{cutoff}"] = idxs, np.array(num)
    out["threefry_split_37"] = impl.threefry_split(jk, 37)
    out["threefry_normal_9"] = impl.threefry_normal(jk, 9)
    out["threefry_normal_1024"] = impl.threefry_normal(jk, 1024)
    out["gamma_alpha"] = np.array([0.05, 0.3, 0.9, 1.0, 1.7, 4.2, 11.0], np.float32)
    out["threefry_gamma"] = impl.threefry_gamma(jk, out["gamma_alpha"])
    skipped = []
    for fam in families:
        data, mask, N, shape = trajectory_inputs(fam)
        try:
            tr = impl.trajectory(fam, data, mask, 3, 7, N, **shape)
        except Exception as e:        # an example module that does not import here (matplotlib, stax): say so in the file
            skipped.append(f"{fam}: {type(e).__name__}: {e}")
            continue
        out[f"traj_{fam}_treedef"] = np.array(tr["treedef"])
        out[f"traj_{fam}_obs_scale"] = np.array(tr["observation_scale"])
        out[f"traj_{fam}_loss"] = np.array(tr["loss"], np.float32)
        out[f"traj_{fam}_rng_key"] = np.stack(tr["rng_key"])
        for i, l in enumerate(tr["p0"]):
            out[f"traj_{fam}_p0_{i}"] = l
        for s, leaves in enumerate(tr["params"]):
            for i, l in enumerate(leaves):
                out[f"traj_{fam}_step{s}_{i}"] = l
    # the other numpyro optimizers and one scheduled Adam, on the logistic-regression case
    data, mask, N, shape = trajectory_inputs("logreg")
    for name, spec in OPTIM_CASES.items():
        try:
            tr = impl.trajectory("logreg", data, mask, 3, 7, N, optim=spec, **shape)
        except Exception as e:
            skipped.append(f"optim {name}: {type(e).__name__}: {e}")
            continue
        out[f"optraj_{name}_loss"] = np.array(tr["loss"], np.float32)
        out[f"optraj_{name}_rng_key"] = np.stack(tr["rng_key"])
        for s, leaves in enumerate(tr["params"]):
            for i, l in enumerate(leaves):
                out[f"optraj_{name}_step{s}_{i}"] = l
    out["skipped"] = np.array("; ".join(skipped))
    np.savez_compressed(path, **out)
    return sorted(out)


def dump_golden(path):
    return dump(ReferenceImpl(), path)


# ----------------------------------------------------------------------------------------------------------------------
def time_update(cfg, steps, warmup, rows):
    """The reference's get_batch + DPSVI.update for logistic regression (BASELINE configs 1 / 2 shapes), jitted, on the
    host CPU, at ``rows`` records x cfg["d"] with the config's q (max_batch_size = the 0.99 Poisson quantile).
    -> dict(value=examples/s, ms_per_step, examples_per_step, max_batch_size)"""
    impl = ReferenceImpl()
    import logistic_regression as ex
    import numpyro.optim as optimizers
    from numpyro.infer import Trace_ELBO
    jax, jnp, rng = impl.jax, impl.jnp, impl.rng
    d, q = cfg["d"], cfg["q"]
    kx, kw, ky = jax.random.split(jax.random.PRNGKey(123), 3)
    X = jax.random.normal(kx, (rows, d), jnp.float32)
    w = jax.random.normal(kw, (d + 1,), jnp.float32)
    y = (jax.random.uniform(ky, (rows,)) < jax.nn.sigmoid(X @ w[:d] + w[d])).astype(jnp.int32)
    init, get_batch = impl.mb.poisson_batchify_data((X, y), q, .99, rng_suite=rng)
    key, k_init, k_fetch = rng.split(rng.PRNGKey(0), 3)
    _, bstate = init(k_fetch)
    batch, mask = get_batch(0, bstate)
    svi = impl.svi.DPSVI(ex.model, ex.guide, optimizers.Adam(1e-3), Trace_ELBO(), dp_scale=1.0, clipping_threshold=cfg["C"],
                         num_obs_total=rows, rng_suite=rng)
    state = svi.init(k_init, *batch)

    @jax.jit
    def step(i, state):
        b, m = get_batch(i, bstate)
        state, loss = svi.update(state, *b, mask=m)
        return state, loss, jnp.sum(m)

    n = 0
    for i in range(warmup):
        state, loss, _ = step(i, state)
    jax.block_until_ready(state)
    t0 = time.perf_counter()
    counts = []
    for i in range(steps):
        state, loss, c = step(warmup + i, state)
        counts.append(c)
    jax.block_until_ready((state, counts))
    dt = time.perf_counter() - t0
    n = int(sum(int(c) for c in counts))
    return {"value": n / dt, "ms_per_step": dt / steps * 1e3, "examples_per_step": n / steps,
            "max_batch_size": int(mask.shape[0]), "versions": impl.versions}


if __name__ == "__main__":
    ok, why = available()
    print("reference available:", ok, "-", why)
    if ok and len(sys.argv) > 1:
        print("\n".join(dump_golden(sys.argv[1])))
