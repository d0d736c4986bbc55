"""Model / guide families with fused CUDA per-example-gradient kernels.

The reference takes arbitrary numpyro ``model`` / ``guide`` callables and differentiates them with
``vmap(value_and_grad)`` (``d3p/svi.py:271-300``).  This build has hand-written kernels for the
model families the reference's examples define; a family object plays the role of the
model/guide pair:

    fam = LogisticRegression(d=1024)                       # examples/logistic_regression.py:49-86
    svi = DPSVI(fam.model, fam.guide, Adam(1e-3), Trace_ELBO(), clipping_threshold=1.,
                dp_scale=1., num_obs_total=N)

Parameters are the *unconstrained* variational parameters, stored as one flat float32 vector
whose leaf order is the jax pytree order of the reference's param dict (sorted site names).
Arbitrary models go through the materialised-gradient stage methods of ``DPSVI``.
"""
import ctypes as C

import numpy as np
import torch

from . import _native as _n


class Trace_ELBO:
    """Stands in for ``numpyro.infer.Trace_ELBO`` in the ``per_example_loss`` slot of
    ``DPSVI(...)``: the fused kernels implement exactly the single-particle Trace_ELBO."""

    def __init__(self, num_particles=1):
        if num_particles != 1:
            raise ValueError("the fused kernels implement single-particle Trace_ELBO")
        self.num_particles = 1


def softplus_inv(x):
    return float(np.log(np.expm1(x)))


class _Handle:
    def __init__(self, family, role):
        self.family, self.role = family, role

    def __repr__(self):
        return f"<{type(self.family).__name__}.{self.role}>"


class Family:
    """What ``DPSVI`` needs from a fused model/guide family.  A subclass supplies the calls of its entry points of the
    library (``_step_workspace_bytes`` / ``_step``, ``_evaluate``, ``_epoch_workspace_bytes`` / ``_epoch``)."""
    # DPSVI.run_epoch has a C driver with device keys / for a batch sharded over NVLink peers (else: step by step)
    epoch_device_keys = True
    epoch_sharded = True

    def layout(self):
        """[(name, offset, shape)] in pytree (sorted-name) order."""
        out, off = [], 0
        for name in sorted(self.param_shapes()):
            shape = self.param_shapes()[name]
            n = int(np.prod(shape)) if len(shape) else 1
            out.append((name, off, shape))
            off += n
        return out

    @property
    def n_params(self):
        name, off, shape = self.layout()[-1]
        return off + (int(np.prod(shape)) if len(shape) else 1)

    def offsets(self):
        return {name: off for name, off, _ in self.layout()}

    def constrain(self, name, value):
        return value

    def observation_scale(self, num_obs_total):
        """``get_observations_scale`` (d3p/svi.py:43-65) on a one-element batch: the plate scale N / 1."""
        return float(num_obs_total)

    def param_shapes(self):
        raise NotImplementedError

    def init_params(self):
        raise NotImplementedError

    def check_args(self, args):
        raise NotImplementedError

    def run_step(self, svi, state, tf_key, args, mask, pos_begin, pos_end, px_norms, px_grads, px_loss):
        """The fused per-example-gradient / clip / sum kernels of batch positions [pos_begin, pos_end)
        -> (partials tensor [n_partials, P + 2], n_partials, B, P)"""
        b = svi._resolve_args(args)
        desc = self.desc(svi._num_obs_total())
        n_part = C.c_uint32(0)
        need = self._step_workspace_bytes(desc, pos_end - pos_begin, n_part)
        ws = svi._workspace(need)
        mask_t, _ = svi._mask_arg(mask, b.B)
        x_p, y_p, m_p = _n.ptr(b.x), _n.ptr(b.y), _n.ptr(mask_t)
        if b.local_rows is not None:
            # minibatch.LocalRows: the tensors hold only rows [first, first + n) of the batch; shift the base
            # pointers so that the kernel's global position p addresses local row p - first
            first, n_local = b.local_rows
            if (first, first + n_local) != (pos_begin, pos_end):
                raise ValueError(f"LocalRows [{first}, {first + n_local}) is not this rank's position range "
                                 f"[{pos_begin}, {pos_end})")
            x_p = C.c_void_p(b.x.data_ptr() - first * b.stride * 4)
            y_p = C.c_void_p(b.y.data_ptr() - first * 4) if b.y is not None else None
            if mask_t is not None:
                if mask_t.numel() != n_local:
                    raise ValueError("with LocalRows the mask must be the matching LocalRows slice")
                m_p = C.c_void_p(mask_t.data_ptr() - first)
        # the arguments idx_d .. C, which every family's step entry point takes in this order
        rows = (_n.ptr(b.idx), m_p, _n.ptr(b.num_valid), b.B, pos_begin, pos_end,
                tf_key.ctypes.data_as(C.POINTER(C.c_uint32)), float(state.observation_scale),
                float(svi._clipping_threshold))
        if svi.event_hook is not None:
            svi.event_hook("step_begin")
        self._step(desc, _n.ptr(state.optim_state.flat), x_p, b.stride, y_p, rows, px_norms, px_grads, px_loss, ws, need)
        if svi.event_hook is not None:
            svi.event_hook("step_end")
        return ws, n_part.value, b.B, desc.n_params

    def desc(self, num_obs_total):
        """The family's descriptor struct of the library."""
        raise NotImplementedError

    def _step_workspace_bytes(self, desc, rows, n_part):
        """Workspace of one step over ``rows`` batch rows; sets ``n_part`` (c_uint32) to the number of partial rows."""
        raise NotImplementedError

    def _step(self, desc, params, x, stride, y, rows, px_norms, px_grads, px_loss, ws, need):
        """The family's ``d3p_dpsvi_step_*`` call (``y``: labels, read by the families that have them)."""
        raise NotImplementedError

    def _evaluate(self, svi, desc, params, b, key, loss):
        """``DPSVI.evaluate`` of the ``ResolvedBatch`` b with the Threefry key ``key`` into the device scalar ``loss``."""
        raise NotImplementedError(f"DPSVI.evaluate: unknown family {type(self).__name__}")

    def _epoch_workspace_bytes(self, desc, sampler, world):
        raise NotImplementedError

    def _epoch(self, device_keys, desc, sampler, x, stride, y, batch_key, rng_key, rest):
        """One ``d3p_dpsvi_run_epoch_*`` call; ``rest`` = the arguments from ``first_step`` on."""
        raise NotImplementedError


class MeanFieldFamily(Family):
    """Mean-field Normal guide over the latents of an elementwise likelihood."""
    family_id = None

    def __init__(self, d, guide="hand", init_scale=0.1):
        if guide not in ("hand", "auto"):
            raise ValueError("guide must be 'hand' (examples' exp-link guide) or 'auto' (AutoDiagonalNormal)")
        self.d, self.guide_kind, self.init_scale = int(d), guide, float(init_scale)
        self.model, self.guide = _Handle(self, "model"), _Handle(self, "guide")

    def init_params(self):
        """Unconstrained initial values (zeros for the hand guides; loc 0 / scale ``init_scale``
        for the auto guide — numpyro draws auto_loc with init_to_uniform, pass your own via
        ``DPSVI.init(..., params=...)`` to reproduce a specific start)."""
        p = {}
        for name, shape in self.param_shapes().items():
            v = np.zeros(shape, np.float32)
            if name == "auto_scale":
                v = np.full(shape, softplus_inv(self.init_scale), np.float32)
            p[name] = v
        return p

    def constrain(self, name, value):
        if name == "auto_scale":
            return torch.nn.functional.softplus(value)
        return value

    def _step_workspace_bytes(self, desc, rows, n_part):
        return _n.lib().d3p_meanfield_workspace_bytes(C.byref(desc), C.byref(n_part))

    def _step(self, desc, params, x, stride, y, rows, px_norms, px_grads, px_loss, ws, need):
        _n.check(_n.lib().d3p_dpsvi_step_meanfield(
            C.byref(desc), params, x, stride, y, *rows, _n.ptr(px_norms), _n.ptr(px_grads), _n.ptr(px_loss), _n.ptr(ws),
            need, _n.stream_ptr()), "dpsvi_step_meanfield")

    def _evaluate(self, svi, desc, params, b, key, loss):
        need = _n.lib().d3p_elbo_evaluate_workspace_bytes()
        ws = svi._workspace(need)
        _n.check(_n.lib().d3p_elbo_evaluate_meanfield(C.byref(desc), params, _n.ptr(b.x), b.stride, _n.ptr(b.y),
                                                      _n.ptr(b.idx), b.B, key, _n.ptr(loss), _n.ptr(ws), need,
                                                      _n.stream_ptr()), "elbo_evaluate")

    def _epoch_workspace_bytes(self, desc, sampler, world):
        return _n.lib().d3p_dpsvi_epoch_workspace_bytes(C.byref(desc), C.byref(sampler))

    def _epoch(self, device_keys, desc, sampler, x, stride, y, batch_key, rng_key, rest):
        lib = _n.lib()
        run = lib.d3p_dpsvi_run_epoch_meanfield_dk if device_keys else lib.d3p_dpsvi_run_epoch_meanfield
        _n.check(run(C.byref(desc), C.byref(sampler), x, stride, y, batch_key, rng_key, *rest),
                 "run_epoch_dk" if device_keys else "run_epoch")


class LogisticRegression(MeanFieldFamily):
    """``examples/logistic_regression.py:49-86``: w ~ N(0, I_d), intercept ~ N(0, 1),
    y ~ Bernoulli(logits = X w + intercept); ``update(state, X, y, mask=...)``."""
    family_id = _n.FAMILY_LOGREG

    def param_shapes(self):
        d = self.d
        if self.guide_kind == "auto":
            return {"auto_loc": (d + 1,), "auto_scale": (d + 1,)}
        return {"intercept_loc": (), "intercept_std_log": (), "w_loc": (d,), "w_std_log": (d,)}

    def desc(self, num_obs_total):
        o, d = self.offsets(), self.d
        m = _n.MeanfieldDesc()
        m.family, m.d, m.n_params = self.family_id, d, self.n_params
        m.num_obs_total, m.lik_scale = float(num_obs_total), 0.0
        if self.guide_kind == "auto":
            m.link, m.joint_site = _n.LINK_SOFTPLUS, 1
            m.loc_off, m.rho_off = o["auto_loc"], o["auto_scale"]
            m.b_loc_off, m.b_rho_off = o["auto_loc"] + d, o["auto_scale"] + d
        else:
            m.link, m.joint_site = _n.LINK_EXP, 0
            m.loc_off, m.rho_off = o["w_loc"], o["w_std_log"]
            m.b_loc_off, m.b_rho_off = o["intercept_loc"], o["intercept_std_log"]
        return m

    def check_args(self, args):
        if len(args) != 2:
            raise ValueError("LogisticRegression expects (batch_X, batch_y)")
        if len(args[0].shape) != 2 or args[0].shape[1] != self.d:
            raise ValueError(f"batch_X must have shape [B, {self.d}]")


class GaussianMean(MeanFieldFamily):
    """``examples/simple_gaussian_posterior.py:50-83``: mu ~ N(0, I_d), x ~ N(mu, lik_scale) per
    dimension (the example's ``x_var = .1`` is used as a *scale*); ``update(state, X)``."""
    family_id = _n.FAMILY_GAUSS

    def __init__(self, d, guide="hand", lik_scale=0.1, init_scale=0.1):
        super().__init__(d, guide, init_scale)
        self.lik_scale = float(lik_scale)

    def param_shapes(self):
        d = self.d
        if self.guide_kind == "auto":
            return {"auto_loc": (d,), "auto_scale": (d,)}
        return {"mu_loc": (d,), "mu_std_log": (d,)}

    def desc(self, num_obs_total):
        o = self.offsets()
        m = _n.MeanfieldDesc()
        m.family, m.d, m.n_params = self.family_id, self.d, self.n_params
        m.num_obs_total, m.lik_scale = float(num_obs_total), self.lik_scale
        m.b_loc_off = m.b_rho_off = 0
        if self.guide_kind == "auto":
            m.link, m.joint_site = _n.LINK_SOFTPLUS, 1
            m.loc_off, m.rho_off = o["auto_loc"], o["auto_scale"]
        else:
            m.link, m.joint_site = _n.LINK_EXP, 0
            m.loc_off, m.rho_off = o["mu_loc"], o["mu_std_log"]
        return m

    def check_args(self, args):
        if len(args) != 1:
            raise ValueError("GaussianMean expects (batch_X,)")
        if len(args[0].shape) != 2 or args[0].shape[1] != self.d:
            raise ValueError(f"batch_X must have shape [B, {self.d}]")


class VAE(Family):
    """``examples/vae.py:65-153``: encoder Dense(D->H) softplus -> {Dense(H->Z), exp(Dense(H->Z))},
    decoder Dense(Z->H) softplus -> Dense(H->D) sigmoid, z ~ N(0, I), x ~ Bernoulli(probs), model and
    guide wrapped in ``scale(1 / num_obs_total)`` (``vae.py:193-194``); ``update(state, batch)`` with
    ``batch`` of shape [B, ...] flattened to [B, D].

    Parameters carry the flat names of the stax pytrees under ``decoder$params`` / ``encoder$params``;
    their sorted order is the jax leaf order W4, b4, W5, b5, W1, b1, W2, b2, W3, b3.  The clipped
    sums of the two large layers run on tcgen05 tensor cores (3xTF32), see csrc/vae.cu.
    """
    NAMES = ("decoder$params.0.W", "decoder$params.0.b", "decoder$params.2.W", "decoder$params.2.b",
             "encoder$params.0.W", "encoder$params.0.b", "encoder$params.3.0.W", "encoder$params.3.0.b",
             "encoder$params.3.1.0.W", "encoder$params.3.1.0.b")

    def __init__(self, out_dim, hidden_dim, z_dim, scaled=True, init_seed=0, init_std=1e-2):
        self.out_dim, self.hidden_dim, self.z_dim = int(out_dim), int(hidden_dim), int(z_dim)
        self.scaled, self.init_seed, self.init_std = bool(scaled), int(init_seed), float(init_std)
        self.model, self.guide = _Handle(self, "model"), _Handle(self, "guide")
        self.profile_events = None   # optional (c_void_p * 2): events around the clipped-sum GEMMs (bench.py)

    def param_shapes(self):
        D, H, Z = self.out_dim, self.hidden_dim, self.z_dim
        return dict(zip(self.NAMES, [(Z, H), (H,), (H, D), (D,), (D, H), (H,), (H, Z), (Z,), (H, Z), (Z,)]))

    def init_params(self):
        """stax.Dense(W_init=randn(1e-2)) shaped values from a fixed numpy seed (initialisation is off
        the hot path; pass ``params=`` to ``DPSVI.init`` to start from specific values)."""
        rs = np.random.RandomState(self.init_seed)
        return {k: (rs.randn(*shp) * self.init_std).astype(np.float32) for k, shp in self.param_shapes().items()}

    def site_scale(self, num_obs_total):
        if not self.scaled:
            return float(num_obs_total)
        return float(np.float32((1.0 / num_obs_total) * num_obs_total))

    def observation_scale(self, num_obs_total):
        return self.site_scale(num_obs_total)

    def check_args(self, args):
        if len(args) != 1:
            raise ValueError("VAE expects (batch,)")
        shape = tuple(args[0].shape)
        if len(shape) < 2 or int(np.prod(shape[1:])) != self.out_dim:
            raise ValueError(f"batch must have shape [B, ...] with {self.out_dim} values per record")

    def desc(self, num_obs_total):
        o = self.offsets()
        d = _n.VaeDesc()
        d.out_dim, d.hidden_dim, d.z_dim, d.n_params = self.out_dim, self.hidden_dim, self.z_dim, self.n_params
        (d.off_w4, d.off_b4, d.off_w5, d.off_b5, d.off_w1, d.off_b1, d.off_w2, d.off_b2, d.off_w3,
         d.off_b3) = [o[k] for k in self.NAMES]
        d.site_scale = self.site_scale(num_obs_total)
        return d

    def _side_streams(self):
        """This family object's ``d3p_vae_ctx`` on the current device (caller-owned side streams: the four clipped-sum
        GEMMs of a step run concurrently on them); created on first use, released with the object."""
        dev = torch.cuda.current_device()
        ctxs = self.__dict__.setdefault("_ctx", {})
        if dev not in ctxs:
            h = C.c_void_p()
            _n.check(_n.lib().d3p_vae_ctx_create(C.byref(h)), "vae_ctx_create")
            ctxs[dev] = h
        return ctxs[dev]

    def close(self):
        """Release the side streams now (re-created on demand)."""
        ctxs = self.__dict__.get("_ctx", {})
        while ctxs:
            _, h = ctxs.popitem()
            try:
                _n.lib().d3p_vae_ctx_destroy(h)
            except Exception:
                pass

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _step_workspace_bytes(self, desc, rows, n_part):
        return _n.lib().d3p_vae_workspace_bytes(C.byref(desc), rows, C.byref(n_part))

    def _step(self, desc, params, x, stride, y, rows, px_norms, px_grads, px_loss, ws, need):
        if px_grads is not None:
            raise NotImplementedError("the VAE path never materialises [B, P] per-example gradients")
        _n.check(_n.lib().d3p_dpsvi_step_vae(
            C.byref(desc), params, x, stride, *rows, _n.ptr(px_norms), _n.ptr(px_loss), _n.ptr(ws), need,
            self.profile_events, self._side_streams(), _n.stream_ptr()), "dpsvi_step_vae")

    def _evaluate(self, svi, desc, params, b, key, loss):
        need = _n.lib().d3p_vae_workspace_bytes(C.byref(desc), b.B, None)
        ws = svi._workspace(need)
        _n.check(_n.lib().d3p_elbo_evaluate_vae(C.byref(desc), params, _n.ptr(b.x), b.stride, _n.ptr(b.idx), b.B, key,
                                                _n.ptr(loss), _n.ptr(ws), need, self._side_streams(), _n.stream_ptr()),
                 "elbo_evaluate_vae")

    def _epoch_workspace_bytes(self, desc, sampler, world):
        return _n.lib().d3p_dpsvi_epoch_vae_workspace_bytes(C.byref(desc), C.byref(sampler), world)

    def _epoch(self, device_keys, desc, sampler, x, stride, y, batch_key, rng_key, rest):
        lib = _n.lib()
        run = lib.d3p_dpsvi_run_epoch_vae_dk if device_keys else lib.d3p_dpsvi_run_epoch_vae
        _n.check(run(C.byref(desc), C.byref(sampler), x, stride, batch_key, rng_key, *rest),
                 "run_epoch_vae_dk" if device_keys else "run_epoch_vae")


class GaussianMixture(Family):
    """``examples/gaussian_mixture_model.py:51-85`` with the ``d3p.gmm.GaussianMixture`` likelihood
    (``d3p/gmm.py:71-86``): pis ~ Dir(1), mus ~ N(0, 10), sigs ~ InvGamma(1, 1); guide
    pis ~ Dir(exp(alpha_log)), mus ~ N(mus_loc, 1), sigs ~ InvGamma(1, 1), every site drawn per
    example; ``update(state, X)`` with X of shape [B, d] (the example's ``k`` positional argument is
    the constructor's ``K``)."""
    epoch_device_keys = False       # the mixture's epoch driver: host keys, one GPU
    epoch_sharded = False

    def __init__(self, K, d):
        self.K, self.d = int(K), int(d)
        self.model, self.guide = _Handle(self, "model"), _Handle(self, "guide")

    def param_shapes(self):
        return {"alpha_log": (self.K,), "mus_loc": (self.K, self.d)}

    def init_params(self):
        return {k: np.zeros(s, np.float32) for k, s in self.param_shapes().items()}

    def check_args(self, args):
        if len(args) != 1:
            raise ValueError("GaussianMixture expects (batch_X,)")
        if len(args[0].shape) != 2 or args[0].shape[1] != self.d:
            raise ValueError(f"batch_X must have shape [B, {self.d}]")

    def desc(self, num_obs_total):
        o = self.offsets()
        g = _n.GmmDesc()
        g.K, g.d, g.n_params = self.K, self.d, self.n_params
        g.alpha_off, g.mus_off = o["alpha_log"], o["mus_loc"]
        g.num_obs_total = float(num_obs_total)
        return g

    def _step_workspace_bytes(self, desc, rows, n_part):
        return _n.lib().d3p_gmm_workspace_bytes(C.byref(desc), C.byref(n_part))

    def _step(self, desc, params, x, stride, y, rows, px_norms, px_grads, px_loss, ws, need):
        _n.check(_n.lib().d3p_dpsvi_step_gmm(
            C.byref(desc), params, x, stride, *rows, _n.ptr(px_norms), _n.ptr(px_grads), _n.ptr(px_loss), _n.ptr(ws),
            need, _n.stream_ptr()), "dpsvi_step_gmm")

    def _evaluate(self, svi, desc, params, b, key, loss):
        need = _n.lib().d3p_elbo_evaluate_gmm_workspace_bytes(C.byref(desc))
        ws = svi._workspace(need)
        _n.check(_n.lib().d3p_elbo_evaluate_gmm(C.byref(desc), params, _n.ptr(b.x), b.stride, _n.ptr(b.idx), b.B, key,
                                                _n.ptr(loss), _n.ptr(ws), need, _n.stream_ptr()), "elbo_evaluate_gmm")

    def _epoch_workspace_bytes(self, desc, sampler, world):
        return _n.lib().d3p_dpsvi_epoch_gmm_workspace_bytes(C.byref(desc), C.byref(sampler))

    def _epoch(self, device_keys, desc, sampler, x, stride, y, batch_key, rng_key, rest):
        _n.check(_n.lib().d3p_dpsvi_run_epoch_gmm(C.byref(desc), C.byref(sampler), x, stride, batch_key, rng_key, *rest),
                 "run_epoch_gmm")
