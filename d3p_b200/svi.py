"""``d3p.svi`` on B200: ``DPSVI`` (init / update / evaluate + the five stage methods),
``DPSVIState``, ``full_norm``, ``normalize_gradient``, ``clip_gradient`` — same names, argument
meaning and error behaviour as ``d3p/svi.py`` — driving the CUDA kernels of libd3p_b200.

One ``update`` is two kernel launches for the fused model families (``d3p_b200.models``):
  1. ``d3p_dpsvi_step_meanfield``  per-example grad + norm + clip + clipped sum (svi.py:238-348)
  2. ``d3p_perturb_finalize_f32``  reduce + mean + ChaCha noise + rescale + optimizer (svi.py:327-393)
Key derivation (``rng_suite.split``, ``convert_to_jax_rng_key``) runs on the host inside the
library and is passed by value, so a step needs no device->host synchronisation.
"""
import ctypes as C
from typing import Any, NamedTuple, Sequence, Tuple

import numpy as np
import torch

from . import _native as _n
from . import random as strong_rng
from .minibatch import BatchView, LocalRows
from .models import Family
from .optimizers import OptimState, unflatten
from .util import example_count

PRNGState = Any


class DPSVIState(NamedTuple):
    optim_state: Any
    rng_key: PRNGState
    observation_scale: float


class ResolvedBatch(NamedTuple):
    """A batch as the step / evaluate / epoch kernels take it (``DPSVI._resolve_args``)."""
    x: torch.Tensor      # float32 rows on the device
    stride: int          # row stride of x in elements
    y: Any               # int32 labels read at the same rows as x, or None
    idx: Any             # int32 row indices of a BatchView into x, or None: row p of x is batch position p
    B: int               # batch size
    num_valid: Any       # device count of the real rows of a Poisson BatchView (the kernels skip the rest), or None
    local_rows: Any      # (first, n_local) of a LocalRows slice, or None


# ---- pytree helpers (dict leaves in sorted-key order, like jax) ----------------------------------
def tree_leaves(tree):
    if tree is None:
        return []
    if isinstance(tree, dict):
        return [l for k in sorted(tree) for l in tree_leaves(tree[k])]
    if isinstance(tree, (tuple, list)):
        return [l for t in tree for l in tree_leaves(t)]
    return [tree]


def tree_unflatten_like(tree, leaves):
    it = iter(leaves)

    def rec(t):
        if isinstance(t, dict):
            vals = {k: rec(t[k]) for k in sorted(t)}
            return {k: vals[k] for k in t}
        if isinstance(t, tuple):
            return tuple(rec(x) for x in t)
        if isinstance(t, list):
            return [rec(x) for x in t]
        return next(it)

    return rec(tree)


_CUDA_OK = False


def _dev():
    global _CUDA_OK
    if not _CUDA_OK:
        if not torch.cuda.is_available():
            raise _n.D3PNativeError("d3p_b200 needs a CUDA device (no CPU fallback)")
        _CUDA_OK = True
    return torch.device("cuda", torch.cuda.current_device())


def _as_dev_f32(x):
    if isinstance(x, torch.Tensor):
        return x.to(device=_dev(), dtype=torch.float32)
    return torch.as_tensor(np.asarray(x, dtype=np.float32)).to(_dev())


def _concat_rows(leaves, batched):
    """leaves -> ([B, P] float32 contiguous, sizes, shapes)."""
    ts = [_as_dev_f32(l) for l in leaves]
    if batched:
        B = ts[0].shape[0]
        flat = [t.reshape(B, -1) for t in ts]
    else:
        flat = [t.reshape(1, -1) for t in ts]
    sizes = [f.shape[1] for f in flat]
    return torch.cat(flat, dim=1).contiguous(), sizes, [tuple(t.shape) for t in ts]


def _aligned_scratch(ws, need):
    """The cached float32 scratch tensor ``ws`` if it holds ``need`` bytes on the device, else a new one; 256-byte
    aligned (the VAE kernels require it)."""
    if ws is None or ws.numel() * 4 < need or ws.device != _dev():
        buf = torch.empty((need + 256 + 3) // 4, dtype=torch.float32, device=_dev())
        ws = buf[((-buf.data_ptr()) % 256) // 4:]
    return ws


def _leaf_layout(layout):
    """A ``LeafTable`` with the offsets and lengths of the leaves of ``layout`` (site states zero)."""
    if len(layout) > _n.MAX_LEAVES:
        raise _n.D3PNativeError(f"more than {_n.MAX_LEAVES} parameter leaves are not supported")
    lt = _n.LeafTable()
    lt.n_leaves = len(layout)
    for l, (name, off, shape) in enumerate(layout):
        lt.leaf_off[l] = off
        lt.leaf_len[l] = int(np.prod(shape)) if len(shape) else 1
    return lt


def _split_rows(mat, sizes, shapes):
    out, o = [], 0
    for n, shp in zip(sizes, shapes):
        out.append(mat[:, o:o + n].reshape(shp))
        o += n
    return out


def full_norm(vector_parts, ord=2):
    """``d3p/svi.py:68-87``: norm of all leaves taken as one long vector (0. for an empty tree)."""
    parts = tree_leaves(vector_parts)
    if len(parts) == 0:
        return 0.
    mat, _, _ = _concat_rows(parts, batched=False)
    norms = torch.empty(1, dtype=torch.float32, device=mat.device)
    if ord != 2:
        _n.check(_n.lib().d3p_vector_norm_f32(_n.ptr(mat), mat.numel(), float(ord), _n.ptr(norms), _n.stream_ptr()),
                 "vector_norm")
        return norms[0]
    scratch = mat.clone()
    _n.check(_n.lib().d3p_clip_rows_f32(_n.ptr(scratch), 1, mat.shape[1], float("inf"), _n.ptr(norms),
                                        _n.stream_ptr()), "full_norm")
    return norms[0]


def normalize_gradient(gradient_parts, ord=2):
    """``d3p/svi.py:90-103``."""
    norm_inv = 1. / full_norm(gradient_parts, ord=ord)
    leaves = [_as_dev_f32(g) * norm_inv for g in tree_leaves(gradient_parts)]
    return tree_unflatten_like(gradient_parts, leaves)


def clip_gradient(gradient_parts, c):
    """``d3p/svi.py:106-124``: every leaf scaled by ``1 / max(1, norm / c)``."""
    if c == 0.:
        raise ValueError("The clipping threshold must be greater than 0.")
    parts = tree_leaves(gradient_parts)
    if len(parts) == 0:
        return gradient_parts
    mat, sizes, shapes = _concat_rows(parts, batched=False)
    _n.check(_n.lib().d3p_clip_rows_f32(_n.ptr(mat), 1, mat.shape[1], float(c), None, _n.stream_ptr()),
             "clip_gradient")
    return tree_unflatten_like(gradient_parts, _split_rows(mat, sizes, shapes))


class DPSVI:
    """Differentially-private SVI (``d3p/svi.py:127-498``).

    ``model`` / ``guide`` are the handles of a ``d3p_b200.models`` family (or ``None`` when only
    the stage methods are driven with caller-supplied per-example gradients, as the reference's
    own tests do).  ``optim`` is a ``d3p_b200.optimizers`` optimizer.

    ``donate_state`` (attribute, default False): when True, ``update`` reuses the buffers of the
    incoming state for the outgoing one (like jit donation); the incoming state must then not be
    used again.
    """

    def __init__(self, model, guide, optim, per_example_loss, clipping_threshold, dp_scale,
                 rng_suite=strong_rng, clip_unscaled_observations=True, **static_kwargs):
        self._clipping_threshold = clipping_threshold
        self._dp_scale = dp_scale
        self._rng_suite = rng_suite
        self._clip_unscaled_observations = clip_unscaled_observations
        if not np.isfinite(clipping_threshold):
            raise ValueError("clipping_threshold must be finite!")
        self.model, self.guide, self.optim, self.loss = model, guide, optim, per_example_loss
        self.static_kwargs = static_kwargs
        fam = getattr(model, "family", model)
        gfam = getattr(guide, "family", guide)
        if fam is not None and not isinstance(fam, Family):
            raise TypeError("model must be the .model handle of a d3p_b200.models family (or None)")
        if fam is not None and gfam is not None and gfam is not fam:
            raise ValueError("model and guide must belong to the same family object")
        self.family = fam
        self.donate_state = False
        self._ws = None
        self.shard = None   # (rank, world_size, reduce_fn | None) set by d3p_b200.parallel.shard_dpsvi
        self.peer_window = None   # parallel.PeerWindow when the sums meet over NVLink peer memory
        self.event_hook = None   # optional callable(tag) around the step kernel launch (bench instrumentation)

    # ---- state plumbing (svi.py:192-211) -----------------------------------------------------------
    @staticmethod
    def _update_state_rng(state, rng_key):
        return DPSVIState(state.optim_state, rng_key, state.observation_scale)

    @staticmethod
    def _update_state_optim_state(state, optim_state):
        return DPSVIState(optim_state, state.rng_key, state.observation_scale)

    def _split_rng_key(self, dp_svi_state, count=1):
        split_keys = self._rng_suite.split(dp_svi_state.rng_key, count + 1)
        return DPSVI._update_state_rng(dp_svi_state, split_keys[0]), split_keys[1:]

    def _num_obs_total(self):
        n = self.static_kwargs.get("num_obs_total", None)
        return 1.0 if n is None else float(n)     # plate(name, batch_size=1, 1) inside the vmap

    def init(self, rng_key, *args, params=None, **kwargs):
        """``d3p/svi.py:213-236``.  ``params`` optionally overrides the family's initial
        (unconstrained) parameter values."""
        if self.family is None:
            raise ValueError("DPSVI.init needs a model family")
        self.family.check_args(args)
        p = dict(self.family.init_params())
        if params is not None:
            p.update(params)
        optim_state = self.optim.init(p, layout=self.family.layout())
        observation_scale = 1.0
        if self._clip_unscaled_observations:
            # get_observations_scale on a one-element batch: plate scale = num_obs_total / 1 (times the
            # family's own scale handler, if any)
            observation_scale = self.family.observation_scale(self._num_obs_total())
        return DPSVIState(optim_state, rng_key, observation_scale)

    def get_params(self, state):
        """Constrained parameter dict (numpyro ``SVI.get_params``)."""
        raw = self.optim.get_params(state.optim_state)
        if self.family is None:
            return raw
        return {k: self.family.constrain(k, v) for k, v in raw.items()}

    # ---- fused path ------------------------------------------------------------------------------
    def _workspace(self, need):
        """A 256-byte aligned float32 view of at least ``need`` bytes into a cached scratch tensor."""
        if need == 0:
            raise _n.D3PNativeError("unsupported model family configuration")
        self._ws = _aligned_scratch(self._ws, need)
        return self._ws

    def _resolve_args(self, args):
        """-> ``ResolvedBatch`` of the batch arrays ``args``."""
        fam = self.family
        fam.check_args(args)
        X = args[0]
        idx = None
        # a Poisson BatchView knows how many of its slots are real: the kernels skip the padding slots even when the
        # caller does not pass mask= (the reference zero-fills those rows, d3p/minibatch.py:126-131)
        num_valid = X.num_valid if isinstance(X, BatchView) else None
        if isinstance(X, LocalRows):
            # rank-local slice of the batch: (first, n_local); the step kernel addresses rows by global
            # position, so the family shifts the base pointers back by `first` rows
            if any(not isinstance(a, LocalRows) or a.first != X.first or a.tensor.shape[0] != X.tensor.shape[0]
                   for a in args):
                raise ValueError("all batch arrays must be LocalRows of the same slice")
            B = X.batch_size
            Xsrc = X.tensor.to(device=_dev(), dtype=torch.float32)
            if Xsrc.dim() > 2:
                Xsrc = Xsrc.reshape(Xsrc.shape[0], -1)
            Xsrc = Xsrc.contiguous()
            ysrc = args[1].tensor.to(device=_dev(), dtype=torch.int32).contiguous() if len(args) > 1 else None
            return ResolvedBatch(Xsrc, int(Xsrc.stride(0)), ysrc, None, B, num_valid, (X.first, int(X.tensor.shape[0])))
        if isinstance(X, BatchView):
            idx, Xsrc = X.idx, X.source
            ysrc = None
            if len(args) > 1:
                Y = args[1]
                if isinstance(Y, BatchView) and Y.idx is idx:
                    ysrc = Y.source
                else:   # mixed: materialise everything
                    idx, Xsrc = None, X.tensor()
                    num_valid = None          # the gather zero-filled the padding rows
                    ysrc = Y.tensor() if isinstance(Y, BatchView) else Y
        else:
            Xsrc = X
            ysrc = None
            if len(args) > 1:
                ysrc = args[1].tensor() if isinstance(args[1], BatchView) else args[1]
        if not isinstance(Xsrc, torch.Tensor):
            Xsrc = torch.as_tensor(np.asarray(Xsrc))
        Xsrc = Xsrc.to(device=_dev(), dtype=torch.float32)
        if Xsrc.dim() > 2:                       # e.g. [N, 28, 28] images: one flat row per record
            Xsrc = Xsrc.reshape(Xsrc.shape[0], -1)
        if Xsrc.stride(-1) != 1:
            Xsrc = Xsrc.contiguous()
        B = example_count(X)
        if ysrc is not None:
            if not isinstance(ysrc, torch.Tensor):
                ysrc = torch.as_tensor(np.asarray(ysrc))
            ysrc = ysrc.to(device=_dev())
            if ysrc.dtype != torch.int32:
                ysrc = ysrc.to(torch.int32)
            ysrc = ysrc.contiguous()
            rows_needed = Xsrc.shape[0] if idx is not None else B       # labels are read at the same rows as X
            if ysrc.dim() == 0 or ysrc.shape[0] < rows_needed:
                raise ValueError(f"the label array has {0 if ysrc.dim() == 0 else ysrc.shape[0]} entries, "
                                 f"{rows_needed} are needed")
        if idx is None and Xsrc.shape[0] < B:
            raise ValueError(f"the batch array has {Xsrc.shape[0]} rows, {B} are needed")
        return ResolvedBatch(Xsrc, int(Xsrc.stride(0)), ysrc, idx, B, num_valid, None)

    @staticmethod
    def _mask_arg(mask, B):
        """-> (mask_uint8_tensor_or_None, all_masked)."""
        if isinstance(mask, (bool, np.bool_)):
            return (None, False) if mask else (torch.zeros(B, dtype=torch.uint8, device=_dev()), True)
        local = isinstance(mask, LocalRows)
        if local:
            mask = mask.tensor
        m = mask if isinstance(mask, torch.Tensor) else torch.as_tensor(np.asarray(mask))
        if not local and m.numel() != B:
            raise ValueError(f"mask has {m.numel()} entries for a batch of {B}")
        m = m.to(_dev())
        if m.dtype == torch.bool:
            m = m.view(torch.uint8)
        elif m.dtype != torch.uint8:
            m = (m != 0).view(torch.uint8)
        return m.contiguous(), False

    def _run_step(self, state, step_rng_key, args, mask, px_norms=None, px_grads=None, px_loss=None):
        """Launches the family's fused per-example-gradient / clip / sum kernels for this rank's batch
        positions; returns (partials tensor [n_partials, P + 2], n_partials, B, P)."""
        fam = self.family
        B = example_count(args[0])
        tf_key = np.ascontiguousarray(self._rng_suite.convert_to_jax_rng_key(step_rng_key), dtype=np.uint32)
        pos_begin, pos_end = 0, B
        if self.shard is not None:
            rank, world = self.shard[0], self.shard[1]
            per = (B + world - 1) // world
            pos_begin, pos_end = min(B, rank * per), min(B, (rank + 1) * per)
        return fam.run_step(self, state, tf_key, args, mask, pos_begin, pos_end, px_norms, px_grads, px_loss)

    def _leaf_table(self, layout, rng_key):
        """Per-leaf site keys: ``rng_suite.split(rng, n_leaves)`` (svi.py:490-491)."""
        lt = _leaf_layout(layout)
        site_keys = np.asarray(self._rng_suite.split(rng_key, len(layout)), dtype=np.uint32).reshape(len(layout), 16)
        for l in range(len(layout)):
            for i in range(16):
                lt.site_state[l][i] = int(site_keys[l, i])
        return lt

    def update(self, svi_state, *args, mask=True, **kwargs):
        """``d3p/svi.py:395-434``: one DP-SVI step; returns ``(new_state, loss)``.  ``loss`` is a
        0-dim CUDA tensor (asynchronous, like a jax array)."""
        return self._update_finalize(self._update_launch_step(svi_state, args, mask))

    def _update_launch_step(self, svi_state, args, mask):
        """First half of ``update``: key split + the fused per-example-gradient / clip / sum kernels of this rank's
        batch positions.  (Split out so that a test can drive several logical ranks on ONE device: all ranks' step
        kernels first, then all ranks' finalize kernels, which wait for each other.)"""
        if self.family is None:
            raise ValueError("DPSVI.update needs a model family; drive the stage methods for custom models")
        svi_state, (k_grad, k_noise) = self._split_rng_key(svi_state, 2)
        ws, n_part, B, P = self._run_step(svi_state, k_grad, args, mask)
        return svi_state, k_noise, ws, n_part, B, P

    def _update_finalize(self, ctx):
        """Second half of ``update``: reduce (+ exchange with the peers) + noise + rescale + optimizer."""
        svi_state, k_noise, ws, n_part, B, P = ctx
        os_ = svi_state.optim_state
        partials = ws
        comm = None
        if self.shard is not None:
            if self.shard[2] is not None:                       # NCCL backend: reduce kernel + all-reduce
                partials, n_part = self.shard[2](ws, n_part, P)
            else:                                               # sums meet inside the finalize kernel
                comm = self.peer_window.ptr
        if self.donate_state:
            new_flat, new_m, new_v = os_.flat, os_.m, os_.v
        else:
            new_flat = os_.flat.clone()
            new_m = os_.m.clone() if os_.m is not None else None
            new_v = os_.v.clone() if os_.v is not None else None
        new_lr = os_.lr if (self.donate_state or os_.lr is None) else os_.lr.clone()
        stats = torch.empty(3, dtype=torch.float32, device=new_flat.device)
        lt = self._leaf_table(os_.layout, k_noise)
        od = self.optim.desc(os_.step, new_lr, P)
        _n.check(_n.lib().d3p_perturb_finalize_p2p_f32(
            _n.ptr(partials), n_part, P, B, C.byref(lt), float(self._dp_scale), float(self._clipping_threshold),
            float(svi_state.observation_scale), 1, None, C.byref(od), _n.ptr(new_flat), _n.ptr(new_m), _n.ptr(new_v),
            _n.ptr(stats), None, comm, _n.stream_ptr()), "perturb_finalize")
        self.optim.finish(od, new_flat, new_v)
        new_os = OptimState(os_.step + 1, new_flat, new_m, new_v, os_.layout, new_lr)
        return DPSVIState(new_os, svi_state.rng_key, svi_state.observation_scale), stats[0]

    def _epoch_ctx(self, dev_index):
        """This object's ``d3p_epoch_ctx`` on the device (the epoch drivers' sampler stream, events and VAE side streams:
        caller-owned, created on first use, released with the object)."""
        ctxs = self.__dict__.setdefault("_epoch_ctxs", {})
        h = ctxs.get(dev_index)
        if h is None:
            h = C.c_void_p()
            _n.check(_n.lib().d3p_epoch_ctx_create(C.byref(h)), "epoch_ctx_create")
            ctxs[dev_index] = h
        return h

    def _release_epoch_ctxs(self):
        ctxs = self.__dict__.get("_epoch_ctxs", {})
        while ctxs:
            _, h = ctxs.popitem()
            try:
                _n.lib().d3p_epoch_ctx_destroy(h)
            except Exception:
                pass

    def close(self):
        """Release the native resources behind this object (the epoch drivers' streams and events, the family's side
        streams) now rather than when the garbage collector gets to them; everything is re-created on demand.  Not to
        be called while another DPSVI object sharing the family is in the middle of a call."""
        self._release_epoch_ctxs()
        self._epoch_plan = None
        fam = getattr(self, "family", None)
        if fam is not None and hasattr(fam, "close"):
            fam.close()

    def __del__(self):
        self._release_epoch_ctxs()      # only what this object alone owns: the family may be shared

    def run_epoch(self, svi_state, get_batch, batchifier_state, num_steps, first_step=0, device_keys=False):
        """The examples' ``lax.fori_loop(first_step, first_step + num_steps, body, state)`` with
        ``body = lambda i, s: update(s, *get_batch(i, batchifier_state))``
        (``examples/logistic_regression.py:149-160``): returns ``(new_state, stats)`` where
        ``stats[num_steps, 3]`` holds ``(loss, n, f)`` per step on the device.

        For the model families fed by ``poisson_batchify_data`` / ``subsample_batchify_data`` /
        ``split_batchify_data`` the whole loop runs inside the family's ``d3p_dpsvi_run_epoch_*`` driver (no
        interpreter between launches); the result is bit-identical to the step-by-step calls, which remain the path for
        everything else (NCCL-backend sharded runs, custom batchifiers, the key modes or sharded runs a family has
        no driver for: ``Family.epoch_device_keys`` / ``Family.epoch_sharded``, and an optimizer whose step size is a
        Python callable other than the named schedules of ``d3p_b200.optimizers``, which the C driver cannot call).
        Either way a schedule is evaluated at the optimizer's own step counter, not at ``first_step``.

        ``device_keys=True`` drives the ``*_dk`` entry points: the batchifier key and the state key are uploaded once
        and every per-step key is derived on the device (what a jitted caller with traced keys binds to, see
        INTEGRATION.md); the results are bit-identical.  This facade then reads the final state key back, which
        synchronises; a binding that keeps its keys on the device does not."""
        fam = self.family
        spec = getattr(get_batch, "spec", None)
        is_split = spec is not None and spec["kind"] == _n.SAMPLER_SPLIT
        fused = (spec is not None and fam is not None and (fam.epoch_device_keys or not device_keys)
                 and (self.shard is None or (fam.epoch_sharded and self.shard[2] is None))
                 and self._rng_suite is strong_rng and spec["rng_suite"] is strong_rng and self.event_hook is None
                 and getattr(self.optim, "fused_epoch", True) and num_steps > 0)
        if not fused:
            stats = torch.zeros(max(num_steps, 0), 3, dtype=torch.float32, device=_dev())
            for s in range(num_steps):
                out = get_batch(first_step + s, batchifier_state)
                batch, mask = out if (isinstance(out, tuple) and len(out) == 2 and isinstance(out[0], tuple)) else (out, True)
                svi_state, loss = self.update(svi_state, *batch, mask=mask)
                stats[s, 0] = loss
            return svi_state, stats
        dev = _dev()
        world = self.shard[1] if self.shard is not None else 1
        # everything about an epoch call that depends only on (batchifier, family, device) is worked out once
        plan_key = (id(spec), dev.index, world, self._num_obs_total())
        plan = getattr(self, "_epoch_plan", None)
        if plan is None or plan[0] != plan_key:
            data = self._resolve_args(spec["dataset"])
            desc = fam.desc(self._num_obs_total())
            sd = _n.SamplerDesc(spec["kind"], spec["q"], spec["n_records"], spec["batch"], 1 if spec["suppress"] else 0, None)
            probe = sd
            if is_split:        # the size query wants a non-null shuffle pointer; the real one is set per call
                probe = _n.SamplerDesc(spec["kind"], spec["q"], spec["n_records"], spec["batch"], 0, 256)
            need = fam._epoch_workspace_bytes(desc, probe, world)
            if need == 0:
                raise _n.D3PNativeError("unsupported family / sampler configuration for run_epoch")
            plan = (plan_key, spec, data.x, data.stride, data.y, desc, sd, need)      # keeps `spec` (and its id) alive
            self._epoch_plan = plan
        _, _, Xsrc, stride, ysrc, desc, sd, need = plan
        perm = None
        if is_split:        # split_batchify_data: the state IS the epoch's shuffled index list (no key)
            perm = torch.as_tensor(batchifier_state).to(device=dev, dtype=torch.int32).contiguous()
            if (first_step + num_steps) * spec["batch"] > perm.numel():
                raise ValueError("run_epoch: the split batchifier has only num_records // batch_size batches per epoch")
            sd = _n.SamplerDesc(spec["kind"], spec["q"], spec["n_records"], spec["batch"], 0, perm.data_ptr())
        self._epoch_ws = ws = _aligned_scratch(getattr(self, "_epoch_ws", None), need)
        if self.peer_window is not None and spec["kind"] == _n.SAMPLER_POISSON:
            self.peer_window = self.peer_window.with_records(spec["n_records"])   # sharded selector draw
        ectx = self._epoch_ctx(dev.index)
        os_ = svi_state.optim_state
        if self.donate_state:
            flat, m, v, lr = os_.flat, os_.m, os_.v, os_.lr
        else:
            flat = os_.flat.clone()
            m = os_.m.clone() if os_.m is not None else None
            v = os_.v.clone() if os_.v is not None else None
            lr = os_.lr.clone() if os_.lr is not None else None
        lt_c = getattr(self, "_epoch_lt", None)
        if lt_c is None or lt_c[0] is not os_.layout:
            self._epoch_lt = lt_c = (os_.layout, _leaf_layout(os_.layout))
        lt = lt_c[1]
        od = self.optim.desc(os_.step, lr, desc.n_params)
        stats = torch.empty(num_steps, 3, dtype=torch.float32, device=dev)
        bkey = (np.zeros(16, np.uint32) if is_split else
                np.ascontiguousarray(np.asarray(batchifier_state, dtype=np.uint32).reshape(16)))
        rkey = np.array(np.asarray(svi_state.rng_key, dtype=np.uint32).reshape(16), copy=True)
        comm = self.peer_window.ptr if self.shard is not None else None
        rest = (int(first_step), int(num_steps), float(svi_state.observation_scale), float(self._clipping_threshold),
                float(self._dp_scale), C.byref(lt), C.byref(od), _n.ptr(flat), _n.ptr(m), _n.ptr(v), _n.ptr(stats), comm,
                _n.ptr(ws), need, ectx, _n.stream_ptr())
        if device_keys:
            bkey_d = torch.as_tensor(bkey.view(np.int32)).to(dev)
            rkey_d = torch.as_tensor(rkey.view(np.int32)).to(dev)
            fam._epoch(True, desc, sd, _n.ptr(Xsrc), stride, _n.ptr(ysrc), _n.ptr(bkey_d), _n.ptr(rkey_d), rest)
            rkey = rkey_d.cpu().numpy().view(np.uint32).copy()
        else:
            u32p = C.POINTER(C.c_uint32)
            fam._epoch(False, desc, sd, _n.ptr(Xsrc), stride, _n.ptr(ysrc), bkey.ctypes.data_as(u32p),
                       rkey.ctypes.data_as(u32p), rest)
        new_os = OptimState(os_.step + num_steps, flat, m, v, os_.layout, lr)
        return DPSVIState(new_os, rkey.reshape(np.asarray(svi_state.rng_key).shape), svi_state.observation_scale), stats

    # ---- stage methods (the de-facto API of tests/test_dpsvi.py) --------------------------------
    def _compute_per_example_gradients(self, dp_svi_state, step_rng_key, *args, mask=True, **kwargs):
        """``d3p/svi.py:238-308``: materialises the per-example gradients ``[B, *shape]`` per site."""
        if self.family is None:
            raise ValueError("needs a model family")
        B = example_count(args[0])
        P = self.family.n_params
        dev = _dev()
        px_grads = torch.zeros((B, P), dtype=torch.float32, device=dev)
        px_loss = torch.zeros(B, dtype=torch.float32, device=dev)
        self._run_step(dp_svi_state, step_rng_key, args, mask, px_grads=px_grads, px_loss=px_loss)
        if isinstance(mask, (bool, np.bool_)):
            num_elements = B * bool(mask)
        else:
            num_elements = int(torch.as_tensor(mask).sum().item())
        f = 0. if num_elements == 0 else B / num_elements
        # kernel wrote obs_scale * loss_i; svi.py:306 multiplies by obs_scale * f
        px_loss = px_loss * f
        grads = {}
        for name, off, shape in self.family.layout():
            size = int(np.prod(shape)) if len(shape) else 1
            grads[name] = px_grads[:, off:off + size].reshape((B,) + tuple(shape))
        return dp_svi_state, px_loss, grads, num_elements, f

    def _clip_gradients(self, dp_svi_state, px_grads):
        """``d3p/svi.py:310-325``."""
        leaves = tree_leaves(px_grads)
        mat, sizes, shapes = _concat_rows(leaves, batched=True)
        if float(self._clipping_threshold) == 0.:
            raise ValueError("The clipping threshold must be greater than 0.")
        _n.check(_n.lib().d3p_clip_rows_f32(_n.ptr(mat), mat.shape[0], mat.shape[1], float(self._clipping_threshold),
                                            None, _n.stream_ptr()), "clip_rows")
        return dp_svi_state, tree_unflatten_like(px_grads, _split_rows(mat, sizes, shapes))

    def _combine_gradients(self, px_clipped_grads, px_loss):
        """``d3p/svi.py:327-348``: means over the (padded) batch axis."""
        leaves = tree_leaves(px_clipped_grads)
        mat, sizes, shapes = _concat_rows(leaves, batched=True)
        B, P = mat.shape
        loss = _as_dev_f32(px_loss).reshape(-1).contiguous()
        lib = _n.lib()
        need = lib.d3p_clip_and_sum_workspace_bytes(B, P)
        ws = torch.empty((need + 3) // 4 + 1, dtype=torch.float32, device=mat.device)
        sums = torch.empty(P + 2, dtype=torch.float32, device=mat.device)
        _n.check(lib.d3p_clip_and_sum_f32(_n.ptr(mat), _n.ptr(loss), None, B, P, float("inf"), _n.ptr(sums), _n.ptr(ws),
                                          need, _n.stream_ptr()), "clip_and_sum")
        avg = torch.empty(P, dtype=torch.float32, device=mat.device)
        stats = torch.empty(3, dtype=torch.float32, device=mat.device)
        nf = (C.c_float * 2)(float(B), 1.0)
        _n.check(lib.d3p_perturb_finalize_f32(_n.ptr(sums), 1, P, B, None, 0.0, 1.0, 1.0, 0, _n.ptr(avg), None, None,
                                              None, None, _n.ptr(stats), nf, _n.stream_ptr()), "combine")
        out_shapes = [s[1:] for s in shapes]
        return stats[0], tree_unflatten_like(px_clipped_grads, _split_rows(avg.reshape(1, -1), sizes, out_shapes))

    def _perturb_and_reassemble_gradients(self, dp_svi_state, step_rng_key, avg_clipped_grads, num_elements,
                                          batch_mask_scaling_factor):
        """``d3p/svi.py:350-377``."""
        leaves = tree_leaves(avg_clipped_grads)
        mat, sizes, shapes = _concat_rows(leaves, batched=False)
        P = mat.shape[1]
        part = torch.zeros(P + 2, dtype=torch.float32, device=mat.device)
        part[:P] = mat.reshape(-1)
        layout, off = [], 0
        for i, (n, shp) in enumerate(zip(sizes, shapes)):
            layout.append((str(i), off, (n,)))
            off += n
        lt = self._leaf_table(layout, step_rng_key)
        out = torch.empty(P, dtype=torch.float32, device=mat.device)
        n_val = float(num_elements.item()) if isinstance(num_elements, torch.Tensor) else float(num_elements)
        f_val = (float(batch_mask_scaling_factor.item()) if isinstance(batch_mask_scaling_factor, torch.Tensor)
                 else float(batch_mask_scaling_factor))
        nf = (C.c_float * 2)(n_val, f_val)
        _n.check(_n.lib().d3p_perturb_finalize_f32(
            _n.ptr(part), 1, P, 1, C.byref(lt), float(self._dp_scale), float(self._clipping_threshold),
            float(dp_svi_state.observation_scale), 1, _n.ptr(out), None, None, None, None, None, nf,
            _n.stream_ptr()), "perturb")
        return dp_svi_state, tree_unflatten_like(avg_clipped_grads, _split_rows(out.reshape(1, -1), sizes, shapes))

    def _apply_gradient(self, dp_svi_state, perturbed_grads):
        """``d3p/svi.py:379-393``."""
        new_optim_state = self.optim.update(perturbed_grads, dp_svi_state.optim_state)
        return self._update_state_optim_state(dp_svi_state, new_optim_state)

    @staticmethod
    def perturbation_function(rng_suite, rng, values, perturbation_scale):
        """``d3p/svi.py:470-498``: independent ``N(0, perturbation_scale^2)`` noise per leaf."""
        leaves = tree_leaves(values)
        per_site_rngs = rng_suite.split(rng, len(leaves))
        out = []
        for a, site_rng in zip(leaves, per_site_rngs):
            a = _as_dev_f32(a)
            out.append(a + rng_suite.normal(site_rng, tuple(a.shape)) * perturbation_scale)
        return tree_unflatten_like(values, out)

    def evaluate_epoch(self, svi_state, get_batch, batchifier_state, num_batches, first_batch=0):
        """The evaluation loops of the examples (``examples/logistic_regression.py:162-180``, ``vae.py:236-247``:
        ``fori_loop`` over ``test_fetch(i, state)`` -> ``svi.evaluate``), typically fed by ``split_batchify_data``:
        returns the ``num_batches`` losses as one device tensor.  Every ``evaluate`` is a few asynchronous launches
        and nothing here synchronises, so the loop runs at kernel speed without a C driver of its own."""
        out = torch.empty(max(num_batches, 0), dtype=torch.float32, device=_dev())
        for i in range(num_batches):
            b = get_batch(first_batch + i, batchifier_state)
            batch = b[0] if (isinstance(b, tuple) and len(b) == 2 and isinstance(b[0], tuple)) else b
            out[i] = self.evaluate(svi_state, *batch)
        return out

    def evaluate(self, svi_state, *args, **kwargs):
        """``d3p/svi.py:436-449``: non-private batch ELBO with one guide sample."""
        from .evaluate import evaluate_elbo
        key = self._rng_suite.convert_to_jax_rng_key(self._rng_suite.split(svi_state.rng_key, 1)[0])
        return evaluate_elbo(self, svi_state, key, args)

    # ---- privacy accounting passthrough (svi.py:451-468) -------------------------------------------
    def _validate_epochs_and_iter(self, num_epochs, num_iter, q):
        if num_epochs is not None:
            num_iter = num_epochs / q
        if num_iter is None:
            raise ValueError("A value must be supplied for either num_iter or num_epochs")
        return num_iter

    def get_epsilon(self, target_delta, q, num_epochs=None, num_iter=None):
        num_iter = self._validate_epochs_and_iter(num_epochs, num_iter, q)
        from .accountant import get_epsilon_R       # restatement of fourier_accountant (svi.py:31,461)
        return get_epsilon_R(target_delta, self._dp_scale, q, ncomp=num_iter)

    def get_delta(self, target_epsilon, q, num_epochs=None, num_iter=None):
        num_iter = self._validate_epochs_and_iter(num_epochs, num_iter, q)
        from .accountant import get_delta_R         # svi.py:32,467
        return get_delta_R(target_epsilon, self._dp_scale, q, ncomp=num_iter)
