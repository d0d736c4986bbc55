"""``numpyro.optim`` SGD / Adam / Momentum / Adagrad / RMSProp / RMSPropMomentum / ClippedAdam as used by
``DPSVI._apply_gradient`` (``d3p/svi.py:379-393``; Adam(b1=.9, b2=.999, eps=1e-8) in every example, e.g.
``examples/logistic_regression.py:141``), the step-size schedules of ``jax.example_libraries.optimizers``, and
``d3p.optimizers.ADADP`` (``d3p/optimizers.py:29-131``).

The optimizer state is ``OptimState(step, flat, m, v, layout)``: one flat float32 CUDA vector of
unconstrained parameters in pytree order plus the optimizer's per-parameter state (``m``: first moment / velocity /
momentum, ``v``: squared-gradient accumulator; ``None`` when the optimizer keeps none).  The update itself runs
inside the finalize kernel of libd3p_b200 (``d3p_perturb_finalize_f32``), fused with noise and rescaling.

``step_size`` is a number, one of the schedules below, or any callable ``i -> float`` of the optimizer's own step
counter ``i`` (``OptimState.step``, from 0).  The named schedules are evaluated by the library
(``d3p_optim_step_size``) once per step, also inside the fused epoch drivers; any other callable is evaluated here
before each step, so ``DPSVI.run_epoch`` takes its step-by-step path for it (same result, interpreter between steps).
"""
import ctypes as C
from typing import Any, NamedTuple, Optional

import numpy as np
import torch

from . import _native as _n


class OptimState(NamedTuple):
    step: int
    flat: torch.Tensor
    m: Optional[torch.Tensor]
    v: Optional[torch.Tensor]
    layout: Any   # [(name, offset, shape)]
    lr: Optional[torch.Tensor] = None   # ADADP: adaptive step size (0-dim CUDA tensor); m = x_stepped, v = x_prev


def _flatten(params, layout, device):
    n = layout[-1][1] + (int(np.prod(layout[-1][2])) if len(layout[-1][2]) else 1)
    flat = torch.empty(n, dtype=torch.float32, device=device)
    for name, off, shape in layout:
        size = int(np.prod(shape)) if len(shape) else 1
        flat[off:off + size] = torch.as_tensor(np.asarray(params[name].cpu() if isinstance(params[name], torch.Tensor)
                                                          else params[name], dtype=np.float32)).reshape(-1).to(device)
    return flat


def layout_of(params):
    out, off = [], 0
    for name in sorted(params):
        shape = tuple(params[name].shape)
        out.append((name, off, shape))
        off += int(np.prod(shape)) if len(shape) else 1
    return out


def unflatten(flat, layout):
    out = {}
    for name, off, shape in layout:
        size = int(np.prod(shape)) if len(shape) else 1
        out[name] = flat[off:off + size].reshape(shape)
    return out


class Schedule:
    """A step-size schedule of ``jax.example_libraries.optimizers``: callable ``i -> step size`` (float32), which also
    carries its parameters so that the library evaluates it inside the fused paths.  Made by the constructors below."""

    def __init__(self, kind, step_size=0.0, **params):
        self.kind, self.step_size, self.params = kind, float(step_size), params

    def fill(self, od):
        """Writes the schedule into an ``OptimDesc`` (its ``step_size`` field and the appended schedule fields)."""
        od.schedule, od.step_size = self.kind, self.step_size
        for name, val in self.params.items():
            if name in ("boundaries", "values"):
                od.n_boundaries = len(self.params["boundaries"])
                getattr(od, name)[:len(val)] = [float(x) for x in val]
            else:
                setattr(od, name, val)

    def __call__(self, i):
        od = _n.OptimDesc(_n.OPT_SGD | _n.OPT_SCHEDULED)
        self.fill(od)
        out = C.c_float()
        _n.check(_n.lib().d3p_optim_step_size(C.byref(od), int(i), C.byref(out)), "step-size schedule")
        return out.value

    def __repr__(self):
        names = {_n.SCHED_CONSTANT: "constant", _n.SCHED_EXPONENTIAL: "exponential_decay",
                 _n.SCHED_INVERSE_TIME: "inverse_time_decay", _n.SCHED_POLYNOMIAL: "polynomial_decay",
                 _n.SCHED_PIECEWISE: "piecewise_constant"}
        return f"{names[self.kind]}(step_size={self.step_size}, {self.params})"


def constant(step_size):
    return Schedule(_n.SCHED_CONSTANT, step_size)


def exponential_decay(step_size, decay_steps, decay_rate):
    """``step_size * decay_rate ** (i / decay_steps)``."""
    return Schedule(_n.SCHED_EXPONENTIAL, step_size, decay_steps=float(decay_steps), decay_rate=float(decay_rate))


def inverse_time_decay(step_size, decay_steps, decay_rate, staircase=False):
    """``step_size / (1 + decay_rate * i / decay_steps)``; with ``staircase``, ``i / decay_steps`` is floored."""
    return Schedule(_n.SCHED_INVERSE_TIME, step_size, decay_steps=float(decay_steps), decay_rate=float(decay_rate),
                    staircase=int(bool(staircase)))


def polynomial_decay(step_size, decay_steps, final_step_size, power=1.0):
    """``(1 - n / decay_steps) ** power * (step_size - final_step_size) + final_step_size``, n = min(i, decay_steps)."""
    return Schedule(_n.SCHED_POLYNOMIAL, step_size, decay_steps=float(decay_steps),
                    final_step_size=float(final_step_size), power=float(power))


def piecewise_constant(boundaries, values):
    """``values[number of boundaries b with i > b]``."""
    boundaries, values = [float(b) for b in boundaries], [float(v) for v in values]
    if len(values) != len(boundaries) + 1:
        raise ValueError("piecewise_constant needs len(values) == len(boundaries) + 1")
    if len(boundaries) > _n.MAX_BOUNDARIES:
        raise ValueError(f"piecewise_constant takes at most {_n.MAX_BOUNDARIES} boundaries")
    return Schedule(_n.SCHED_PIECEWISE, values[0], boundaries=boundaries, values=values)


def _step_size_arg(step_size):
    return step_size if callable(step_size) else float(step_size)


class _Optim:
    kind = _n.OPT_NONE
    uses_m = uses_v = False       # which of OptimState.m / .v the update keeps

    @property
    def fused_epoch(self):
        """False when the step size is a Python callable that only this process can evaluate."""
        ss = getattr(self, "step_size", None)
        return not callable(ss) or isinstance(ss, Schedule)

    def _desc(self, step, **fields):
        """``OptimDesc`` of this optimizer at optimizer step ``step``: the schedule travels with it (named schedules)
        or is evaluated here (any other callable)."""
        od = _n.OptimDesc(self.kind)
        ss = self.step_size
        if isinstance(ss, Schedule):
            ss.fill(od)
            od.kind = self.kind | _n.OPT_SCHEDULED
        elif callable(ss):
            od.step_size = float(ss(int(step)))
        else:
            od.step_size = ss
        od.step = int(step)
        for name, val in fields.items():
            setattr(od, name, val)
        return od

    def init(self, params, layout=None) -> OptimState:
        dev = torch.device("cuda", torch.cuda.current_device())
        layout = layout or layout_of(params)
        flat = _flatten(params, layout, dev)
        m = torch.zeros_like(flat) if self.uses_m else None
        v = torch.zeros_like(flat) if self.uses_v else None
        lr = None
        if self.kind == _n.OPT_ADADP:          # optimizers.py:54-57: (x0, lr, zeros, x0)
            v = flat.clone()
            lr = torch.full((), self.step_size, dtype=torch.float32, device=dev)
        return OptimState(0, flat, m, v, layout, lr)

    def get_params(self, state: OptimState):
        return unflatten(state.flat, state.layout)

    def desc(self, step, lr=None, n_params=0) -> _n.OptimDesc:
        raise NotImplementedError

    def finish(self, od, flat, x_prev):
        """Second launch of a step, if the optimizer needs one (ADADP odd steps)."""

    def update(self, grads, state: OptimState) -> OptimState:
        """Functional update (a new state is returned, like numpyro's)."""
        dev = state.flat.device
        g = _flatten(grads, state.layout, dev) if isinstance(grads, dict) else grads.reshape(-1)
        P = g.numel()
        part = torch.zeros(P + 2, dtype=torch.float32, device=dev)
        part[:P] = g
        flat = state.flat.clone()
        m = state.m.clone() if state.m is not None else None
        v = state.v.clone() if state.v is not None else None
        lr = state.lr.clone() if state.lr is not None else None
        nf = (C.c_float * 2)(1.0, 1.0)
        od = self.desc(state.step, lr, P)
        _n.check(_n.lib().d3p_perturb_finalize_f32(_n.ptr(part), 1, P, 1, None, 0.0, 1.0, 1.0, 0, None, C.byref(od),
                                                   _n.ptr(flat), _n.ptr(m), _n.ptr(v), None, nf, _n.stream_ptr()),
                 "optimizer update")
        self.finish(od, flat, v)
        return OptimState(state.step + 1, flat, m, v, state.layout, lr)


class SGD(_Optim):
    kind = _n.OPT_SGD

    def __init__(self, step_size):
        self.step_size = _step_size_arg(step_size)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step)


class Adam(_Optim):
    kind = _n.OPT_ADAM
    uses_m = uses_v = True

    def __init__(self, step_size, b1=0.9, b2=0.999, eps=1e-8):
        self.step_size, self.b1, self.b2, self.eps = _step_size_arg(step_size), float(b1), float(b2), float(eps)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step, b1=self.b1, b2=self.b2, eps=self.eps)


class ClippedAdam(Adam):
    """``numpyro.optim.ClippedAdam``: Adam on the gradient clipped element-wise to ``[-clip_norm, clip_norm]``."""
    kind = _n.OPT_CLIPPED_ADAM

    def __init__(self, step_size, b1=0.9, b2=0.999, eps=1e-8, clip_norm=10.0):
        super().__init__(step_size, b1, b2, eps)
        self.clip_norm = float(clip_norm)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step, b1=self.b1, b2=self.b2, eps=self.eps, clip_norm=self.clip_norm)


class Momentum(_Optim):
    """``numpyro.optim.Momentum``: ``m = mass * m + g; x -= lr * m``."""
    kind = _n.OPT_MOMENTUM
    uses_m = True

    def __init__(self, step_size, mass):
        self.step_size, self.mass = _step_size_arg(step_size), float(mass)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step, momentum=self.mass)


class Adagrad(_Optim):
    """``numpyro.optim.Adagrad``: ``v += g^2; m = (1 - momentum) * g / sqrt(v) + momentum * m; x -= lr * m`` (an
    element whose ``v`` is still 0 takes 0 for ``g / sqrt(v)``)."""
    kind = _n.OPT_ADAGRAD
    uses_m = uses_v = True

    def __init__(self, step_size, momentum=0.9):
        self.step_size, self.momentum = _step_size_arg(step_size), float(momentum)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step, momentum=self.momentum)


class RMSProp(_Optim):
    """``numpyro.optim.RMSProp``: ``v = gamma * v + (1 - gamma) * g^2; x -= lr * g / sqrt(v + eps)``."""
    kind = _n.OPT_RMSPROP
    uses_v = True

    def __init__(self, step_size, gamma=0.9, eps=1e-8):
        self.step_size, self.gamma, self.eps = _step_size_arg(step_size), float(gamma), float(eps)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step, gamma=self.gamma, eps=self.eps)


class RMSPropMomentum(_Optim):
    """``numpyro.optim.RMSPropMomentum``: ``v`` as RMSProp; ``m = momentum * m + lr * g / sqrt(v + eps); x -= m``."""
    kind = _n.OPT_RMSPROP_MOMENTUM
    uses_m = uses_v = True

    def __init__(self, step_size, gamma=0.9, eps=1e-8, momentum=0.9):
        self.step_size, self.gamma, self.eps = _step_size_arg(step_size), float(gamma), float(eps)
        self.momentum = float(momentum)

    def desc(self, step, lr=None, n_params=0):
        return self._desc(step, gamma=self.gamma, eps=self.eps, momentum=self.momentum)


class ADADP(_Optim):
    """``d3p.optimizers.ADADP`` (``d3p/optimizers.py:119-131``): Koskela & Honkela's step-size
    adaptation.  Two gradient steps form one ADADP iteration: the even one takes half a step and
    remembers the full step, the odd one takes the second half step, compares both end points,
    adapts the step size and (``stability_check``) rejects the iteration if they disagree by more
    than ``tol``.  ``alpha_min`` / ``alpha_max`` are accepted and ignored, as in the reference
    (``:88-90`` hard-codes 0.9 / 1.1).  State: ``flat`` = x, ``m`` = x_stepped, ``v`` = x_prev,
    ``lr`` = step size (device scalar: nothing here synchronises with the host)."""
    kind = _n.OPT_ADADP
    uses_m = True             # x_stepped; v (x_prev) starts as a copy of x

    def __init__(self, step_size=1e-3, tol=1.0, stability_check=True, alpha_min=0.9, alpha_max=1.1):
        if callable(step_size):
            raise TypeError("ADADP adapts its own step size: step_size is its initial value, not a schedule")
        self.step_size, self.tol, self.stability_check = float(step_size), float(tol), bool(stability_check)
        self._ws = None

    def desc(self, step, lr=None, n_params=0):
        if lr is None:
            raise ValueError("ADADP needs the state's step-size tensor")
        self._ensure_ws(int(n_params), lr.device)
        return _n.OptimDesc(self.kind, self.step_size, 0.0, 0.0, 0.0, int(step), self.tol,
                            int(self.stability_check), lr.data_ptr(), self._ws.data_ptr())

    def _ensure_ws(self, P, device):
        need = int(_n.lib().d3p_adadp_workspace_floats(P))
        if self._ws is None or self._ws.device != device or self._ws.numel() < need:
            self._ws = torch.zeros(max(need, 1 << 12), dtype=torch.float32, device=device)

    def finish(self, od, flat, x_prev):
        if od.step & 1:
            _n.check(_n.lib().d3p_adadp_finish_f32(C.byref(od), flat.numel(), _n.ptr(flat), _n.ptr(x_prev),
                                                   _n.stream_ptr()), "ADADP finish")
