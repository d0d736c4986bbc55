"""Oracle: the other ``numpyro.optim`` optimizers and the step-size schedules (numpy float32).  TEST INFRASTRUCTURE ONLY.

Restates ``jax.example_libraries.optimizers`` (momentum, adagrad, rmsprop, rmsprop_momentum and the schedules
constant / exponential_decay / inverse_time_decay / polynomial_decay / piecewise_constant) and numpyro's ClippedAdam,
which numpyro.optim wraps with the step counter ``i`` starting at 0 [3P-unverified: restated from published source,
jax and numpyro are not importable here].  Same interface as ``oracle.svi.SGD`` / ``Adam`` (state ``(i, ...)``,
``init`` / ``get_params`` / ``update``), so any of them plugs into ``oracle.svi.DPSVI``.  ``SGD`` and ``Adam`` here are
``oracle.svi``'s with a schedule for ``step_size``.
"""
import numpy as np

from . import svi as _svi

f32 = np.float32


# ---- schedules: i -> float32 step size ------------------------------------------------------------------------------
def constant(step_size):
    return lambda i: f32(step_size)


def exponential_decay(step_size, decay_steps, decay_rate):
    return lambda i: f32(f32(step_size) * np.power(f32(decay_rate), f32(i) / f32(decay_steps), dtype=f32))


def inverse_time_decay(step_size, decay_steps, decay_rate, staircase=False):
    if staircase:
        return lambda i: f32(f32(step_size) / (f32(1) + f32(decay_rate) * np.floor(f32(i) / f32(decay_steps))))
    return lambda i: f32(f32(step_size) / (f32(1) + f32(decay_rate) * f32(i) / f32(decay_steps)))


def polynomial_decay(step_size, decay_steps, final_step_size, power=1.0):
    def schedule(i):
        n = np.minimum(f32(i), f32(decay_steps))
        mult = np.power(f32(1) - n / f32(decay_steps), f32(power), dtype=f32)
        return f32(mult * (f32(step_size) - f32(final_step_size)) + f32(final_step_size))
    return schedule


def piecewise_constant(boundaries, values):
    boundaries, values = np.asarray(boundaries), np.asarray(values, f32)
    if not boundaries.ndim == values.ndim == 1 or values.shape[0] != boundaries.shape[0] + 1:
        raise ValueError("piecewise_constant needs len(values) == len(boundaries) + 1")
    return lambda i: f32(values[int(np.sum(i > boundaries))])


def make_schedule(step_size):
    return step_size if callable(step_size) else constant(step_size)


# ---- optimizers -----------------------------------------------------------------------------------------------------
def _f(a):
    return np.asarray(a, f32)


class _Optim:
    n_state = 0          # per-parameter state arrays besides x

    def init(self, params):
        x = {k: _f(v).copy() for k, v in params.items()}
        return 0, (x,) + tuple({k: np.zeros_like(v) for k, v in x.items()} for _ in range(self.n_state))

    def get_params(self, state):
        return state[1][0]

    def update(self, g, state):
        i, st = state
        lr = f32(self.step_size(i))
        out = [dict() for _ in st]
        for k in st[0]:
            new = self.element(lr, _f(g[k]), *(s[k] for s in st))
            for o, n in zip(out, new):
                o[k] = _f(n)
        return i + 1, tuple(out)


class Momentum(_Optim):
    n_state = 1

    def __init__(self, step_size, mass):
        self.step_size, self.mass = make_schedule(step_size), f32(mass)

    def element(self, lr, g, x, m):
        m = _f(self.mass * m + g)
        return x - lr * m, m


class Adagrad(_Optim):
    n_state = 2          # (g_sq, m)

    def __init__(self, step_size, momentum=0.9):
        self.step_size, self.momentum = make_schedule(step_size), f32(momentum)

    def element(self, lr, g, x, g_sq, m):
        g_sq = _f(g_sq + np.square(g))
        with np.errstate(divide="ignore"):
            inv = np.where(g_sq > 0, f32(1) / np.sqrt(g_sq), f32(0)).astype(f32)
        m = _f((f32(1) - self.momentum) * (g * inv) + self.momentum * m)
        return x - lr * m, g_sq, m


class RMSProp(_Optim):
    n_state = 1          # avg_sq_grad

    def __init__(self, step_size, gamma=0.9, eps=1e-8):
        self.step_size, self.gamma, self.eps = make_schedule(step_size), f32(gamma), f32(eps)

    def element(self, lr, g, x, avg_sq):
        avg_sq = _f(avg_sq * self.gamma + np.square(g) * (f32(1) - self.gamma))
        return x - lr * g / np.sqrt(avg_sq + self.eps), avg_sq


class RMSPropMomentum(_Optim):
    n_state = 2          # (avg_sq_grad, mom)

    def __init__(self, step_size, gamma=0.9, eps=1e-8, momentum=0.9):
        self.step_size, self.gamma, self.eps = make_schedule(step_size), f32(gamma), f32(eps)
        self.momentum = f32(momentum)

    def element(self, lr, g, x, avg_sq, mom):
        avg_sq = _f(avg_sq * self.gamma + np.square(g) * (f32(1) - self.gamma))
        mom = _f(self.momentum * mom + lr * g / np.sqrt(avg_sq + self.eps))
        return x - mom, avg_sq, mom


class ClippedAdam(_Optim):
    n_state = 2          # (m, v)

    def __init__(self, step_size, b1=0.9, b2=0.999, eps=1e-8, clip_norm=10.0):
        self.step_size = make_schedule(step_size)
        self.b1, self.b2, self.eps, self.clip_norm = f32(b1), f32(b2), f32(eps), f32(clip_norm)

    def update(self, g, state):
        self._i = state[0]
        return super().update(g, state)

    def element(self, lr, g, x, m, v):
        g = np.clip(g, -self.clip_norm, self.clip_norm)
        one, t = f32(1), f32(self._i + 1)
        m = _f((one - self.b1) * g + self.b1 * m)
        v = _f((one - self.b2) * np.square(g) + self.b2 * v)
        mhat = m / (one - np.power(self.b1, t, dtype=f32))
        vhat = v / (one - np.power(self.b2, t, dtype=f32))
        return x - lr * mhat / (np.sqrt(vhat) + self.eps), m, v


class SGD(_svi.SGD):
    def __init__(self, step_size):
        super().__init__(0.0)
        self.schedule = make_schedule(step_size)

    def update(self, g, state):
        self.step_size = f32(self.schedule(state[0]))
        return super().update(g, state)


class Adam(_svi.Adam):
    def __init__(self, step_size, b1=0.9, b2=0.999, eps=1e-8):
        super().__init__(0.0, b1, b2, eps)
        self.schedule = make_schedule(step_size)

    def update(self, g, state):
        self.step_size = f32(self.schedule(state[0]))
        return super().update(g, state)
