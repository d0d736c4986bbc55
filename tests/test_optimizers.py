"""CPU tests of the optimizers and step-size schedules: the oracle restatements against float64 hand computations, the
library's host-side schedule evaluation (d3p_optim_step_size) against the closed forms, the ctypes mirror of
d3p_optim_desc, and the descriptor checks that need no device."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from oracle import optim as oopt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from d3p_b200 import _build, _native
    _build.build()
    return _native.lib()


G = np.array([0.5, -2.0, 0.0, 3.0, -0.25], np.float32)        # includes a zero gradient element
G2 = np.array([-1.0, 0.75, 0.0, 12.0, 0.5], np.float32)
X0 = np.array([0.1, -0.3, 0.7, 1.5, -2.0], np.float32)


def _run(opt, grads):
    st = opt.init({"x": X0})
    for g in grads:
        st = opt.update({"x": g}, st)
    return st


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-6)))


def test_oracle_momentum():
    st = _run(oopt.Momentum(0.1, 0.9), [G, G2])
    m = G.astype(float)
    x = X0 - 0.1 * m
    m = 0.9 * m + G2
    x = x - 0.1 * m
    assert st[0] == 2 and _rel(st[1][0]["x"], x) < 1e-6 and _rel(st[1][1]["x"], m) < 1e-6


def test_oracle_adagrad_zero_gradient():
    st = _run(oopt.Adagrad(0.05, momentum=0.8), [G, G2])
    v = np.zeros(5)
    m = np.zeros(5)
    x = X0.astype(float)
    for g in (G, G2):
        v = v + g.astype(float) ** 2
        with np.errstate(divide="ignore"):
            r = np.where(v > 0, 1 / np.sqrt(v), 0.0)
        m = 0.2 * g * r + 0.8 * m
        x = x - 0.05 * m
    assert np.all(np.isfinite(st[1][0]["x"])) and st[1][0]["x"][2] == X0[2]      # element 2 never saw a gradient
    assert _rel(st[1][0]["x"], x) < 1e-6 and _rel(st[1][1]["x"], v) < 1e-6 and _rel(st[1][2]["x"], m) < 1e-6


def test_oracle_rmsprop_eps_inside_root():
    eps = 1e-2                                                          # large enough to tell inside from outside
    st = _run(oopt.RMSProp(0.01, gamma=0.5, eps=eps), [G])
    v = 0.5 * G.astype(float) ** 2
    x = X0 - 0.01 * G / np.sqrt(v + eps)
    assert _rel(st[1][0]["x"], x) < 1e-6 and _rel(st[1][1]["x"], v) < 1e-6
    assert _rel(X0 - 0.01 * G / (np.sqrt(v) + eps), x) > 1e-3


def test_oracle_rmsprop_momentum():
    st = _run(oopt.RMSPropMomentum(0.01, gamma=0.8, eps=1e-3, momentum=0.7), [G, G2])
    v, mom, x = np.zeros(5), np.zeros(5), X0.astype(float)
    for g in (G, G2):
        v = v * 0.8 + g.astype(float) ** 2 * 0.2
        mom = 0.7 * mom + 0.01 * g / np.sqrt(v + 1e-3)
        x = x - mom
    assert _rel(st[1][0]["x"], x) < 1e-6 and _rel(st[1][1]["x"], v) < 1e-6 and _rel(st[1][2]["x"], mom) < 1e-6


def test_oracle_clipped_adam_clips_before_the_moments():
    st = _run(oopt.ClippedAdam(1e-2, clip_norm=1.0), [G, G2])
    m, v, x = np.zeros(5), np.zeros(5), X0.astype(float)
    for t, g in enumerate((G, G2), 1):
        gc = np.clip(g.astype(float), -1, 1)
        m = 0.1 * gc + 0.9 * m
        v = 0.001 * gc ** 2 + 0.999 * v
        x = x - 1e-2 * (m / (1 - 0.9 ** t)) / (np.sqrt(v / (1 - 0.999 ** t)) + 1e-8)
    # 1 - b2 is 1.0000467e-3 in float32: v is 5e-5 off the float64 value by construction
    assert _rel(st[1][0]["x"], x) < 1e-5 and _rel(st[1][1]["x"], m) < 1e-6 and _rel(st[1][2]["x"], v) < 1e-4


def test_oracle_scheduled_sgd_and_adam():
    sched = oopt.exponential_decay(0.1, 2, 0.5)
    st = _run(oopt.SGD(sched), [G, G2])
    x = X0 - 0.1 * G.astype(float) - 0.1 * 0.5 ** 0.5 * G2
    assert _rel(st[1]["x"], x) < 1e-6
    st = _run(oopt.Adam(sched), [G])
    assert _rel(st[1][0]["x"], X0 - 0.1 * np.sign(G) * (np.abs(G) > 0)) < 1e-5


SCHEDULES = [
    ("constant", (0.3,), lambda i: 0.3, 10),
    ("exponential_decay", (0.1, 10, 0.5), lambda i: 0.1 * 0.5 ** (i / 10), 10),
    ("inverse_time_decay", (0.1, 10, 2.0), lambda i: 0.1 / (1 + 2.0 * i / 10), 10),
    ("inverse_time_decay", (0.1, 10, 2.0, True), lambda i: 0.1 / (1 + 2.0 * math.floor(i / 10)), 10),
    ("polynomial_decay", (0.1, 10, 0.01), lambda i: (1 - min(i, 10) / 10) * 0.09 + 0.01, 10),
    ("polynomial_decay", (0.1, 7, 0.01, 2.5), lambda i: (1 - min(i, 7) / 7) ** 2.5 * 0.09 + 0.01, 7),
    ("piecewise_constant", ([3, 10], [0.1, 0.05, 0.01]), lambda i: [0.1, 0.05, 0.01][(i > 3) + (i > 10)], 10),
]


def _points(ds):
    return [0, 1, ds - 1, ds, 10 * ds, 3, 4, 11]          # 3 and 10 are the piecewise boundaries


@pytest.mark.parametrize("name,args,closed,ds", SCHEDULES)
def test_oracle_schedules_closed_form(name, args, closed, ds):
    fn = getattr(oopt, name)(*args)
    for i in _points(ds):
        got = fn(i)
        assert isinstance(got, np.float32)
        assert abs(float(got) - closed(i)) <= 2e-7 * max(abs(closed(i)), 1e-3), (name, i)


@pytest.mark.parametrize("name,args,closed,ds", SCHEDULES)
def test_library_schedules_match_oracle(lib, name, args, closed, ds):
    from d3p_b200 import optimizers
    fn, ofn = getattr(optimizers, name)(*args), getattr(oopt, name)(*args)
    for i in _points(ds):
        # the same float32 operations; numpy's float32 power and the C library's powf round apart by up to 2 ulp
        assert abs(np.float32(fn(i)) - ofn(i)) <= 2 * np.spacing(ofn(i)), (name, i, fn(i), ofn(i))


def test_optim_desc_layout_matches_header(lib):
    from d3p_b200 import _native as _n
    text = open(os.path.join(ROOT, "include", "d3p_b200.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} d3p_optim_desc;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"(\w+)(?:\[[^\]]*\])?\s*[;,]", body)
    assert [f[0] for f in _n.OptimDesc._fields_] == names
    # offsets of a C compiler's layout, computed here from the header's types: 4-byte fields, two pointers at 32 / 40
    off = {f[0]: getattr(_n.OptimDesc, f[0]).offset for f in _n.OptimDesc._fields_}
    assert [off[k] for k in ("kind", "step_size", "b1", "b2", "eps", "step", "tol", "stability_check")] == \
        list(range(0, 32, 4))
    assert off["lr_d"] == 32 and off["err_ws_d"] == 40 and off["momentum"] == 48
    assert off["values"] == off["boundaries"] + 4 * _n.MAX_BOUNDARIES
    assert C.sizeof(_n.OptimDesc) == off["values"] + 4 * (_n.MAX_BOUNDARIES + 1) + 4     # padded to 8
    od = _n.OptimDesc(_n.OPT_ADAM, 1e-3, 0.9, 0.999, 1e-8, 7)             # the positional form older callers use
    assert (od.kind, od.step, od.momentum, od.schedule) == (_n.OPT_ADAM, 7, 0.0, 0)
    assert np.float32(od.step_size) == np.float32(1e-3) and np.float32(od.b2) == np.float32(0.999)


def test_optim_desc_layout_from_c(lib, tmp_path):
    """The offsets a C compiler gives d3p_optim_desc equal the ctypes ones."""
    import shutil
    import subprocess
    from d3p_b200 import _native as _n
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    names = [f[0] for f in _n.OptimDesc._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "d3p_b200.h"\nint main(void) {\n'
                   + "".join(f'  printf("%zu\\n", offsetof(d3p_optim_desc, {n}));\n' for n in names)
                   + '  printf("%zu\\n", sizeof(d3p_optim_desc));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    assert got == [getattr(_n.OptimDesc, n).offset for n in names] + [C.sizeof(_n.OptimDesc)]


def _step_size(lib, od, step=0):
    out = C.c_float()
    return lib.d3p_optim_step_size(C.byref(od), step, C.byref(out)), out.value


def test_step_size_refusals(lib):
    from d3p_b200 import _native as _n
    INVALID, UNSUPPORTED = -1, -3
    S = _n.OPT_SCHEDULED
    assert _step_size(lib, _n.OptimDesc(9, 0.1))[0] == UNSUPPORTED
    assert _step_size(lib, _n.OptimDesc(-1, 0.1))[0] == UNSUPPORTED
    assert _step_size(lib, _n.OptimDesc(_n.OPT_NONE | S, 0.1))[0] == INVALID
    assert _step_size(lib, _n.OptimDesc(_n.OPT_ADADP | S, 0.1))[0] == INVALID
    for ds in (0.0, -3.0, float("nan")):
        for sched in (_n.SCHED_EXPONENTIAL, _n.SCHED_INVERSE_TIME, _n.SCHED_POLYNOMIAL):
            od = _n.OptimDesc(_n.OPT_ADAM | S, 0.1)
            od.schedule, od.decay_steps, od.decay_rate = sched, ds, 0.5
            assert _step_size(lib, od)[0] == INVALID, (sched, ds)
    od = _n.OptimDesc(_n.OPT_SGD | S, 0.1)
    od.schedule, od.n_boundaries = _n.SCHED_PIECEWISE, _n.MAX_BOUNDARIES + 1
    assert _step_size(lib, od)[0] == INVALID
    od.schedule = 17
    assert _step_size(lib, od)[0] == UNSUPPORTED
    od.schedule = _n.SCHED_CONSTANT
    assert _step_size(lib, od, step=-1)[0] == INVALID
    for clip in (0.0, -1.0, float("nan")):
        od = _n.OptimDesc(_n.OPT_CLIPPED_ADAM, 0.1)
        od.clip_norm = clip
        assert _step_size(lib, od)[0] == INVALID, clip
    od.clip_norm = 2.0
    assert _step_size(lib, od) == (0, pytest.approx(0.1))
    # an unscheduled old kind never has its appended fields read
    od = _n.OptimDesc(_n.OPT_SGD, 0.25)
    od.clip_norm, od.decay_steps, od.n_boundaries = -1.0, -1.0, 99
    assert _step_size(lib, od) == (0, 0.25)


def test_facade_step_sizes(lib):
    from d3p_b200 import _native as _n, optimizers as o
    with pytest.raises(TypeError):
        o.ADADP(lambda i: 0.1)
    with pytest.raises(ValueError):
        o.piecewise_constant([1, 2], [0.1])
    with pytest.raises(ValueError):
        o.piecewise_constant(list(range(17)), [0.1] * 18)
    sched = o.polynomial_decay(0.1, 10, 0.01)
    od = o.RMSPropMomentum(sched, gamma=0.8).desc(4)
    assert od.kind == _n.OPT_RMSPROP_MOMENTUM | _n.OPT_SCHEDULED and od.step == 4
    assert np.float32(od.gamma) == np.float32(0.8) and od.schedule == _n.SCHED_POLYNOMIAL
    assert _step_size(lib, od, 4)[1] == np.float32(sched(4))
    lam = o.Momentum(lambda i: 0.5 / (1 + i), 0.9)
    od = lam.desc(3)
    assert od.kind == _n.OPT_MOMENTUM and np.float32(od.step_size) == np.float32(0.125) and not lam.fused_epoch
    assert o.Adam(sched).fused_epoch and o.SGD(0.1).fused_epoch and o.ADADP().fused_epoch
    for cls, m, v in ((o.SGD, False, False), (o.Adam, True, True), (o.Momentum, True, False), (o.Adagrad, True, True),
                      (o.RMSProp, False, True), (o.RMSPropMomentum, True, True), (o.ClippedAdam, True, True)):
        assert (cls.uses_m, cls.uses_v) == (m, v), cls
