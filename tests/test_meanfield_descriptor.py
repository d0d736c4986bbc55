"""The mean-field descriptor checks that the step and evaluate entry points share, and the softplus guide where
s' = sigmoid(rho) underflows to 0 on the d = 256 / 512 / 1024 step kernel."""
import ctypes as C

import numpy as np
import pytest

from oracle import chacha

D3P_ERR_INVALID_ARGUMENT, D3P_ERR_UNSUPPORTED = -1, -3
LOGREG, GAUSS, EXP, SOFTPLUS = 0, 1, 0, 1


@pytest.fixture(scope="module")
def lib():
    from d3p_b200 import _build, _native
    _build.build()
    return _native.lib()


def _desc(**kw):
    from d3p_b200._native import MeanfieldDesc
    f = dict(family=LOGREG, link=SOFTPLUS, joint_site=0, d=8, n_params=18, loc_off=0, rho_off=8, b_loc_off=16,
             b_rho_off=17, num_obs_total=100.0, lik_scale=1.0)
    f.update(kw)
    return MeanfieldDesc(**f)


def _evaluate(lib, desc, x_row_stride=8):
    key = np.zeros(2, np.uint32)
    ws = C.c_void_p(256)         # never dereferenced: every case is refused before a launch
    return lib.d3p_elbo_evaluate_meanfield(C.byref(desc), ws, ws, x_row_stride, ws, None, 4,
                                           key.ctypes.data_as(C.POINTER(C.c_uint32)), ws, ws, 1 << 20, None)


@pytest.mark.parametrize("bad", [dict(loc_off=11), dict(rho_off=12), dict(b_loc_off=18), dict(b_rho_off=18),
                                 dict(joint_site=1, n_params=17, rho_off=9), dict(link=2), dict(d=0)])
def test_evaluate_refuses_malformed_descriptors(lib, bad):
    assert _evaluate(lib, _desc(**bad)) == D3P_ERR_INVALID_ARGUMENT


def test_evaluate_refuses_short_rows(lib):
    assert _evaluate(lib, _desc(), x_row_stride=7) == D3P_ERR_INVALID_ARGUMENT
    assert _evaluate(lib, _desc(family=GAUSS, n_params=16), x_row_stride=7) == D3P_ERR_INVALID_ARGUMENT


def test_evaluate_refuses_unknown_family_as_unsupported(lib):
    assert _evaluate(lib, _desc(family=2)) == D3P_ERR_UNSUPPORTED


def _step(desc, params, X, stride, y, B, key, C_=1.0, obs_scale=100.0):
    """d3p_dpsvi_step_meanfield on the whole batch: (px_norms, px_grads, px_loss, partial rows)."""
    import torch
    from d3p_b200 import _native as _n
    lib = _n.lib()
    n_part = C.c_uint32(0)
    need = lib.d3p_meanfield_workspace_bytes(C.byref(desc), C.byref(n_part))
    ws = torch.zeros(need // 4, device="cuda")
    norms, loss = torch.full((B,), -7.0, device="cuda"), torch.full((B,), -7.0, device="cuda")
    grads = torch.full((B, desc.n_params), -7.0, device="cuda")
    kp = np.ascontiguousarray(key, np.uint32).ctypes.data_as(C.POINTER(C.c_uint32))
    _n.check(lib.d3p_dpsvi_step_meanfield(C.byref(desc), _n.ptr(params), _n.ptr(X), stride, _n.ptr(y), None, None, None,
                                          B, 0, B, kp, obs_scale, C_, _n.ptr(norms), _n.ptr(grads), _n.ptr(loss),
                                          _n.ptr(ws), need, _n.stream_ptr()), "step")
    torch.cuda.synchronize()
    parts = ws[:n_part.value * (desc.n_params + 2)].view(n_part.value, desc.n_params + 2)
    return [t.cpu().numpy() for t in (norms, grads, loss, parts)]


@pytest.mark.gpu
def test_softplus_step_where_sigmoid_underflows(cuda):
    """rho = -100 on a softplus guide: softplus(rho) is a denormal and sigmoid(rho) == 0, so s / s' must not be formed
    (theta = loc there).  The d = 256 kernel (rows of a 16-byte multiple) against the generic kernel (a row stride of
    257 floats), which the oracle tests pin, on the same inputs."""
    import torch
    from helpers.tolerance import assert_rel
    d, B = 256, 37
    desc = _desc(d=d, n_params=2 * d + 2, rho_off=d, b_loc_off=2 * d, b_rho_off=2 * d + 1, num_obs_total=10000.0)
    rs = np.random.RandomState(4)
    p = (rs.randn(2 * d + 2) * .3).astype(np.float32)
    p[d + 17] = -100.0
    X = rs.randn(B, d + 1).astype(np.float32)
    y = torch.as_tensor((rs.rand(B) < .5).astype(np.int32)).cuda()
    params = torch.as_tensor(p).cuda()
    Xv = torch.as_tensor(np.ascontiguousarray(X[:, :d])).cuda()
    Xg = torch.as_tensor(X).cuda()
    key = np.array([3, 9], np.uint32)
    got = _step(desc, params, Xv, d, y, B, key)
    ref = _step(desc, params, Xg, d + 1, y, B, key)
    for g in got:
        assert np.all(np.isfinite(g))
    for g, r, what in zip(got, ref, ["px_norms", "px_grads", "px_loss"]):
        assert_rel(g, r, what=what)
    assert_rel(got[3].sum(0), ref[3].sum(0), what="partial rows")
