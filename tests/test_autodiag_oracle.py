"""CPU tests of the AutoDiagonalNormal user-model path: the oracle's generic family reproduces the fused families'
oracle when given their log densities, and d3p_b200.models.AutoDiagonalNormalModel refuses malformed models and
batches before it reaches the library."""
import numpy as np
import pytest
import torch

from helpers import autodiag_models as M
from oracle import autodiag as oad, chacha, families as ofam, svi as osvi


def _px(fam, args, params, mask):
    o = osvi.DPSVI(fam, None, osvi.SGD(1.), None, 1.0, 1.0)
    o.grad_dtype = np.float64
    st = o.init(chacha.PRNGKey(4), *args, params=params)
    st1, keys = o._split_rng_key(st, 2)
    _, loss, grads, n, f = o._compute_per_example_gradients(st1, keys[0], *args, mask=mask)
    return loss, grads, n, f


@pytest.mark.parametrize("kind,d", [("logreg", 1), ("logreg", 6), ("gauss", 5)])
def test_generic_oracle_equals_fused_family_oracle(kind, d):
    N, B = 1000, 9
    rs = np.random.RandomState(d)
    X = rs.randn(B, d).astype(np.float32)
    if kind == "logreg":
        args = (X, (rs.rand(B) < .5).astype(np.int32))
        ref = ofam.LogisticRegression(d, N, guide="auto")
        gen = oad.AutoDiagonalNormalModel([("w", (d,)), ("intercept", ())], M.logreg_ll, N)
        D = d + 1
    else:
        args = (X,)
        ref = ofam.GaussianMean(d, N, guide="auto")
        gen = oad.AutoDiagonalNormalModel([("mu", (d,))], M.gauss_ll, N)
        D = d
    assert gen.latent_dim() == D
    params = {"auto_loc": (.3 * rs.randn(D)).astype(np.float32),
              "auto_scale": (.2 * rs.randn(D) - 1.).astype(np.float32)}
    mask = np.arange(B) < B - 2
    l0, g0, n0, f0 = _px(ref, args, params, mask)
    l1, g1, n1, f1 = _px(gen, args, params, mask)
    assert (n0, f0) == (n1, f1)
    np.testing.assert_allclose(l1, l0, rtol=1e-12, atol=1e-9)
    for k in ("auto_loc", "auto_scale"):
        np.testing.assert_allclose(g1[k], g0[k], rtol=1e-10, atol=1e-12)


def test_generic_oracle_evaluate_equals_fused_family_oracle():
    N, B, d = 500, 12, 4
    rs = np.random.RandomState(0)
    X, y = rs.randn(B, d).astype(np.float32), (rs.rand(B) < .5).astype(np.int32)
    ref = ofam.LogisticRegression(d, N, guide="auto")
    gen = oad.AutoDiagonalNormalModel([("w", (d,)), ("intercept", ())], M.logreg_ll, N)
    vals = []
    for fam in (ref, gen):
        o = osvi.DPSVI(fam, None, osvi.SGD(1.), None, 1.0, 1.0)
        vals.append(o.evaluate(o.init(chacha.PRNGKey(2), X, y, params=fam.init_params(.1 * np.arange(d + 1))), X, y))
    np.testing.assert_allclose(vals[1], vals[0], rtol=1e-6)


def _user(sites=(("w", (3,)), ("b", ()), ("log_sigma", ())), ll=M.linreg_ll, **kw):
    from d3p_b200 import models
    return models.AutoDiagonalNormalModel(list(sites), ll, **kw)


def test_layout_and_descriptor():
    fam = _user([("W", (3, 4)), ("b", (3,)), ("s", ())], M.softmax_ll)
    assert fam.latent_dim == 16 and fam.n_params == 32
    assert fam.layout() == [("auto_loc", 0, (16,)), ("auto_scale", 16, (16,))]
    d = fam.desc(1234.)
    assert (d.latent_dim, d.n_params, d.loc_off, d.scale_off, d.num_obs_total) == (16, 32, 0, 16, 1234.)
    p = fam.init_params()
    np.testing.assert_allclose(torch.nn.functional.softplus(torch.tensor(p["auto_scale"])).numpy(), .1, rtol=1e-6)
    lat = fam.latents(torch.arange(32.).reshape(2, 16))
    assert lat["W"].shape == (2, 3, 4) and lat["b"].shape == (2, 3) and lat["s"].shape == (2,)
    assert lat["W"][1, 2, 3] == 16 + 11 and lat["b"][0, 1] == 13 and lat["s"][1] == 31


def test_potential_and_grad_on_cpu_tensors():
    """U and h of the default N(0, 1) prior + a linear regression, against closed forms."""
    fam = _user()
    rs = np.random.RandomState(1)
    th = torch.tensor(rs.randn(6, 5).astype(np.float32))
    X, y = torch.tensor(rs.randn(6, 3).astype(np.float32)), torch.tensor(rs.randn(6).astype(np.float32))
    U, h = fam.potential_and_grad(th, [X, y], 100.)
    w, b, ls = th[:, :3], th[:, 3], th[:, 4]
    sig = torch.exp(ls)
    r = (y - (X * w).sum(-1) - b) / sig
    U_ref = 0.5 * (th * th).sum(1) + 5 * M.LOG_SQRT_2PI - 100. * (-0.5 * r * r - ls - M.LOG_SQRT_2PI)
    np.testing.assert_allclose(U.numpy(), U_ref.numpy(), rtol=1e-5)
    h_w = w - 100. * (r / sig)[:, None] * X
    np.testing.assert_allclose(h[:, :3].numpy(), h_w.numpy(), rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(h[:, 4].numpy(), (ls - 100. * (r * r - 1)).numpy(), rtol=1e-4, atol=1e-3)
    assert U.is_contiguous() and h.is_contiguous() and h.shape == th.shape


def test_shape_and_arity_errors_before_any_native_call():
    from d3p_b200 import _native, minibatch as mb
    lib_before = _native._lib
    fam = _user()
    X, y = np.zeros((4, 3), np.float32), np.zeros(4, np.float32)
    fam.check_args((X, y))
    with pytest.raises(ValueError, match="does not take"):
        fam.check_args((X,))
    with pytest.raises(ValueError, match="does not take"):
        fam.check_args((X, y, y))
    with pytest.raises(ValueError, match="leading"):
        fam.check_args((X, np.zeros(5, np.float32)))
    with pytest.raises(ValueError, match="LocalRows"):
        fam.check_args((mb.LocalRows(torch.zeros(2, 3), 0, 4), mb.LocalRows(torch.zeros(2), 0, 4)))
    th = torch.zeros(4, 5)
    bad = _user(ll=lambda lat, X, y: M.linreg_ll(lat, X, y)[:, None])         # [B, 1] instead of [B]
    with pytest.raises(ValueError, match="one value per example"):
        bad.potential_and_grad(th, [torch.tensor(X), torch.tensor(y)], 10.)
    scalar = _user(ll=lambda lat, X, y: M.linreg_ll(lat, X, y).sum())        # summed over the batch
    with pytest.raises(ValueError, match="one value per example"):
        scalar.potential_and_grad(th, [torch.tensor(X), torch.tensor(y)], 10.)
    with pytest.raises(ValueError):
        _user(sites=())
    with pytest.raises(ValueError):
        _user(sites=(("a", (2,)), ("a", ())))
    with pytest.raises(TypeError):
        _user(ll=None)
    assert _native._lib is lib_before
