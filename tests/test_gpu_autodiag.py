"""GPU tests of AutoDiagonalNormalModel (user models under an AutoDiagonalNormal guide): the draw against the oracle's
key plumbing, the step against the fused guide="auto" families and against float64 autodiff of new likelihoods, the
edge cases of the step, the epoch / evaluate / sharded paths and the example.

Tolerances: tests/helpers/tolerance.py (1e-5 element-wise, rms floor) unless stated; the draws use the Threefry-normal
tolerance of tests/test_gpu_random.py (the step kernels' normal transform against the oracle's exact one)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import autodiag_models as M
from helpers.tolerance import assert_rel
from oracle import autodiag as oad, chacha, families as ofam, svi as osvi, threefry

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NORMAL_RTOL, NORMAL_ATOL = 2e-6, 2e-7


def _np(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def _user_logreg(d):
    from d3p_b200 import models
    return models.AutoDiagonalNormalModel([("w", (d,)), ("intercept", ())], M.logreg_ll)


def _user_gauss(d):
    from d3p_b200 import models
    return models.AutoDiagonalNormalModel([("mu", (d,))], M.gauss_ll)


def _sgd_step(N, C):
    """SGD step size that moves a parameter by at most ~0.02 per step: the released gradient is up to N * C."""
    return float(np.float32(0.02 / (N * C)))


def _svi(fam, N, optim="adam", C=1.0, dp_scale=1.0):
    from d3p_b200 import models, optimizers, svi
    opt = optimizers.Adam(1e-3) if optim == "adam" else optimizers.SGD(_sgd_step(N, C))
    return svi.DPSVI(fam.model, fam.guide, opt, models.Trace_ELBO(), C, dp_scale, num_obs_total=N)


def _rand_params(D, seed, scale=.3):
    rs = np.random.RandomState(seed)
    return {"auto_loc": (scale * rs.randn(D)).astype(np.float32),
            "auto_scale": (.2 * rs.randn(D) - 1.5).astype(np.float32)}


# ---- 1. draw ------------------------------------------------------------------------------------------------------
def _draw(D, B, key, pos=None, ld=None, device_key=False, params=None):
    from d3p_b200 import _native as _n, models
    fam = models.AutoDiagonalNormalModel([("z", (D,))], M.unit_gauss_ll)
    params = params if params is not None else _rand_params(D, D)
    flat = torch.tensor(np.concatenate([params["auto_loc"], params["auto_scale"]])).cuda()
    pb, pe = pos if pos is not None else (0, max(B, 1))
    ld = ld or D
    rows = pe - pb if B else 1
    theta = torch.full((rows, ld), -7.0, device="cuda")
    eps = torch.full((rows, ld), -7.0, device="cuda")
    desc = fam.desc(100.)
    k = np.ascontiguousarray(key, dtype=np.uint32)
    if device_key:
        kd = torch.as_tensor(k.view(np.int32)).cuda()
        rc = _n.lib().d3p_autodiag_draw_f32_dk(C.byref(desc), _n.ptr(flat), _n.ptr(kd), B, pb, pe, _n.ptr(theta),
                                               _n.ptr(eps), ld, _n.stream_ptr())
    else:
        rc = _n.lib().d3p_autodiag_draw_f32(C.byref(desc), _n.ptr(flat), k.ctypes.data_as(C.POINTER(C.c_uint32)), B,
                                            pb, pe, _n.ptr(theta), _n.ptr(eps), ld, _n.stream_ptr())
    _n.check(rc, "draw")
    t, e = _np(theta), _np(eps)
    assert np.all(t[:, D:] == -7.0) and np.all(e[:, D:] == -7.0)     # the row padding of ld is not written
    return t[:, :D], e[:, :D], params


@pytest.mark.parametrize("D", [1, 7, 1025, 40000])
def test_draw_matches_oracle_joint_site(cuda, D):
    B = 5 if D < 40000 else 3
    key = threefry.PRNGKey(1000 + D)
    theta, eps, p = _draw(D, B, key, ld=D + 3)
    ref = oad.AutoDiagonalNormalModel([("z", (D,))], M.unit_gauss_ll, 100.).sample_eps(threefry.split(key, B))
    assert np.allclose(eps, ref["_auto_latent"], rtol=NORMAL_RTOL, atol=NORMAL_ATOL)
    s = np.log1p(np.exp(p["auto_scale"].astype(np.float64)))
    assert_rel(theta, p["auto_loc"] + eps.astype(np.float64) * s, rtol=1e-6, what="theta")
    t2, e2, _ = _draw(D, B, key, device_key=True)
    assert np.array_equal(t2, theta) and np.array_equal(e2, eps)


def test_draw_sub_range_and_evaluate_draw(cuda):
    D, B = 301, 40
    key = threefry.PRNGKey(7)
    t_full, e_full, _ = _draw(D, B, key)
    t_sub, e_sub, _ = _draw(D, B, key, pos=(13, 29), ld=D + 1)
    assert np.array_equal(t_sub, t_full[13:29]) and np.array_equal(e_sub, e_full[13:29])
    # B == 0: SVI.evaluate's single draw from the key itself, the exact transform of the evaluate kernel
    t0, e0, p = _draw(D, 0, key)
    ref = oad.AutoDiagonalNormalModel([("z", (D,))], M.unit_gauss_ll, 100.).sample_eps(key.reshape(1, 2))
    assert np.allclose(e0, ref["_auto_latent"], rtol=NORMAL_RTOL, atol=NORMAL_ATOL)
    assert not np.allclose(e0, e_full[:1])
    t0d, e0d, _ = _draw(D, 0, key, device_key=True)
    assert np.array_equal(t0d, t0) and np.array_equal(e0d, e0)


# ---- 2. the same results as the fused guide="auto" families -------------------------------------------------------
def _batch(kind, N, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.randn(N, d).astype(np.float32) if kind == "logreg" else (1. + .1 * rs.randn(N, d)).astype(np.float32)
    if kind == "logreg":
        return (torch.tensor(X).cuda(), torch.tensor((rs.rand(N) < .5).astype(np.int32)).cuda())
    return (torch.tensor(X).cuda(),)


def _step_outputs(s, st, key, args, mask, B, P):
    px_norms = torch.zeros(B, device="cuda")
    px_grads = torch.zeros(B, P, device="cuda")
    px_loss = torch.zeros(B, device="cuda")
    ws, n_part, _, _ = s._run_step(st, key, args, mask, px_norms, px_grads, px_loss)
    sums = ws[:n_part * (P + 2)].reshape(n_part, P + 2).double().sum(0)
    return _np(px_norms), _np(px_grads), _np(px_loss), _np(sums)


@pytest.mark.parametrize("kind,d,batch", [("logreg", 8, "plain"), ("logreg", 8, "poisson"), ("logreg", 1024, "plain"),
                                          ("logreg", 1024, "poisson"), ("gauss", 8, "plain"), ("gauss", 8, "poisson"),
                                          ("gauss", 300, "poisson")])
def test_user_model_equals_fused_auto_family(cuda, kind, d, batch):
    from d3p_b200 import minibatch as mb, models
    N = 3000
    data = _batch(kind, N, d, seed=d)
    if batch == "plain":
        B = 37 if d < 1024 else 19
        args = tuple(a[:B] for a in data)
        mask = torch.as_tensor(np.arange(B) < B - 4).cuda()
    else:
        init, get = mb.poisson_batchify_data(data, 0.01, .99)
        _, bst = init(chacha.PRNGKey(3))
        args, mask = get(0, bst)
        B = int(args[0].shape[0])
        assert int(args[0].num_valid.item()) < B          # padding rows present
    fused = models.LogisticRegression(d, guide="auto") if kind == "logreg" else models.GaussianMean(d, guide="auto")
    user = _user_logreg(d) if kind == "logreg" else _user_gauss(d)
    assert fused.layout() == user.layout()
    P = user.n_params
    p = _rand_params(P // 2, seed=5, scale=.2)
    sf, su = _svi(fused, N), _svi(user, N)
    key = chacha.PRNGKey(9)
    stf, stu = sf.init(key, *args, params=p), su.init(key, *args, params=p)
    k = chacha.split(key, 2)[1]
    of = _step_outputs(sf, stf, k, args, mask, B, P)
    ou = _step_outputs(su, stu, k, args, mask, B, P)
    # one floor (the rms) per compared vector, as tests/test_gpu_svi.py: in a row whose logit saturates on the side of
    # its label, sigmoid(z) - y is below float32's resolution of sigmoid(z) near 1 on both sides (the fused kernel's
    # sigmoid_f, autograd's sum of the BernoulliLogits terms), so that row agrees only to ~1e-3 of its own size
    for name, a, b in zip(("norms", "px_grads", "S*loss"), ou, of):
        assert_rel(a, b, what=name)
    assert_rel(ou[3][:P], of[3][:P], what="summed partial rows: gradient")
    assert_rel(ou[3][P:], of[3][P:], what="summed partial rows: loss, count")
    for step in range(3):
        stf, lf = sf.update(stf, *args, mask=mask)
        stu, lu = su.update(stu, *args, mask=mask)
        assert np.isclose(float(lu), float(lf), rtol=1e-5), (step, float(lu), float(lf))
        assert_rel(stu.optim_state.flat, stf.optim_state.flat, what=f"Adam step {step}")


# ---- 3. new likelihoods against float64 autodiff ------------------------------------------------------------------
def _model_data(kind, B, d, seed):
    rs = np.random.RandomState(seed)
    X = (rs.randn(B, d) / np.sqrt(d)).astype(np.float32)
    if kind == "real":
        return (X, (X.sum(1) + .3 * rs.randn(B)).astype(np.float32))
    if kind == "count":
        return (X, rs.poisson(2.0, B).astype(np.float32))
    if kind == "class3":
        return (X, rs.randint(0, 3, B).astype(np.int32))
    return ((.5 + .3 * rs.randn(B, d)).astype(np.float32),)


def _pair(name, d, N, optim, C):
    from d3p_b200 import models
    sites_of, ll, kind = M.MODELS[name]
    fam = models.AutoDiagonalNormalModel(sites_of(d), ll)
    ofm = oad.AutoDiagonalNormalModel(sites_of(d), ll, N)
    oopt = osvi.Adam(1e-3) if optim == "adam" else osvi.SGD(_sgd_step(N, C))
    o = osvi.DPSVI(ofm, None, oopt, None, C, 1.0)
    o.grad_dtype = np.float64
    return fam, _svi(fam, N, optim, C), o, kind


@pytest.mark.parametrize("name", sorted(M.MODELS))
def test_new_likelihoods_match_float64_oracle(cuda, name):
    N, B, d = 2000, 33, 6
    _, _, o, kind = _pair(name, d, N, "sgd", 1.0)
    args = _model_data(kind, B, d, seed=11)
    targs = tuple(torch.tensor(a).cuda() for a in args)
    key = chacha.PRNGKey(21)
    mask = np.arange(B) % 5 != 3
    tmask = torch.as_tensor(mask).cuda()
    ost = o.init(key, *args, params=_rand_params(sum(int(np.prod(s)) for _, s in M.MODELS[name][0](d)), 12, .2))
    _, olosses, ograds, on, of = o._compute_per_example_gradients(ost, ost.rng_key, *args, mask=mask)
    og = np.concatenate([ograds["auto_loc"], ograds["auto_scale"]], axis=1).astype(np.float64)
    onorm = np.linalg.norm(og, axis=1)
    C = float(np.float32(np.median(onorm[mask])))          # about half of the examples are clipped
    fam, s, o, _ = _pair(name, d, N, "sgd", C)
    p = _rand_params(fam.latent_dim, seed=12, scale=.2)
    st, ost = s.init(key, *targs, params=p), o.init(key, *args, params=p)
    _, losses, grads, n, f = s._compute_per_example_gradients(st, st.rng_key, *targs, mask=tmask)
    assert n == on and np.isclose(f, of)
    for k in grads:
        assert_rel(grads[k], ograds[k], what=f"px_grads[{k}]", axis=0)
        assert np.all(_np(grads[k])[~mask] == 0)
    assert_rel(losses, olosses, what="px_losses")
    # norms and clipped sums: the oracle's per-example gradients, clipped and summed in float64
    P = fam.n_params
    oc = og / np.maximum(1., onorm / C)[:, None]
    norms, _, sloss, sums = _step_outputs(s, st, st.rng_key, targs, tmask, B, P)
    assert_rel(norms[mask], onorm[mask], what="norms")
    assert np.all(norms[~mask] == 0)
    assert_rel(sums[:P], oc[mask].sum(0), what="clipped sum")
    assert_rel(sums[P], np.sum(olosses[mask] / f), what="loss sum")
    assert sums[P + 1] == mask.sum()
    for optim in ("sgd", "adam"):
        fam, s, o, _ = _pair(name, d, N, optim, C)
        st, ost = s.init(key, *targs, params=p), o.init(key, *args, params=p)
        for step in range(3):
            st, loss = s.update(st, *targs, mask=tmask)
            ost, oloss = o.update(ost, *args, mask=mask)
            assert np.isclose(float(loss), float(oloss), rtol=1e-5), (optim, step, float(loss), float(oloss))
            got, ref = s.get_params(st), o.get_params(ost)
            assert_rel(got["auto_loc"], ref["auto_loc"], what=f"{optim} step {step} auto_loc")
            assert_rel(got["auto_scale"], np.log1p(np.exp(ref["auto_scale"].astype(np.float64))),
                       what=f"{optim} step {step} auto_scale")


# ---- 4. edge cases ------------------------------------------------------------------------------------------------
def test_quad_finalize_size(cuda):
    """D = 20000: P = 40000 >= 32768, the step keeps n_partials <= 64 so that finalize_quad_kernel runs."""
    from d3p_b200 import _native as _n
    d, N, B = 20000, 1000, 24
    fam, s, o, _ = _pair("generic_normal_mean", d, N, "adam", 5.0)
    n_part = C.c_uint32(0)
    assert _n.lib().d3p_autodiag_workspace_bytes(C.byref(fam.desc(N)), B, C.byref(n_part)) > 0
    assert 1 <= n_part.value <= 64
    X = (.5 + .3 * np.random.RandomState(0).randn(B, d)).astype(np.float32)
    tX = torch.tensor(X).cuda()
    p = _rand_params(d, seed=3, scale=.1)
    key = chacha.PRNGKey(1)
    st, ost = s.init(key, tX, params=p), o.init(key, X, params=p)
    for step in range(2):
        st, loss = s.update(st, tX)
        ost, oloss = o.update(ost, X)
        assert np.isclose(float(loss), float(oloss), rtol=1e-5)
        assert_rel(s.get_params(st)["auto_loc"], o.get_params(ost)["auto_loc"], what=f"step {step}")


def test_nan_padding_rows_leave_sums_finite(cuda):
    """A likelihood that is NaN on an all-zero record: the zero-filled padding rows of a Poisson batch are skipped,
    and the valid rows give exactly what the NaN-free likelihood gives."""
    from d3p_b200 import minibatch as mb, models
    d, N = 16, 4000
    X = torch.tensor((1. + .1 * np.random.RandomState(2).randn(N, d)).astype(np.float32)).cuda()
    init, get = mb.poisson_batchify_data((X,), 0.01, .99)
    _, bst = init(chacha.PRNGKey(8))
    args, mask = get(0, bst)
    B = int(args[0].shape[0])
    assert int(args[0].num_valid.item()) < B
    out = []
    for ll in (M.nan_at_zero_gauss_ll, M.gauss_ll):
        fam = models.AutoDiagonalNormalModel([("mu", (d,))], ll)
        s = _svi(fam, N)
        st = s.init(chacha.PRNGKey(0), *args, params=_rand_params(d, 4))
        o = _step_outputs(s, st, chacha.PRNGKey(5), args, mask, B, fam.n_params)
        st, loss = s.update(st, *args, mask=mask)
        out.append((o[3], _np(st.optim_state.flat), float(loss)))
    assert np.all(np.isfinite(out[0][0])) and np.all(np.isfinite(out[0][1])) and np.isfinite(out[0][2])
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]) and out[0][2] == out[1][2]


def test_all_masked_batch_as_fused_family(cuda):
    d, N, B = 8, 1000, 20
    X, y = _batch("logreg", B, d, seed=1)
    mask = torch.zeros(B, dtype=torch.bool, device="cuda")
    from d3p_b200 import models
    res = []
    for fam in (_user_logreg(d), models.LogisticRegression(d, guide="auto")):
        s = _svi(fam, N)
        st = s.init(chacha.PRNGKey(2), X, y, params=_rand_params(d + 1, 6))
        st, loss = s.update(st, X, y, mask=mask)
        res.append((_np(st.optim_state.flat), float(loss)))
    assert np.array_equal(res[0][0], res[1][0], equal_nan=True)
    assert np.array_equal(np.float32(res[0][1]), np.float32(res[1][1]), equal_nan=True)


def test_refusals(cuda):
    from d3p_b200 import _native as _n
    lib = _n.lib()
    fam = _user_gauss(4)
    P, D, B = 8, 4, 3
    flat = torch.zeros(P, device="cuda")
    eps, h, U = torch.zeros(B, 5, device="cuda"), torch.zeros(B, 5, device="cuda"), torch.zeros(B, device="cuda")
    ws = torch.zeros(1 << 20, device="cuda")
    key = np.zeros(2, np.uint32)
    kp = key.ctypes.data_as(C.POINTER(C.c_uint32))

    def step(desc, ld=5, Cc=1.0, S=10.0):
        return lib.d3p_dpsvi_step_autodiag(C.byref(desc), _n.ptr(flat), _n.ptr(eps), _n.ptr(h), ld, _n.ptr(U), None,
                                           None, B, 0, B, S, Cc, None, None, None, _n.ptr(ws), ws.numel() * 4,
                                           _n.stream_ptr())

    def draw(desc, ld=5):
        return lib.d3p_autodiag_draw_f32(C.byref(desc), _n.ptr(flat), kp, B, 0, B, _n.ptr(eps), _n.ptr(h), ld,
                                         _n.stream_ptr())

    good = fam.desc(10.)
    assert step(good) == 0 and draw(good) == 0
    bad = [_n.AutodiagDesc(D, P, 5, 0, 10.), _n.AutodiagDesc(D, P, 0, 5, 10.), _n.AutodiagDesc(D, P, 0, 2, 10.),
           _n.AutodiagDesc(0, P, 0, 4, 10.)]
    for d in bad:
        assert step(d) == -1 and draw(d) == -1
        assert lib.d3p_autodiag_workspace_bytes(C.byref(d), B, None) == 0
    assert step(good, ld=3) == -1 and draw(good, ld=3) == -1
    assert step(good, Cc=0.0) == -1 and step(good, S=0.0) == -1
    torch.cuda.synchronize()


# ---- 5. loops and sharding ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("sampler", ["poisson", "subsample", "split"])
def test_run_epoch_equals_update_loop(cuda, sampler):
    from d3p_b200 import minibatch as mb
    d, N = 5, 2000
    fam, s, _, kind = _pair("poisson", d, N, "adam", 2.0)
    X, y = (torch.tensor(a).cuda() for a in _model_data(kind, N, d, seed=4))
    if sampler == "poisson":
        init, get = mb.poisson_batchify_data((X, y), 0.02, .99)
    elif sampler == "subsample":
        init, get = mb.subsample_batchify_data((X, y), batch_size=40)
    else:
        init, get = mb.split_batchify_data((X, y), batch_size=40)
    _, bst = init(chacha.PRNGKey(6))
    p = _rand_params(fam.latent_dim, 8, .1)
    st0 = s.init(chacha.PRNGKey(1), X, y, params=p)
    st_e, stats = s.run_epoch(st0, get, bst, 4)
    st = st0
    losses = []
    for i in range(4):
        out = get(i, bst)
        batch, mask = (out, True) if sampler == "subsample" or sampler == "split" else out
        st, loss = s.update(st, *batch, mask=mask)
        losses.append(float(loss))
    assert np.array_equal(_np(st_e.optim_state.flat), _np(st.optim_state.flat))
    assert np.array_equal(_np(stats[:, 0]), np.asarray(losses, np.float32))


def test_evaluate_matches_oracle(cuda):
    d, N, B = 7, 1500, 50
    for name in ("linreg", "softmax"):
        fam, s, o, kind = _pair(name, d, N, "adam", 1.0)
        args = _model_data(kind, B, d, seed=9)
        targs = tuple(torch.tensor(a).cuda() for a in args)
        p = _rand_params(fam.latent_dim, 10, .2)
        st, ost = s.init(chacha.PRNGKey(4), *targs, params=p), o.init(chacha.PRNGKey(4), *args, params=p)
        assert np.isclose(float(s.evaluate(st, *targs)), o.evaluate(ost, *args), rtol=1e-5), name
    # the fused family's evaluate on the same draw
    from d3p_b200 import models
    X, y = _batch("logreg", B, d, seed=2)
    p = _rand_params(d + 1, 11, .2)
    vals = []
    for fam in (_user_logreg(d), models.LogisticRegression(d, guide="auto")):
        s = _svi(fam, N)
        vals.append(float(s.evaluate(s.init(chacha.PRNGKey(3), X, y, params=p), X, y)))
    assert np.isclose(vals[0], vals[1], rtol=1e-5), vals


def test_sharded_update_equals_unsharded(cuda):
    from d3p_b200 import parallel
    d, N, B, world = 12, 3000, 45, 2
    X, y = (torch.tensor(a).cuda() for a in _model_data("real", B, d, seed=13))
    mask = torch.as_tensor(np.arange(B) % 7 != 2).cuda()
    p = _rand_params(d + 2, 14, .2)
    ref_fam, ref, _, _ = _pair("linreg", d, N, "adam", 2.0)
    st_ref = ref.init(chacha.PRNGKey(2), X, y, params=p)
    fams = [_pair("linreg", d, N, "adam", 2.0)[0] for _ in range(world)]
    wins = parallel.PeerWindow.local_group(world, fams[0].n_params)
    for w in wins:
        w.set_timeout_ms(4000)
    svis = [parallel.shard_dpsvi(_svi(f, N, "adam", 2.0), window=w) for f, w in zip(fams, wins)]
    states = [sv.init(chacha.PRNGKey(2), X, y, params=p) for sv in svis]
    streams = [torch.cuda.Stream() for _ in range(world)]
    for step in range(3):
        st_ref, loss_ref = ref.update(st_ref, X, y, mask=mask)
        torch.cuda.synchronize()
        ctx, out = [None] * world, [None] * world
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                ctx[r] = svis[r]._update_launch_step(states[r], (X, y), mask)
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                states[r], out[r] = svis[r]._update_finalize(ctx[r])
        torch.cuda.synchronize()
        assert all(w.timeouts() == 0 for w in wins)
        assert np.array_equal(_np(states[0].optim_state.flat), _np(states[1].optim_state.flat))
        assert float(out[0]) == float(out[1])
        assert_rel(states[0].optim_state.flat, st_ref.optim_state.flat, what=f"sharded step {step}")
        assert np.isclose(float(out[0]), float(loss_ref), rtol=1e-5)
    for w in wins:
        w.close()


# ---- 6. the example -----------------------------------------------------------------------------------------------
def test_example_recovers_the_weights(cuda, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "autodiag_linear_regression.py"),
                        "--json", str(tmp_path / "out.json")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    import json
    out = json.load(open(tmp_path / "out.json"))
    assert 0.5 < out["epsilon"] < 2.0
    w, w_true = np.asarray(out["w_loc"]), np.asarray(out["w_true"])
    assert np.all(np.sign(w) == np.sign(w_true)), (w, w_true)
    assert np.max(np.abs(w - w_true)) < 0.25 * np.max(np.abs(w_true)), (w, w_true)
    assert abs(out["sigma"] - out["sigma_true"]) < 0.5 * out["sigma_true"], out
