"""GPU tests of the numpyro optimizers Momentum / Adagrad / RMSProp / RMSPropMomentum / ClippedAdam and the step-size
schedules, fused into the finalize kernels: DP-SVI trajectories against the oracle (oracle/optim.py plugged into
oracle.svi.DPSVI) for every model family, both finalize kernels called directly for every kind, the stage-method
``optim.update``, the epoch drivers (bit-identical to the step loop), the sharded in-kernel exchange on one device, and
the descriptor refusals.  Tolerance: tests/helpers/tolerance.py, 1e-5 element-wise with the vector's rms as floor."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers.tolerance import assert_rel
from oracle import chacha, families as ofam, gmm as ogmm, optim as oopt, svi as osvi, vae as ovae

pytestmark = pytest.mark.gpu

RTOL = 1e-5

# name -> (constructor taking (optimizers module, step size), step size, schedule (name, args), oracle state index of
# OptimState.m, of OptimState.v).  RMSProp's eps sits inside the root: with the default 1e-8, g / sqrt(v + eps) of a
# gradient element near 1e-4 (the VAE has many) turns a 1e-6 difference of g into a 1e-5 one of the update, so the
# comparison uses eps = 1e-3, which keeps the step well conditioned and eps still far from negligible.
KINDS = {
    "momentum": (lambda o, ss: o.Momentum(ss, 0.9), 1e-3, ("exponential_decay", (1e-3, 2, 0.5)), 1, None),
    "adagrad": (lambda o, ss: o.Adagrad(ss, momentum=0.8), 1e-2, ("inverse_time_decay", (1e-2, 2, 1.0, True)), 2, 1),
    "rmsprop": (lambda o, ss: o.RMSProp(ss, gamma=0.8, eps=1e-3), 1e-3, ("polynomial_decay", (1e-3, 3, 1e-4, 2.0)),
                None, 1),
    "rmsprop_momentum": (lambda o, ss: o.RMSPropMomentum(ss, gamma=0.8, eps=1e-3, momentum=0.7), 1e-3,
                         ("piecewise_constant", ([0, 2], [1e-3, 5e-4, 2e-4])), 2, 1),
    "clipped_adam": (lambda o, ss: o.ClippedAdam(ss, clip_norm=10.0), 1e-3, ("inverse_time_decay", (1e-3, 2, 0.5)), 1, 2),
    "adam": (lambda o, ss: o.Adam(ss), 1e-3, ("exponential_decay", (1e-3, 3, 0.3)), 1, 2),
    "sgd": (lambda o, ss: o.SGD(ss), 1e-4, ("polynomial_decay", (1e-4, 3, 1e-5)), None, None),
}
NEW = ["momentum", "adagrad", "rmsprop", "rmsprop_momentum", "clipped_adam"]


def make_optims(name, scheduled):
    """-> (d3p_b200 optimizer, oracle optimizer) of the same configuration."""
    from d3p_b200 import optimizers
    ctor, lr, (sname, sargs), _, _ = KINDS[name]
    if scheduled:
        return ctor(optimizers, getattr(optimizers, sname)(*sargs)), ctor(oopt, getattr(oopt, sname)(*sargs))
    return ctor(optimizers, lr), ctor(oopt, lr)


def _family(fam, opt, oopt_):
    """-> (DPSVI, oracle DPSVI, gpu args, numpy args, mask, initial params, init key)"""
    from d3p_b200 import models, svi
    rs = np.random.RandomState(3)
    if fam == "logreg":
        d, N, B, clip = 8, 5000, 41, 1.0
        f, of = models.LogisticRegression(d, guide="hand"), ofam.LogisticRegression(d, N, guide="hand")
        args = (rs.randn(B, d).astype(np.float32), (rs.rand(B) < .5).astype(np.int32))
    elif fam == "gauss":
        d, N, B, clip = 7, 5000, 37, 50.0
        f, of = models.GaussianMean(d, guide="auto"), ofam.GaussianMean(d, N, guide="auto")
        args = ((1. + .1 * rs.randn(B, d)).astype(np.float32),)
    elif fam == "gmm":
        K, d, N, B, clip = 3, 2, 2000, 24, 20.0
        centers = rs.randn(K, d).astype(np.float32) * 3
        args = ((centers[rs.randint(0, K, B)] + rs.randn(B, d)).astype(np.float32),)
        f, of = models.GaussianMixture(K, d), ogmm.GaussianMixture(K, d, N)
        p0 = {"alpha_log": (rs.randn(K) * 0.4).astype(np.float32),
              "mus_loc": (centers + rs.randn(K, d) * 0.5).astype(np.float32)}
    else:
        # 256-64-8: P = 34 960 >= 32 768 with the step's few partial rows, i.e. finalize_quad_kernel
        D, H, Z, N, B, clip = 256, 64, 8, 1000, 12, 5.0
        args = ((rs.rand(B, 16, 16) < 0.35).astype(np.float32),)
        f, of = models.VAE(D, H, Z), ovae.VAE(D, H, Z, N)
        p0 = of.init_params(0, 0.03)
    if fam in ("logreg", "gauss"):
        p0 = {k: np.asarray(rs.randn(*v.shape) * .2, dtype=np.float32) for k, v in f.init_params().items()}
    s = svi.DPSVI(f.model, f.guide, opt, models.Trace_ELBO(), clip, 1.0, num_obs_total=N)
    o = osvi.DPSVI(of, None, oopt_, None, clip, 1.0)
    B = args[0].shape[0]
    mask = np.arange(B) != 2
    return s, o, [torch.as_tensor(a).cuda() for a in args], args, mask, p0


def _check_state(name, s, st, ost, what):
    """parameters and the optimizer's m / v against the oracle's state tuple (raw, unconstrained values)."""
    from d3p_b200.optimizers import unflatten
    os_ = st.optim_state
    _, _, _, mi, vi = KINDS[name]
    ref = ost.optim_state[1]
    ref = ref if isinstance(ref, tuple) else (ref,)
    for buf, idx, tag in ((os_.flat, 0, "x"), (os_.m, mi, "m"), (os_.v, vi, "v")):
        if idx is None:
            continue
        got = unflatten(buf, os_.layout)
        for k in ref[idx]:
            assert_rel(got[k], ref[idx][k], rtol=RTOL, what=f"{what} {tag}[{k}]")


@pytest.mark.parametrize("fam", ["logreg", "gauss", "gmm", "vae"])
@pytest.mark.parametrize("scheduled", [False, True], ids=["const", "sched"])
@pytest.mark.parametrize("name", NEW + ["adam"])
def test_trajectory_matches_oracle(cuda, name, scheduled, fam):
    if name == "adam" and not scheduled:
        pytest.skip("unscheduled Adam: tests/test_gpu_svi.py and friends")
    opt, oo = make_optims(name, scheduled)
    s, o, targs, args, mask, p0 = _family(fam, opt, oo)
    key = chacha.PRNGKey(9)
    st, ost = s.init(key, *targs, params=p0), o.init(key, *args, params=p0)
    tmask = torch.as_tensor(mask).cuda()
    for step in range(4):
        st, loss = s.update(st, *targs, mask=tmask)
        ost, oloss = o.update(ost, *args, mask=mask)
        assert np.array_equal(st.rng_key, ost.rng_key)
        assert np.isclose(float(loss), float(oloss), rtol=2e-5), (step, float(loss), float(oloss))
        _check_state(name, s, st, ost, f"{name} {fam} step {step}")
    assert st.optim_state.step == 4
    want_m, want_v = KINDS[name][3] is not None, KINDS[name][4] is not None
    assert (st.optim_state.m is not None, st.optim_state.v is not None) == (want_m, want_v)


def _leaf_table(lens, key):
    from d3p_b200 import _native as _n
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(int)
    site_keys = chacha.split(key, len(lens))
    lt = _n.LeafTable()
    lt.n_leaves = len(lens)
    for l, n in enumerate(lens):
        lt.leaf_off[l], lt.leaf_len[l] = int(offs[l]), int(n)
        for i in range(16):
            lt.site_state[l][i] = int(np.asarray(site_keys[l], np.uint32).reshape(16)[i])
    return lt, site_keys


@pytest.mark.parametrize("shape", [(40000, 4), (40000, 1), (2050, 296)], ids=["quad4", "quad1", "c2"])
@pytest.mark.parametrize("scheduled", [False, True], ids=["const", "sched"])
@pytest.mark.parametrize("name", NEW + ["adam", "sgd"])
def test_finalize_kernels_direct(cuda, name, scheduled, shape):
    """d3p_perturb_finalize_f32 with a leaf table: P >= 32 768 and <= 4 partial rows runs finalize_quad_kernel, the C2
    shape (P = 2 050, 296 rows) finalize_kernel.  grad_out against a numpy restatement of reduce + noise + rescale, then
    x / m / v against the oracle optimizer applied to that gradient, from non-zero state at step 5."""
    from d3p_b200 import _native as _n
    P, n_part = shape
    rs = np.random.RandomState(P + n_part)
    lens = [P // 3, P // 3, P - 2 * (P // 3)]
    lt, site_keys = _leaf_table(lens, chacha.fold_in(chacha.PRNGKey(4), P))
    B, n, step = 300, 280, 5
    part = (rs.randn(n_part, P + 2) * 0.5).astype(np.float32)
    part[:, P + 1] = 0
    part[0, P + 1] = n
    dp_scale, clip, obs = 1.0, 2.0, 30.0
    gpu_opt, o_opt = make_optims(name, scheduled)
    if name == "clipped_adam":             # |g| is O(1) here: a bound inside that range clips some elements, not all
        gpu_opt.clip_norm, o_opt.clip_norm = 0.2, np.float32(0.2)
    od = gpu_opt.desc(step)
    x0 = rs.randn(P).astype(np.float32)
    m0, v0 = (rs.randn(P) * .1).astype(np.float32), (rs.rand(P) * .1).astype(np.float32)
    d = {k: torch.as_tensor(a).cuda() for k, a in (("part", part), ("x", x0), ("m", m0), ("v", v0))}
    d_g = torch.empty(P, device=cuda)
    lib = _n.lib()
    _n.check(lib.d3p_perturb_finalize_f32(_n.ptr(d["part"]), n_part, P, B, C.byref(lt), dp_scale, clip, obs, 1,
                                          _n.ptr(d_g), C.byref(od), _n.ptr(d["x"]), _n.ptr(d["m"]), _n.ptr(d["v"]),
                                          None, None, _n.stream_ptr()), "finalize")
    f32 = np.float32
    f, sigma = f32(B) / f32(n), f32(dp_scale) * (f32(clip) / f32(n))
    noise = np.concatenate([chacha.normal(site_keys[l], (lens[l],)) for l in range(3)])
    want_g = ((part.astype(np.float64).sum(0)[:P] / B).astype(f32) + noise * sigma) * f32(obs) * f
    g = d_g.cpu().numpy()
    assert_rel(g, want_g, rtol=RTOL, what="grad_out (unclipped gradient)")
    if name == "clipped_adam":
        assert np.abs(g).max() > 0.2 > np.abs(g).min(), "the clip must bite on some elements and not on others"
    _, _, _, mi, vi = KINDS[name]
    init = [x0] + [None, None]
    if mi is not None:
        init[mi] = m0
    if vi is not None:
        init[vi] = v0
    state = (step, tuple({"x": a} for a in init if a is not None)) if name != "sgd" else (step, {"x": x0})
    _, new = o_opt.update({"x": g}, state)
    new = new if isinstance(new, tuple) else (new,)
    assert_rel(d["x"].cpu(), new[0]["x"], rtol=RTOL, what=f"{name} x")
    if mi is not None:
        assert_rel(d["m"].cpu(), new[mi]["x"], rtol=RTOL, what=f"{name} m")
    else:
        assert torch.equal(d["m"].cpu(), torch.as_tensor(m0)), "m must be left alone"
    if vi is not None:
        assert_rel(d["v"].cpu(), new[vi]["x"], rtol=RTOL, what=f"{name} v")
    else:
        assert torch.equal(d["v"].cpu(), torch.as_tensor(v0)), "v must be left alone"


@pytest.mark.parametrize("scheduled", [False, True], ids=["const", "sched"])
@pytest.mark.parametrize("name", NEW)
def test_stage_method_update(cuda, name, scheduled):
    """optim.update(grads, state) (the stage method) against the oracle, with an all-zero leaf."""
    rs = np.random.RandomState(1)
    params = {"a": rs.randn(5).astype(np.float32), "b": rs.randn(3, 2).astype(np.float32),
              "z": rs.randn(4).astype(np.float32)}
    opt, oo = make_optims(name, scheduled)
    st, ost = opt.init(params), oo.init(params)
    for it in range(3):
        grads = {k: (rs.randn(*v.shape) * 3).astype(np.float32) for k, v in params.items()}
        grads["z"][:] = 0
        st, ost = opt.update(grads, st), oo.update(grads, ost)
    got = opt.get_params(st)
    for k in params:
        assert torch.isfinite(got[k]).all(), k
        assert_rel(got[k], ost[1][0][k], rtol=RTOL, what=f"{name} {k}")
    assert torch.equal(got["z"].cpu(), torch.as_tensor(params["z"])), "a leaf that never had a gradient stays put"
    assert st.step == 3


def _epoch_setup(fam_name, opt):
    from d3p_b200 import minibatch as mb, models, svi
    import d3p_b200.random as rng
    rs = np.random.RandomState(5)
    if fam_name == "meanfield":
        N, d = 4000, 16
        X = torch.as_tensor(rs.randn(N, d).astype(np.float32)).cuda()
        y = torch.as_tensor((rs.rand(N) < .5).astype(np.int32)).cuda()
        fam, data, clip = models.LogisticRegression(d), (X, y), 1.0
        init, get = mb.poisson_batchify_data(data, .02, .99)
    elif fam_name == "gmm":
        K, d, N = 4, 3, 4000
        centers = rs.randn(K, d).astype(np.float32) * 3
        X = torch.as_tensor((centers[rs.randint(0, K, N)] + rs.randn(N, d)).astype(np.float32)).cuda()
        fam, clip = models.GaussianMixture(K, d), 20.0
        init, get = mb.poisson_batchify_data((X,), 0.02, .99)
    else:
        N, B = 600, 48
        X = torch.as_tensor((rs.rand(N, 8, 8) < 0.35).astype(np.float32)).cuda()
        fam, clip = models.VAE(64, 40, 8, init_std=0.1), 2.0
        init, get = mb.subsample_batchify_data((X,), batch_size=B, return_mask=True)
    s = svi.DPSVI(fam.model, fam.guide, opt, models.Trace_ELBO(), clip, 1.0, num_obs_total=N)
    key, k_init, k_fetch = rng.split(rng.PRNGKey(6), 3)
    _, bst = init(k_fetch)
    batch, _ = get(0, bst)
    return s, s.init(k_init, *batch), get, bst


def _stepwise(s, st, get, bst, first_step, n_steps):
    losses = []
    for i in range(first_step, first_step + n_steps):
        batch, mask = get(i, bst)
        st, loss = s.update(st, *batch, mask=mask)
        losses.append(float(loss))
    return st, losses


def _same(a, b):
    for x, y in ((a.optim_state.flat, b.optim_state.flat), (a.optim_state.m, b.optim_state.m),
                 (a.optim_state.v, b.optim_state.v)):
        assert (x is None and y is None) or torch.equal(x, y), "run_epoch must be bit-identical to the step loop"
    assert np.array_equal(np.asarray(a.rng_key), np.asarray(b.rng_key))
    assert a.optim_state.step == b.optim_state.step


@pytest.mark.parametrize("device_keys", [False, True], ids=["host_keys", "device_keys"])
@pytest.mark.parametrize("fam", ["meanfield", "gmm", "vae"])
def test_run_epoch_equals_step_loop(cuda, fam, device_keys):
    from d3p_b200 import optimizers
    opt = optimizers.RMSPropMomentum(optimizers.exponential_decay(2e-3, 2, 0.5), gamma=0.8)
    s, st0, get, bst = _epoch_setup(fam, opt)
    a, la = _stepwise(s, st0, get, bst, 3, 6)
    # two consecutive calls, the second with first_step > 0: the schedule follows the optimizer's counter (0 .. 5),
    # not the batch index (3 .. 8)
    b1, s1 = s.run_epoch(st0, get, bst, 2, first_step=3, device_keys=device_keys)
    b, s2 = s.run_epoch(b1, get, bst, 4, first_step=5, device_keys=device_keys)
    _same(a, b)
    assert [float(v) for v in torch.cat([s1, s2])[:, 0].cpu()] == la
    # and the whole trajectory depends on the schedule: a constant step size ends elsewhere
    s.optim = optimizers.RMSPropMomentum(2e-3, gamma=0.8)
    c, _ = s.run_epoch(st0, get, bst, 6, first_step=3, device_keys=device_keys)
    assert not torch.equal(c.optim_state.flat, b.optim_state.flat)


@pytest.mark.parametrize("fam", ["meanfield", "vae"])
def test_run_epoch_with_python_callable_schedule(cuda, fam):
    """A lambda step size cannot run inside the C driver: run_epoch takes the step loop and returns its result."""
    from d3p_b200 import optimizers
    opt = optimizers.Momentum(lambda i: 1e-3 / (1.0 + i), 0.9)
    assert not opt.fused_epoch
    s, st0, get, bst = _epoch_setup(fam, opt)
    a, la = _stepwise(s, st0, get, bst, 2, 4)
    b, stats = s.run_epoch(st0, get, bst, 4, first_step=2)
    _same(a, b)
    assert [float(v) for v in stats[:, 0].cpu()] == la


def _sharded_run(make_fam, data, clip, world, opt_factory, steps=3):
    import d3p_b200.random as rng
    from d3p_b200 import minibatch as mb, models, parallel, svi as dsvi
    N = len(data[0])
    fams = [make_fam() for _ in range(world)]
    wins = []
    if world > 1:
        wins = parallel.PeerWindow.local_group(world, fams[0].n_params, max_records=N)
        for w in wins:
            w.set_timeout_ms(4000)
    svis = []
    for r in range(world):
        s = dsvi.DPSVI(fams[r].model, fams[r].guide, opt_factory(), models.Trace_ELBO(), clip, 1.0, num_obs_total=N)
        if world > 1:
            parallel.shard_dpsvi(s, window=wins[r])
        svis.append(s)
    init, get = mb.poisson_batchify_data(data, 0.05, .99)
    key, k_init, k_fetch = rng.split(rng.PRNGKey(5), 3)
    _, bst = init(k_fetch)
    batch, mask = get(0, bst)
    states = [s.init(k_init, *batch) for s in svis]
    streams = [torch.cuda.Stream() for _ in range(world)]
    torch.cuda.synchronize()
    for i in range(steps):
        batch, mask = get(i, bst)
        torch.cuda.synchronize()
        ctx = [None] * world
        # all ranks' step kernels, then all ranks' finalize kernels (which wait for each other), as
        # tests/test_gpu_comm_loopback.py does on one device
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                ctx[r] = svis[r]._update_launch_step(states[r], batch, mask)
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                states[r], _ = svis[r]._update_finalize(ctx[r])
        torch.cuda.synchronize()
    for w in wins:
        assert w.timeouts() == 0
    out = [(st.optim_state.flat.clone(), st.optim_state.m.clone(), st.optim_state.v.clone()) for st in states]
    for w in wins:
        w.close()
    return out


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_replicas_identical(cuda, world):
    from d3p_b200 import models, optimizers
    g = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn((3000, 64), device=cuda, generator=g)
    y = (torch.rand(3000, device=cuda, generator=g) < 0.5).to(torch.int32)
    Xv = (torch.rand((3000, 16, 16), device=cuda, generator=g) < 0.3).float()
    opt = lambda: optimizers.RMSPropMomentum(optimizers.inverse_time_decay(1e-3, 1, 0.5), gamma=0.8)   # noqa: E731
    for name, make_fam, data, clip in (("logreg", lambda: models.LogisticRegression(64), (X, y), 1.0),
                                       ("vae", lambda: models.VAE(256, 64, 8, init_std=0.1), (Xv,), 5.0)):
        (ref,) = _sharded_run(make_fam, data, clip, 1, opt)
        reps = _sharded_run(make_fam, data, clip, world, opt)
        for r in range(world):
            for a, b in zip(reps[r], reps[0]):
                assert torch.equal(a, b), f"{name}: replica {r} differs from replica 0"
        for a, b, tag in zip(reps[0], ref, "xmv"):
            assert_rel(a, b, rtol=RTOL, what=f"{name} sharded {tag}")


def test_refusals_launch_nothing(cuda):
    """Every invalid descriptor returns its code from the finalize and from the epoch driver, and no kernel runs."""
    from d3p_b200 import _native as _n, optimizers
    lib = _n.lib()
    P = 64
    part = torch.zeros(P + 2, device=cuda)
    x, m, v, g = (torch.full((P,), 7.0, device=cuda) for _ in range(4))
    S = _n.OPT_SCHEDULED

    def desc(kind, **kw):
        od = _n.OptimDesc(kind, 0.1, 0.9, 0.999, 1e-8, 0)
        for k, val in kw.items():
            setattr(od, k, val)
        return od

    cases = [(desc(9), (x, m, v), -3), (desc(_n.OPT_NONE | S), (x, m, v), -1), (desc(_n.OPT_ADADP | S), (x, m, v), -1),
             (desc(_n.OPT_MOMENTUM), (x, None, v), -1), (desc(_n.OPT_RMSPROP), (x, m, None), -1),
             (desc(_n.OPT_ADAGRAD), (x, m, None), -1), (desc(_n.OPT_RMSPROP_MOMENTUM), (x, None, v), -1),
             (desc(_n.OPT_CLIPPED_ADAM, clip_norm=10.0), (x, None, v), -1),
             (desc(_n.OPT_CLIPPED_ADAM, clip_norm=0.0), (x, m, v), -1),
             (desc(_n.OPT_CLIPPED_ADAM, clip_norm=float("nan")), (x, m, v), -1),
             (desc(_n.OPT_ADAM | S, schedule=_n.SCHED_EXPONENTIAL, decay_steps=0.0), (x, m, v), -1),
             (desc(_n.OPT_SGD | S, schedule=_n.SCHED_POLYNOMIAL, decay_steps=-2.0), (x, m, v), -1),
             (desc(_n.OPT_SGD | S, schedule=_n.SCHED_PIECEWISE, n_boundaries=17), (x, m, v), -1),
             (desc(_n.OPT_SGD | S, schedule=11), (x, m, v), -3)]
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for od, (px, pm, pv), code in cases:
            rc = lib.d3p_perturb_finalize_f32(_n.ptr(part), 1, P, 1, None, 0.0, 1.0, 1.0, 0, _n.ptr(g), C.byref(od),
                                              _n.ptr(px), _n.ptr(pm), _n.ptr(pv), None, None, _n.stream_ptr())
            assert rc == code, (od.kind, rc, code)
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert kernels == [], kernels
    for t in (x, m, v, g):
        assert bool((t == 7.0).all())
    # the epoch driver refuses before its first step kernel: donated state stays as it was
    s, st0, get, bst = _epoch_setup("meanfield", optimizers.ClippedAdam(1e-3, clip_norm=-1.0))
    s.donate_state = True
    before = st0.optim_state.flat.clone()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with pytest.raises(_n.D3PNativeError, match="code -1"):
            s.run_epoch(st0, get, bst, 3)
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "d3p" in e.name]
    assert kernels == [], kernels
    assert torch.equal(st0.optim_state.flat, before)
