"""The step, evaluate and clipping kernels at batch sizes where every warp or CTA handles many examples, and on
strided / unaligned batch arrays, against plain float64 references of the same operations.

The fused step kernels run on ``2 * SM`` CTAs of 8 warps (``launch.cuh: sm_count()``), so ``T = 2 * SM * 8`` warps
(2368 on a B200).  Every batch size here is written as a multiple of ``T`` (or of the CTA count) plus a remainder and
derived from the device, so that each case crosses the same boundary on any part: several examples per warp in the
vectorised kernel's 16-example tiles and lane groups, a second grid-stride pass of the generic kernel, several
examples per CTA of the mixture kernel, several rows per warp of the evaluate kernels.

References (float64, computed chunk by chunk so that no ``[B, P]`` float64 array is ever held):
  * guide noise from the oracle: ``threefry.split(convert_to_jax_rng_key(step_key), B)[positions]`` -> ``sample_eps``;
  * per-example gradients by autodiff of the oracle's ``neg_elbo`` (``vmap(grad_and_value)``) on the same float32
    parameters, noise and data, evaluated in float64 - independent of the kernels' closed-form algebra;
  * clipping ``c_i = 1 / max(1, |g_i| / C)``; masked / padding positions have weight 0 and are not counted.

Tolerances (tests/helpers/tolerance.py): clipped sums element-wise 1e-5 with the rms of the whole vector as floor,
loss sums 1e-5 relative, counts exact; per-example norms exactly 0 where no example is, ``assert_rel`` elsewhere, and
1e-5 of each norm on well-conditioned examples.
"""
import numpy as np
import pytest
import torch

from helpers.tolerance import assert_rel, rel_err
from oracle import chacha, families as ofam, gmm as ogmm, threefry

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _sm():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _T():
    """warps of the fused step kernels' grid: 2 CTAs of 8 warps per SM"""
    return 2 * _sm() * 8


def _flat_names(p):
    return sorted(p)


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def _partial_sum(ws, n_part, P):
    """the step's CTA partial rows [n_part, P + 2] added in float64"""
    return ws.view(-1)[:n_part * (P + 2)].view(n_part, P + 2).double().sum(0).cpu().numpy()


# ---- float64 reference of one clipped-sum step -----------------------------------------------------------------
def _reference(ofm, p, args, weight, jax_key, C_, obs, chunk=2048, eps_params=None):
    """One step's per-example gradients, norms and losses in float64 for the positions with ``weight`` True, clipped
    at C_ and summed.  ``args``: the batch arrays in position order.  -> dict(sum [P], loss, count, norms [B],
    losses [B]); norms / losses are 0 at positions without an example."""
    B = len(weight)
    names = _flat_names(p)
    P = sum(np.asarray(p[k]).size for k in names)
    keys = threefry.split(jax_key, B)          # split(key, B) depends on the total B: split once, slice by position
    tp = {k: torch.tensor(np.asarray(v, np.float32)).double() for k, v in p.items()}

    def loss(prm, e, *xi):
        return ofm.neg_elbo(prm, e, *(a.unsqueeze(0) for a in xi)) / obs

    fn = torch.func.vmap(torch.func.grad_and_value(loss), in_dims=(None, 0) + (0,) * len(args))
    acc = np.zeros(P)
    loss_sum, norms, losses = 0.0, np.zeros(B), np.zeros(B)
    pos = np.flatnonzero(weight)
    for lo in range(0, len(pos), chunk):
        sel = pos[lo:lo + chunk]
        eps = ofm.sample_eps(keys[sel]) if eps_params is None else ofm.sample_eps(keys[sel], eps_params)
        te = {k: torch.tensor(np.asarray(v)).double() for k, v in eps.items()}
        ta = [torch.tensor(np.asarray(a)[sel]) for a in args]
        ta = [t.double() if t.is_floating_point() else t for t in ta]
        g, v = fn(tp, te, *ta)
        G = torch.cat([g[k].reshape(len(sel), -1) for k in names], dim=1).numpy()
        nr = np.sqrt(np.sum(G * G, axis=1))
        c = 1.0 / np.maximum(1.0, nr / C_)
        acc += c @ G
        norms[sel] = nr
        losses[sel] = v.numpy() * obs          # px_loss is reported on the observation scale (svi.py:306)
        loss_sum += float(np.sum(v.numpy() * obs))
    return dict(sum=acc, loss=loss_sum, count=len(pos), norms=norms, losses=losses)


def _check_step(tag, part, P, ref, norms=None, losses=None, weight=None, well=None):
    assert part[P + 1] == ref["count"], f"{tag}: count {part[P + 1]} != {ref['count']}"
    assert_rel(part[:P], ref["sum"], rtol=RTOL, what=f"{tag}: clipped sum")
    assert abs(part[P] - ref["loss"]) <= RTOL * abs(ref["loss"]), f"{tag}: loss sum {part[P]} vs {ref['loss']}"
    if norms is not None:
        assert np.all(norms[~weight] == 0) and np.all(losses[~weight] == 0), f"{tag}: written where no example is"
        assert np.all(norms[weight] > 0), f"{tag}: an example's norm is missing"
        assert_rel(norms[weight], ref["norms"][weight], rtol=RTOL, what=f"{tag}: per-example norms")
        assert_rel(losses[weight], ref["losses"][weight], rtol=RTOL, what=f"{tag}: per-example losses")
        w = weight if well is None else (weight & well)
        e = np.max(np.abs(norms[w] - ref["norms"][w]) / ref["norms"][w])
        assert e < RTOL, f"{tag}: per-example norm relative error {e:.3e} on well-conditioned examples"


# ---- 1. mean-field step: every kernel instantiation with several examples per warp ----------------------------
def _mf_setup(kind, guide, d, B, seed, N=100_000, lr=1.0):
    """DPSVI (SGD(1), dp_scale = 0) and oracle family for a mean-field family, data and parameters that keep the
    logits moderate (|z| ~ 2: rows of norm 2) so that no per-example gradient is a saturated logit's rounding."""
    from d3p_b200 import models, optimizers, svi
    rs = np.random.RandomState(seed)
    if kind == "logreg":
        fam, ofm = models.LogisticRegression(d, guide=guide), ofam.LogisticRegression(d, N, guide=guide)
        X = (rs.randn(B, d) * (2.0 / np.sqrt(d))).astype(np.float32)
        args = (X, (rs.rand(B) < .5).astype(np.int32))
        C_ = 1.0
        p = {k: np.asarray(rs.randn(*v.shape) * .2, dtype=np.float32) for k, v in fam.init_params().items()}
    else:
        fam, ofm = models.GaussianMean(d, guide=guide), ofam.GaussianMean(d, N, guide=guide)
        args = ((1.0 + .1 * rs.randn(B, d)).astype(np.float32),)
        C_ = 1.0
        p = {}
        for k, v in fam.init_params().items():
            if k.endswith("loc"):
                p[k] = (1.0 + .05 * rs.randn(*v.shape)).astype(np.float32)      # near the data
            else:
                base = np.log(.05) if guide == "hand" else float(np.log(np.expm1(.05)))
                p[k] = (base + .1 * rs.randn(*v.shape)).astype(np.float32)
    s = svi.DPSVI(fam.model, fam.guide, optimizers.SGD(lr), models.Trace_ELBO(), C_, 0., num_obs_total=N)
    return s, fam, ofm, p, args, C_, N


def _batch_inputs(args, B, rs, view):
    """-> (kernel batch arguments, device mask, weight): ~10 % of the positions masked; with ``view`` the batch is a
    BatchView of a permuted copy of the rows with a device-side valid count below B."""
    from d3p_b200.minibatch import BatchView
    mask = rs.rand(B) >= .1
    if view:
        # one padding slot: the last positions are the ones a second grid-stride pass or a short last tile reaches,
        # so the device-side count must not cut them all off
        n_valid = B - 1
        mask[n_valid - 2:n_valid] = True
    else:
        n_valid = B
        mask[-2:] = True
    weight = mask & (np.arange(B) < n_valid)
    if view:
        perm = rs.permutation(B).astype(np.int32)
        inv = np.argsort(perm).astype(np.int32)                  # source row inv[i] holds the example at position i
        idx = _dev(inv)
        nv = torch.tensor([n_valid], dtype=torch.int32, device="cuda")
        targs = [BatchView(_dev(a[perm]), idx, nv) for a in args]
    else:
        targs = [_dev(a) for a in args]
    return targs, _dev(mask), weight


# (kind, guide, d, kernel path, B = mult * T + add, BatchView input, also sharded over 3 position ranges)
MF_CASES = [
    ("logreg", "hand", 1024, "vec-lpe32", (16, 5), False, True),     # runs of 16 / 17: a full tile + a 1-example tile
    ("gauss", "auto", 512, "vec-lpe16-g2", (3.5, 0), True, False),   # partial tiles, pairs of one valid + one masked
    ("gauss", "hand", 256, "vec-lpe8-g4", (17, 1), False, True),     # the 4-group fold with every group non-zero
    ("logreg", "auto", 1024, "generic-32x32", (8, 3), True, False),  # joint 1025-element site: second grid-stride pass
    ("logreg", "hand", 100, "generic-16x4", (16, 17), False, False),  # SUB = 2, TILE = 8: second pass
    ("gauss", "hand", 7, "generic-1x4", (32, 33), True, False),      # SUB = 32, TILE = 1: second pass, smallest shape
]


def _mf_id(c):
    kind, guide, d, path, (m, a), view, shard = c
    return f"{kind}-{guide}-d{d}-{path}-B{m}T+{a}" + ("-view" if view else "") + ("-shard3" if shard else "")


@pytest.mark.parametrize("case", MF_CASES, ids=_mf_id)
def test_meanfield_step_many_examples_per_warp(cuda, case):
    kind, guide, d, path, (mult, add), view, shard = case
    B = int(mult * _T()) + add
    seed = d + int(10 * mult)
    s, fam, ofm, p, args, C_, N = _mf_setup(kind, guide, d, B, seed)
    rs = np.random.RandomState(seed + 1)
    targs, tmask, weight = _batch_inputs(args, B, rs, view)
    st = s.init(chacha.PRNGKey(seed), *[_dev(a) for a in args], params=p)
    _, (k_grad, _) = s._split_rng_key(st, 2)          # the key update() hands to the step kernel
    ref = _reference(ofm, p, args, weight, chacha.random_bits(k_grad, 32, (2,)), C_, float(N))
    P = fam.n_params
    tag = _mf_id(case)

    norms = torch.zeros(B, device=cuda)
    losses = torch.zeros(B, device=cuda)
    ws, n_part, _, _ = s._run_step(st, k_grad, targs, tmask, px_norms=norms, px_loss=losses)
    part = _partial_sum(ws, n_part, P)
    n_np, l_np = norms.cpu().numpy().astype(np.float64), losses.cpu().numpy().astype(np.float64)
    well = ref["norms"] > .25 * np.median(ref["norms"][weight])
    assert (weight & well).sum() > weight.sum() // 2
    _check_step(tag, part, P, ref, n_np, l_np, weight, well)

    if shard:         # three position ranges: their partial sums add up to the reference, not only to each other
        tot = np.zeros(P + 2)
        sn = torch.zeros(B, device=cuda)
        for r in range(3):
            s.shard = (r, 3, None)
            try:
                ws, n_part, _, _ = s._run_step(st, k_grad, targs, tmask, px_norms=sn)
                tot += _partial_sum(ws, n_part, P)
            finally:
                s.shard = None
        _check_step(tag + " sharded 3 ways", tot, P, ref)
        assert torch.equal(sn, norms)

    # one full update (the finalize kernel's reduction of the 2 * SM partial rows): with SGD(1) and dp_scale = 0 the
    # parameters move by obs_scale * clipped sum / n
    st2, loss = s.update(st, *targs, mask=tmask)
    moved = st.optim_state.flat.double().cpu().numpy() - st2.optim_state.flat.double().cpu().numpy()
    assert_rel(moved, ref["sum"] * N / ref["count"], rtol=RTOL, what=f"{tag}: update")
    f = np.float32(B) / np.float32(ref["count"])
    assert abs(float(loss) - ref["loss"] / B * f) <= RTOL * abs(ref["loss"] / B * f)


# ---- 2. mixture step with several examples per CTA -------------------------------------------------------------
def _gmm_setup(K, d, B, seed, C_=1.5, N=2000):
    from d3p_b200 import models, optimizers, svi
    rs = np.random.RandomState(seed)
    centers = rs.randn(K, d).astype(np.float32) * 3
    X = (centers[rs.randint(0, K, B)] + rs.randn(B, d)).astype(np.float32)
    p = {"alpha_log": (rs.randn(K) * 0.4).astype(np.float32), "mus_loc": (centers + rs.randn(K, d) * 0.5).astype(np.float32)}
    fam, ofm = models.GaussianMixture(K, d), ogmm.GaussianMixture(K, d, N)
    s = svi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.), models.Trace_ELBO(), C_, 0., num_obs_total=N)
    return s, fam, ofm, p, X, C_, N


# (K, d, B = mult * (2 SM) + add, BatchView input)
GMM_CASES = [(3, 2, (3, 37), False), (17, 7, (2, 5), True)]      # K = 17: not a multiple of the warp, n = 119 < 256


@pytest.mark.parametrize("K,d,bs,view", GMM_CASES, ids=[f"K{k}-d{d}-B{m}x2SM+{a}" + ("-view" if v else "")
                                                        for k, d, (m, a), v in GMM_CASES])
def test_gmm_step_many_examples_per_cta(cuda, K, d, bs, view):
    B = bs[0] * 2 * _sm() + bs[1]
    s, fam, ofm, p, X, C_, N = _gmm_setup(K, d, B, K * 10 + d)
    rs = np.random.RandomState(K)
    targs, tmask, weight = _batch_inputs((X,), B, rs, view)
    st = s.init(chacha.PRNGKey(K), _dev(X), params=p)
    _, (k_grad, _) = s._split_rng_key(st, 2)
    ref = _reference(ofm, p, (X,), weight, chacha.random_bits(k_grad, 32, (2,)), C_, float(N), chunk=256,
                     eps_params=p)
    P = fam.n_params
    norms = torch.zeros(B, device=cuda)
    losses = torch.zeros(B, device=cuda)
    ws, n_part, _, _ = s._run_step(st, k_grad, targs, tmask, px_norms=norms, px_loss=losses)
    _check_step(f"gmm K={K} d={d} B={B}", _partial_sum(ws, n_part, P), P, ref, norms.cpu().numpy().astype(np.float64),
                losses.cpu().numpy().astype(np.float64), weight)
    st2, _ = s.update(st, *targs, mask=tmask)
    moved = st.optim_state.flat.double().cpu().numpy() - st2.optim_state.flat.double().cpu().numpy()
    assert_rel(moved, ref["sum"] * N / ref["count"], rtol=RTOL, what="gmm update")


# ---- 3. evaluate over many rows per warp ------------------------------------------------------------------------
def _evaluate_f64(ofm, p, args, rng_key, N):
    """The oracle's DPSVI.evaluate (one guide draw for the whole batch, plate scale N / B) in float64."""
    key = threefry.split(chacha.convert_to_jax_rng_key(chacha.split(rng_key, 1)[0]), 2)[1]
    eps = ofm.sample_eps(key.reshape(1, 2), p) if getattr(ofm, "needs_params_for_eps", False) else ofm.sample_eps(key.reshape(1, 2))
    tp = {k: torch.tensor(np.asarray(v, np.float32)).double() for k, v in p.items()}
    te = {k: torch.tensor(np.asarray(v)[0]).double() for k, v in eps.items()}
    ta = [torch.tensor(np.asarray(a)) for a in args]
    ta = [t.double() if t.is_floating_point() else t for t in ta]
    B = len(args[0])
    ofm.num_obs_total = N / B
    try:
        return float(ofm.neg_elbo(tp, te, *ta))
    finally:
        ofm.num_obs_total = N


# (family, B = mult * T + add)
EVAL_CASES = [("logreg-hand-d1024", (16, 5)), ("gauss-auto-d37", (3, 1)), ("gmm-K17-d7", (3, 11))]


@pytest.mark.parametrize("what,bs", EVAL_CASES, ids=[f"{w}-B{m}T+{a}" for w, (m, a) in EVAL_CASES])
def test_evaluate_many_rows_per_warp(cuda, what, bs):
    B = bs[0] * _T() + bs[1]
    if what.startswith("gmm"):
        s, fam, ofm, p, X, _, N = _gmm_setup(17, 7, B, 3)
        args = (X,)
    else:
        kind, guide, d = what.split("-")
        s, fam, ofm, p, args, _, N = _mf_setup(kind, guide, int(d[1:]), B, 5)
    st = s.init(chacha.PRNGKey(12), *[_dev(a) for a in args], params=p)
    got = float(s.evaluate(st, *[_dev(a) for a in args]))
    want = _evaluate_f64(ofm, p, args, st.rng_key, float(N))
    assert abs(got - want) <= RTOL * abs(want), (what, B, got, want)


# ---- 4. the clipping C ABI (clip.cu) ------------------------------------------------------------------------------
def _clip_rows_data(B, P, C_, seed):
    """rows of norms log-uniform in [C / 10, 10 C] (some clipped, some not), a few all-zero rows"""
    rs = np.random.RandomState(seed)
    g = rs.randn(B, P)
    g /= np.maximum(np.linalg.norm(g, axis=1, keepdims=True), 1e-30)
    g *= C_ * np.exp(rs.uniform(np.log(.1), np.log(10.), size=(B, 1)))
    g[rs.rand(B) < .03] = 0
    return g.astype(np.float32), rs


CLIP_B = ["1", "7", "64", "65", "8SM+1", "5000"]
CLIP_P = [1, 31, 33, 2050, 70_000]
CLIP_CASES = [(b, P) for b in CLIP_B for P in CLIP_P
              if (5000 if b == "5000" else 1200 if b == "8SM+1" else int(b)) * P <= 20_000_000]


@pytest.mark.parametrize("b,P", CLIP_CASES, ids=[f"B{b}-P{P}" for b, P in CLIP_CASES])
def test_clip_and_sum_masked_finite_C(cuda, b, P):
    """d3p_clip_and_sum_f32 with a finite C, a mask and per-example losses, against float64 numpy."""
    from d3p_b200 import _native as _n
    lib = _n.lib()
    B = 8 * _sm() + 1 if b == "8SM+1" else int(b)
    C_ = 0.7
    g, rs = _clip_rows_data(B, P, C_, B * 7 + P)
    mask = rs.rand(B) >= .2
    if B > 1:
        mask[0] = True
    px_loss = rs.randn(B).astype(np.float32)
    need = lib.d3p_clip_and_sum_workspace_bytes(B, P)
    ws = torch.empty((need + 3) // 4, dtype=torch.float32, device=cuda)
    out = torch.full((P + 2,), float("nan"), device=cuda)
    dg, dl, dm = _dev(g), _dev(px_loss), _dev(mask.astype(np.uint8))
    _n.check(lib.d3p_clip_and_sum_f32(_n.ptr(dg), _n.ptr(dl), _n.ptr(dm), B, P, C_, _n.ptr(out), _n.ptr(ws), need,
                                      _n.stream_ptr()), "clip_and_sum")
    got = out.cpu().numpy().astype(np.float64)
    g64 = g.astype(np.float64)
    c = np.where(mask, 1.0 / np.maximum(1.0, np.linalg.norm(g64, axis=1) / C_), 0.0)
    want = c @ g64
    assert_rel(got[:P], want, rtol=RTOL, what=f"clip_and_sum B={B} P={P}")
    wl = float(np.sum(px_loss.astype(np.float64)[mask]))
    assert abs(got[P] - wl) <= RTOL * np.sum(np.abs(px_loss[mask])), (got[P], wl)
    assert got[P + 1] == mask.sum()


def test_clip_rows_grid_stride(cuda):
    """d3p_clip_rows_f32 at B = 5000 (> 8 SM rows: the grid-stride loop) with norms_d, against float64 numpy."""
    from d3p_b200 import _native as _n
    B, P, C_ = 5000, 2050, 0.7
    g, _ = _clip_rows_data(B, P, C_, 17)
    dg = _dev(g)
    norms = torch.full((B,), float("nan"), device=cuda)
    _n.check(_n.lib().d3p_clip_rows_f32(_n.ptr(dg), B, P, C_, _n.ptr(norms), _n.stream_ptr()), "clip_rows")
    g64 = g.astype(np.float64)
    nr = np.linalg.norm(g64, axis=1)
    want = g64 / np.maximum(1.0, nr / C_)[:, None]
    got_n = norms.cpu().numpy().astype(np.float64)
    assert np.all(got_n[nr == 0] == 0)
    assert np.max(np.abs(got_n[nr > 0] - nr[nr > 0]) / nr[nr > 0]) < RTOL
    assert rel_err(dg.cpu().numpy()[nr > 0], want[nr > 0], axis=0) < RTOL


VNORM_ORDS = [1, 3, 2.5, .5, np.inf, -np.inf, 0, -1]


@pytest.mark.parametrize("n", [1023, 1024, 1025, 1_000_003])
def test_vector_norm_orders(cuda, n):
    """d3p_vector_norm_f32 against np.linalg.norm in float64.  max / min / count are exact in float32.  The power sums
    are float32 sums of up to n / 1024 ~ 1000 terms per thread plus a 1024-way tree, each term with the ~2 ulp error of
    powf: a relative error of a few 1e-6 at n = 1e6 (worst case ~6e-5 if every rounding went one way), which the
    final power 1 / ord multiplies by 1 / |ord| - hence rtol 2e-5 * max(1, 1 / |ord|)."""
    from d3p_b200 import _native as _n
    rs = np.random.RandomState(n % 1000)
    x = (rs.randn(n) * np.exp(rs.uniform(-2, 2, n))).astype(np.float32)
    x[rs.rand(n) < .05] = 0                       # zeros for ord = 0
    nz = np.where(x == 0, np.float32(.5), x)      # no zero element: ord = -1 is a finite harmonic sum
    dx, dnz = _dev(x), _dev(nz)
    out = torch.empty(1, device=cuda)
    for ord_ in VNORM_ORDS:
        for arr, darr in ([(nz, dnz), (x, dx)] if ord_ == -1 else [(x, dx)]):
            _n.check(_n.lib().d3p_vector_norm_f32(_n.ptr(darr), n, float(ord_), _n.ptr(out), _n.stream_ptr()), "norm")
            got = float(out.cpu())
            with np.errstate(divide="ignore"):            # 0 ** -1 = inf -> norm 0, as in the kernel
                want = float(np.linalg.norm(arr.astype(np.float64), ord=ord_))
            if np.isinf(ord_) or ord_ == 0 or want == 0:
                assert got == want, (n, ord_, got, want)
            else:
                tol = 2e-5 * max(1.0, 1.0 / abs(ord_))
                assert abs(got - want) <= tol * abs(want), (n, ord_, got, want)


# ---- 5. strided and unaligned batch arrays ----------------------------------------------------------------------
def _strided(a, how):
    """the rows of ``a`` as a column slice of a wider device array: 'a' = row stride d + 4 from column 0 (an aligned
    base), 'b' = row stride d + 3 from column 1 (a base 4 bytes past a 16-byte boundary, stride % 4 != 0)"""
    B, d = a.shape
    extra, col = (4, 0) if how == "a" else (3, 1)
    big = torch.full((B, d + extra), float("nan"), device="cuda")
    v = big[:, col:col + d]
    v.copy_(_dev(a))
    assert v.stride(0) == d + extra and v.stride(1) == 1
    assert (v.data_ptr() % 16 == 0) == (how == "a")
    return v


def _assert_stride_reaches_kernel(s, args, d):
    # the facade must hand the column slice to the kernels as it is, not a contiguous copy
    assert s._resolve_args(args).stride != d, "the strided batch was copied to a contiguous array"


def _step_outputs(s, st, key, args, mask, B, P):
    norms = torch.zeros(B, device="cuda")
    losses = torch.zeros(B, device="cuda")
    ws, n_part, _, _ = s._run_step(st, key, args, mask, px_norms=norms, px_loss=losses)
    return ws.view(-1)[:n_part * (P + 2)].clone(), norms, losses


@pytest.mark.parametrize("kind,guide,d", [("logreg", "hand", 1024), ("gauss", "hand", 256)])
@pytest.mark.parametrize("how", ["a", "b"])
def test_meanfield_strided_batch(cuda, kind, guide, d, how):
    """(a): the vectorised kernel both times, so bit-identical to the contiguous batch; (b): the unaligned base sends
    the batch to the generic kernel, which is compared with the float64 reference instead."""
    B = 3 * 16 * 8 + 5
    s, fam, ofm, p, args, C_, N = _mf_setup(kind, guide, d, B, 31)
    rs = np.random.RandomState(32)
    mask = rs.rand(B) >= .1
    tmask = _dev(mask)
    st = s.init(chacha.PRNGKey(3), *[_dev(a) for a in args], params=p)
    _, (k_grad, _) = s._split_rng_key(st, 2)
    P = fam.n_params
    sargs = (_strided(args[0], how),) + tuple(_dev(a) for a in args[1:])
    _assert_stride_reaches_kernel(s, sargs, d)
    got = _step_outputs(s, st, k_grad, sargs, tmask, B, P)
    if how == "a":
        want = _step_outputs(s, st, k_grad, [_dev(a) for a in args], tmask, B, P)
        for g_, w_ in zip(got, want):
            assert torch.equal(g_, w_)
    else:
        ref = _reference(ofm, p, args, mask, chacha.random_bits(k_grad, 32, (2,)), C_, float(N))
        ws, norms, losses = got
        part = ws.view(-1, P + 2).double().sum(0).cpu().numpy()
        well = ref["norms"] > .25 * np.median(ref["norms"][mask])
        _check_step(f"{kind} d={d} strided (b)", part, P, ref, norms.cpu().numpy().astype(np.float64),
                    losses.cpu().numpy().astype(np.float64), mask, well)


@pytest.mark.parametrize("how", ["a", "b"])
def test_gmm_strided_batch(cuda, how):
    """the mixture kernel reads rows element by element: the same kernel either way, so bit-identical"""
    K, d = 3, 5
    B = 2 * 2 * _sm() + 3
    s, fam, ofm, p, X, C_, N = _gmm_setup(K, d, B, 41)
    mask = _dev(np.random.RandomState(42).rand(B) >= .1)
    st = s.init(chacha.PRNGKey(4), _dev(X), params=p)
    _, (k_grad, _) = s._split_rng_key(st, 2)
    sx = _strided(X, how)
    _assert_stride_reaches_kernel(s, (sx,), d)
    got = _step_outputs(s, st, k_grad, (sx,), mask, B, fam.n_params)
    want = _step_outputs(s, st, k_grad, (_dev(X),), mask, B, fam.n_params)
    for g_, w_ in zip(got, want):
        assert torch.equal(g_, w_)


@pytest.mark.parametrize("D,H,Z", [(36, 24, 4), (784, 400, 20)])
@pytest.mark.parametrize("how", ["a", "b"])
def test_vae_strided_batch(cuda, D, H, Z, how):
    """(a): vae_prep_x_kernel<true> both times, bit-identical; (b): the unaligned rows go through
    vae_prep_x_kernel<false>, which sums |x|^2 in another order - compared with the oracle's clipped sum."""
    from test_gpu_vae import make
    B, C_ = 48, 2.0
    X, o, ost, s, st = make(D, H, Z, 60000, B, C_, 0.0, optim="sgd", seed=D)
    X2 = X.reshape(B, D)
    mask = np.ones(B, dtype=bool)
    mask[B // 3::5] = False
    tmask = _dev(mask)
    sx = _strided(X2, how)
    _assert_stride_reaches_kernel(s, (sx,), D)
    st1, keys = s._split_rng_key(st, 2)
    P = s.family.n_params
    got = _step_outputs(s, st1, keys[0], (sx,), tmask, B, P)
    if how == "a":
        want = _step_outputs(s, st1, keys[0], (_dev(X2),), tmask, B, P)
        for g_, w_ in zip(got, want):
            assert torch.equal(g_, w_)
        return
    ost1, okeys = o._split_rng_key(ost, 2)
    _, opx_loss, opx, _, f = o._compute_per_example_gradients(ost1, okeys[0], X, mask=mask)
    onorm = np.sqrt(sum(np.sum(np.square(np.asarray(g, np.float64).reshape(B, -1)), axis=1) for g in opx.values()))
    _, oclipped = o._clip_gradients(ost1, opx)
    ws, norms, losses = got
    part = ws.view(-1, P + 2).double().sum(0).cpu().numpy()
    for name, off, shape in s.family.layout():
        size = int(np.prod(shape)) if len(shape) else 1
        assert_rel(part[off:off + size], oclipped[name].astype(np.float64).sum(0).ravel(), rtol=RTOL, what=name)
    assert part[P + 1] == mask.sum()
    np.testing.assert_allclose(norms.cpu().numpy()[mask], onorm[mask], rtol=RTOL)
    np.testing.assert_allclose(losses.cpu().numpy()[mask], (opx_loss / f)[mask], rtol=RTOL)
    assert np.all(norms.cpu().numpy()[~mask] == 0)


def test_evaluate_and_run_epoch_on_strided_data(cuda):
    """DPSVI.evaluate of an unaligned column slice and run_epoch over a strided data set: the same kernels as for the
    contiguous arrays (the evaluate kernel and the generic step kernel read rows element by element), so the
    results are bit-identical."""
    from d3p_b200 import minibatch as mb
    d, B = 1024, 3 * _T() + 7
    s, fam, ofm, p, args, C_, N = _mf_setup("logreg", "hand", d, B, 51)
    st = s.init(chacha.PRNGKey(5), *[_dev(a) for a in args], params=p)
    sx, y = _strided(args[0], "b"), _dev(args[1])
    _assert_stride_reaches_kernel(s, (sx, y), d)
    assert float(s.evaluate(st, sx, y)) == float(s.evaluate(st, _dev(args[0]), y))

    d, Nr = 100, 20_000
    s, fam, ofm, p, args, C_, N = _mf_setup("logreg", "hand", d, Nr, 52, N=Nr, lr=1e-5)     # 4 steps that stay finite
    runs = []
    for strided in (True, False):
        X = _strided(args[0], "b") if strided else _dev(args[0])
        init, get = mb.poisson_batchify_data((X, _dev(args[1])), .02, .99)
        if strided:
            # poisson_batchify_data keeps a contiguous copy of the data set; run_epoch takes the data set from the
            # batchifier's spec, so the strided array goes in there to put the epoch kernels' stride under test
            assert get.spec["dataset"][0].stride(0) == d
            get.spec["dataset"] = (X, get.spec["dataset"][1])
        _, bst = init(chacha.PRNGKey(6))
        st = s.init(chacha.PRNGKey(7), _dev(args[0][:10]), _dev(args[1][:10]), params=p)
        s._epoch_plan = None
        st2, stats = s.run_epoch(st, get, bst, 4)
        if strided:
            assert s._epoch_plan[3] != d, "run_epoch was not handed the strided data set"
        runs.append((st2.optim_state.flat.clone(), stats.clone()))
    assert bool(torch.isfinite(runs[0][0]).all()) and bool(torch.isfinite(runs[0][1]).all())
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
