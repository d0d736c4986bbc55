"""The VAE step, evaluate and epoch paths (csrc/vae.cu) on real-valued inputs and on saturated decoder logits, against
the autodiff oracle (oracle/vae.py: vmap(grad) of the per-example ELBO with numpyro's clamp_probs) and, at the full
784-400-20 shape, against oracle.vae.explicit_clipped_sum.

Real-valued X.  vae_prep_x_kernel writes every row of X twice, unchanged (x_hi) and as its remainder below TF32
(x_lo = x - tf32_hi(x)), and raises a device flag when some x_lo of a valid row is non-zero.  The two GEMMs that read
X run their lo MMA only under that flag: G1 (pre1 = X W1) then loads four TMA operands per stage, GW1 ([X | 1]^T
(c delta1), dW1 / db1) loads the lo part of A beside the in-kernel hi / lo split of B.  0 and 1 are exact in TF32, so
binary data never raises the flag.  Grey levels k / 255 and uniform [0, 1) values have lo parts of up to 2^-10
relative (tf32_hi truncates), far above the 1e-5 bar: dropping them anywhere shows.

Saturated logits.  EpiFwd5 reproduces numpyro's clamp_probs = jnp.clip(p, tiny, 1 - eps) with jax's gradient rule:
factor 1 inside the clip, 1/2 at a bound, 0 outside.  Logits of +-40 and +-100 put p outside the clip (+40: p rounds
to 1; -100: exp(100) overflows float32, p = 0); a logit of 16.1 puts p exactly on 1 - eps = 1 - 2^-23.

Comparisons as in tests/test_gpu_vae.py: per-example ghost norms and losses at 1e-5 relative, the step's partial rows
summed in float64 and compared leaf by leaf element-wise (helpers/tolerance.py, 1e-5), the loss / count columns, and
the parameters after one SGD(1) step with dp_scale = 0 (they move by exactly the clipped-sum gradient).
"""
import numpy as np
import pytest
import torch

from d3p_b200 import minibatch as mb, models, optimizers, svi as dsvi
from helpers.tolerance import l2_err, rel_err
from oracle import chacha, svi as osvi, threefry, vae as ovae
from test_gpu_batch_scale import _step_outputs, _strided

REL = 1e-5
EPS32 = 2.0 ** -23          # float32 eps: numpyro's upper clip bound is 1 - EPS32


# ---- data and parameter builders ------------------------------------------------------------------------------------
def tf32_hi(a):
    """tc::tf32_hi: the float32 value with the low 13 mantissa bits cleared"""
    return (np.ascontiguousarray(a, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def real_x(kind, B, D, seed):
    rs = np.random.RandomState(seed)
    if kind == "k255":                        # grey levels, as 8-bit image intensities come
        return (rs.randint(0, 256, (B, D)) / 255.0).astype(np.float32)
    assert kind == "uniform"
    return rs.rand(B, D).astype(np.float32)


def binary_x(B, D, seed):
    return (np.random.RandomState(seed).rand(B, D) < 0.35).astype(np.float32)


def batch_mask(B):
    """some masked rows (as tests/test_gpu_vae.py), the last row valid"""
    mask = np.ones(B, dtype=bool)
    mask[B // 3::5] = False
    mask[-1] = True
    return mask


def setup(D, H, Z, X, C, N=60000, seed=0, init_std=None, params=None):
    """Oracle and CUDA DPSVI with SGD(1) and dp_scale = 0 on the same float32 parameters (test_gpu_vae.make's
    initialisation unless ``params`` is given)."""
    if init_std is None:                     # as test_gpu_vae.make
        init_std = 0.1 if D <= 64 and H <= 400 else 0.03
    ofam = ovae.VAE(D, H, Z, N)
    p0 = ofam.init_params(seed, init_std) if params is None else params
    o = osvi.DPSVI(ofam, None, osvi.SGD(1.0), None, C, 0.0)
    fam = models.VAE(D, H, Z)
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.0), models.Trace_ELBO(), C, 0.0, num_obs_total=N)
    key = chacha.PRNGKey(11)
    return o, o.init(key, X, params=p0), s, s.init(key, torch.as_tensor(X).cuda(), params=p0)


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def prep_buffers(s, n_part, Bl):
    """x_hi, x_lo [Bl, D + 4] and the lo flag as vae_prep_x_kernel left them in the step's workspace.  Offsets of
    vae_layout (vae.cu): 256-byte aligned blocks partials [S, P + 2], W1 hi, W1 lo, W5 hi, W5 lo, X hi, X lo, flag.
    (A wrong offset cannot pass: x_hi is compared with X bit for bit.)"""
    fam = s.family
    D, H, P = fam.out_dim, fam.hidden_dim, fam.n_params
    blk = lambda n: (n * 4 + 255) // 256 * 64             # floats of an aligned block of n floats  # noqa: E731
    w = s._ws.view(-1)
    off = blk(n_part * (P + 2)) + 4 * blk(D * H)
    n = Bl * (D + 4)
    x_hi = w[off:off + n].view(Bl, D + 4).cpu().numpy()
    off += blk(n)
    x_lo = w[off:off + n].view(Bl, D + 4).cpu().numpy()
    off += blk(n)
    flag = int(w[off:off + 1].view(torch.int32).item())
    return x_hi, x_lo, flag


def check_prep(s, n_part, X, mask):
    """valid rows: x_hi = x bit for bit (no cast, no binarisation), x_lo = x - tf32_hi(x); masked rows all zero; the
    ones column; the flag set exactly when a valid row has a non-zero lo part."""
    B, D = X.shape
    x_hi, x_lo, flag = prep_buffers(s, n_part, B)
    Xm = np.where(mask[:, None], X, np.float32(0))
    lo = Xm - tf32_hi(Xm)
    assert np.array_equal(x_hi[:, :D].view(np.uint32), Xm.view(np.uint32)), "x_hi is not the batch as handed in"
    assert np.array_equal(x_lo[:, :D], lo), "x_lo is not x - tf32_hi(x)"
    assert np.all(x_hi[:, D] == 1) and np.all(x_hi[:, D + 1:] == 0) and np.all(x_lo[:, D:] == 0)
    assert flag == int(bool(np.any(lo != 0))), (flag, int(np.count_nonzero(lo)))
    return flag


# ---- one step against the autodiff oracle ---------------------------------------------------------------------------
def oracle_step(o, ost, X, mask):
    """-> per-example norms [B] (float64), per-example losses on the kernels' scale, clipped sum {name: [..]}"""
    B = X.shape[0]
    ost1, okeys = o._split_rng_key(ost, 2)
    _, opx_loss, opx, _, f = o._compute_per_example_gradients(ost1, okeys[0], X, mask=mask)
    onorm = np.sqrt(sum(np.sum(np.square(np.asarray(g, np.float64).reshape(B, -1)), axis=1) for g in opx.values()))
    _, oclipped = o._clip_gradients(ost1, opx)
    csum = {k: v.astype(np.float64).sum(0).ravel() for k, v in oclipped.items()}
    return onorm, np.asarray(opx_loss, np.float64) / f, csum


def check_step(tag, o, ost, s, st, X, Xd, mask, check_update=True):
    """One step of the CUDA path on the device batch Xd (the rows of X) against the oracle; returns the flag."""
    B = X.shape[0]
    onorm, oloss, csum = oracle_step(o, ost, X, mask)
    st1, keys = s._split_rng_key(st, 2)
    P = s.family.n_params
    tmask = _dev(mask)
    ws, norms, losses = _step_outputs(s, st1, keys[0], (Xd,), tmask, B, P)
    n_part = ws.numel() // (P + 2)
    flag = check_prep(s, n_part, X, mask)
    part = ws.view(n_part, P + 2).double().sum(0).cpu().numpy()
    norms, losses = norms.cpu().numpy().astype(np.float64), losses.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(norms[mask], onorm[mask], rtol=REL, err_msg=f"{tag}: per-example norms")
    np.testing.assert_allclose(losses[mask], oloss[mask], rtol=REL, err_msg=f"{tag}: per-example losses")
    assert np.all(norms[~mask] == 0) and np.all(losses[~mask] == 0), f"{tag}: written where no example is"
    for name, off, shape in s.family.layout():
        size = int(np.prod(shape)) if len(shape) else 1
        e = rel_err(part[off:off + size], csum[name])
        assert e < REL, (tag, name, e)
    assert part[P + 1] == mask.sum(), tag
    assert abs(part[P] - oloss[mask].sum()) <= REL * np.abs(oloss[mask]).sum(), (tag, part[P], oloss[mask].sum())
    if check_update:
        ost2, ol = o.update(ost, X, mask=mask)
        st2, loss = s.update(st, Xd, mask=tmask)
        assert np.isclose(float(loss), float(ol), rtol=REL), (tag, float(loss), float(ol))
        oref, got = o.get_params(ost2), s.get_params(st2)
        for k in oref:
            assert rel_err(got[k], oref[k]) < REL, (tag, k, rel_err(got[k], oref[k]))
    return flag


# ---- 1. real-valued X -----------------------------------------------------------------------------------------------
# (D, H, Z, B, kind, layout): the thin-layer shapes of tests/test_gpu_vae.py, padded (H % 8 == 4, 2Z % 8 != 0, Z = 32)
# and not; D + 1 = 129 / 257 leaves GW1's last 128-row M tile with the bias row alone; B is never a multiple of 16 (the
# warp-MMA CTA) or of 32 (the GEMM k-block).  Layout "c": aligned contiguous rows (vae_prep_x_kernel<true>); "b": a
# column slice 4 bytes past a 16-byte boundary with an odd row stride (vae_prep_x_kernel<false>).
REAL_CASES = [
    (36, 20, 3, 19, "k255", "c"), (36, 20, 3, 45, "uniform", "b"),
    (36, 24, 4, 21, "uniform", "c"), (36, 24, 4, 19, "k255", "b"),
    (64, 40, 20, 37, "k255", "c"), (64, 40, 20, 50, "uniform", "b"),
    (128, 40, 8, 45, "k255", "c"), (128, 40, 8, 61, "uniform", "b"),
    (256, 64, 8, 77, "uniform", "c"), (256, 64, 8, 33, "k255", "b"),
    (784, 400, 20, 300, "k255", "c"), (784, 400, 20, 300, "uniform", "b"),
    (36, 20, 4, 21, "uniform", "c"), (36, 24, 3, 19, "k255", "b"), (36, 20, 1, 23, "k255", "c"),
    (64, 44, 30, 37, "uniform", "b"), (64, 44, 32, 29, "k255", "c"), (64, 416, 32, 45, "uniform", "b"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("D,H,Z,B,kind,layout", REAL_CASES,
                         ids=[f"{d}-{h}-{z}-B{b}-{k}-{l}" for d, h, z, b, k, l in REAL_CASES])
def test_vae_real_valued_x_matches_oracle(cuda, D, H, Z, B, kind, layout):
    X = real_x(kind, B, D, seed=D + B)
    o, ost, s, st = setup(D, H, Z, X, C=2.0 if D > 64 else 0.5, seed=D)
    Xd = _strided(X, "b") if layout == "b" else _dev(X)
    if layout == "b":
        assert s._resolve_args((Xd,)).stride == D + 3, "the strided batch was copied to a contiguous array"
    flag = check_step(f"{D}-{H}-{Z} B={B} {kind} {layout}", o, ost, s, st, X, Xd, batch_mask(B))
    assert flag == 1


@pytest.mark.gpu
def test_vae_facade_hands_x_through_untouched(cuda):
    """A float32 batch of any shape [B, ...] reaches the kernels as it is: the resolved batch is the caller's memory
    (no cast, copy or binarisation), and the prep kernel's x_hi holds the same bits."""
    D, H, Z, B = 36, 24, 4, 19
    X = real_x("k255", B, D, seed=3)
    o, ost, s, st = setup(D, H, Z, X, C=0.5)
    Xd = _dev(X.reshape(B, 6, 6))
    b = s._resolve_args((Xd,))
    assert b.x.data_ptr() == Xd.data_ptr() and b.x.dtype == torch.float32 and b.stride == D
    mask = np.ones(B, dtype=bool)
    st1, keys = s._split_rng_key(st, 2)
    ws, _, _ = _step_outputs(s, st1, keys[0], (Xd,), _dev(mask), B, s.family.n_params)
    assert check_prep(s, ws.numel() // (s.family.n_params + 2), X, mask) == 1
    assert torch.equal(Xd.reshape(B, D).cpu(), torch.as_tensor(X))           # the caller's batch is not written


# ---- 2. the full shape against the float64 explicit oracle ----------------------------------------------------------
def test_vae_explicit_oracle_matches_autodiff_on_real_valued_x():
    """oracle.vae.explicit_clipped_sum (what the full-shape test below is held against) == vmap(grad) -> clip -> sum on
    grey-level and uniform X; tests/test_oracle_families.py pins it on binary X only.  Bounds as there: the autodiff
    side is float32."""
    for (D, H, Z, B, C, std, kind) in [(36, 24, 4, 16, 0.5, 0.1, "k255"), (64, 40, 8, 33, 3.0, 0.1, "uniform"),
                                       (196, 64, 20, 20, 10.0, 0.05, "k255")]:
        X = real_x(kind, B, D, seed=D)
        fam = ovae.VAE(D, H, Z, 1000)
        p0 = fam.init_params(0, std)
        o = osvi.DPSVI(fam, None, osvi.SGD(1.0), None, C, 0.0)
        st = o.init(chacha.PRNGKey(11), X, params=p0)
        st1, keys = o._split_rng_key(st, 2)
        mask = np.ones(B, bool)
        mask[3::4] = False
        _, pxl, pxg, n, f = o._compute_per_example_gradients(st1, keys[0], X, mask=mask)
        eps = fam.sample_eps(threefry.split(chacha.convert_to_jax_rng_key(keys[0]), B))["z"]
        loss, norm, cs = ovae.explicit_clipped_sum(p0, X, eps, C, mask, fam.site_scale, st.observation_scale)
        onorm = np.sqrt(sum(np.sum(np.square(g.reshape(B, -1).astype(np.float64)), axis=1) for g in pxg.values()))
        assert np.max(np.abs(norm - onorm)[mask] / onorm[mask]) < 2e-6, (D, kind)
        assert np.all(norm[~mask] == 0) and np.all(onorm[~mask] == 0)
        np.testing.assert_allclose(loss * st.observation_scale * f, pxl, rtol=2e-6, atol=0)
        _, clipped = o._clip_gradients(st1, pxg)
        for k in cs:
            ref = clipped[k].astype(np.float64).sum(0)
            assert np.max(np.abs(cs[k] - ref)) < 2e-6 * np.sqrt(np.mean(ref ** 2)) + 1e-12, (D, kind, k)


@pytest.mark.gpu
def test_vae_real_valued_full_shape_matches_explicit_oracle(cuda):
    """784-400-20 at B = 4096 (4 batch splits of the clipped-sum GEMMs, GW1 with its lo part of A loaded) on grey-level
    X, with the bounds of test_gpu_vae.test_vae_full_shape_matches_explicit_oracle: the extra lo MMA per k-step of G1
    and GW1 adds one more truncating accumulation of a product 2^-10 smaller than the hi product, which changes
    neither bound."""
    D, H, Z, B, N, C = 784, 400, 20, 4096, 60000, 200.0
    X = real_x("k255", B, D, seed=0)
    mask = np.ones(B, bool)
    mask[B // 3::5] = False
    ofam = ovae.VAE(D, H, Z, N)
    p0 = ofam.init_params(0, 0.03)
    fam = models.VAE(D, H, Z)
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.0), models.Trace_ELBO(), C, 0.0, num_obs_total=N)
    Xd, md = _dev(X.reshape(B, 28, 28)), _dev(mask)
    st = s.init(chacha.PRNGKey(11), Xd, params=p0)
    st1, keys = s._split_rng_key(st, 2)
    norms, loss = torch.zeros(B, device=cuda), torch.zeros(B, device=cuda)
    ws, n_part, _, P = s._run_step(st1, keys[0], (Xd,), md, px_norms=norms, px_loss=loss)
    assert P == 652824 and n_part == 4
    assert prep_buffers(s, n_part, B)[2] == 1
    part = ws.view(-1)[: n_part * (P + 2)].view(n_part, P + 2).double().sum(0).cpu().numpy()
    eps = ofam.sample_eps(threefry.split(chacha.convert_to_jax_rng_key(np.asarray(keys[0])), B))["z"]
    ref_loss, ref_norm, ref_sum = ovae.explicit_clipped_sum(p0, X, eps, C, mask, ofam.site_scale, st.observation_scale)
    assert 0.2 < np.mean(ref_norm[mask] > C) < 1.0            # the clip is active for part of the batch
    got_norm, got_loss = norms.cpu().numpy().astype(np.float64), loss.cpu().numpy().astype(np.float64)
    assert np.max(np.abs(got_norm - ref_norm)[mask] / ref_norm[mask]) < 2e-5
    assert np.max(np.abs(got_loss - ref_loss * st.observation_scale)[mask] / np.abs(ref_loss[mask])) < REL
    assert np.all(got_norm[~mask] == 0)
    assert part[P + 1] == mask.sum()
    assert abs(part[P] - ref_loss.sum() * st.observation_scale) < REL * abs(ref_loss.sum())
    for name, off, shape in fam.layout():
        size = int(np.prod(shape)) if len(shape) else 1
        got, ref = part[off:off + size], ref_sum[name].ravel()
        assert l2_err(got, ref) < REL, (name, l2_err(got, ref))
        assert rel_err(got, ref) < 2e-5, (name, rel_err(got, ref))


# ---- 3. which rows raise the flag -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("lane", [0, 1, 2, 3])
def test_vae_flag_from_last_example_alone(cuda, lane):
    """A binary batch whose last example has grey levels in the columns of one float4 lane only (the vector path of
    vae_prep_x_kernel tests each lane for a lo part): the flag is raised and that example matches the oracle."""
    D, H, Z, B = 64, 40, 8, 19
    X = binary_x(B, D, seed=lane)
    cols = np.arange(lane, D, 4)
    X[-1, cols] = real_x("k255", 1, cols.size, seed=10 + lane)[0]
    assert np.any(X[-1] != tf32_hi(X[-1])) and np.all(X[:-1] == tf32_hi(X[:-1]))
    o, ost, s, st = setup(D, H, Z, X, C=0.5, seed=lane)
    assert check_step(f"lane {lane}", o, ost, s, st, X, _dev(X), batch_mask(B)) == 1


@pytest.mark.gpu
def test_vae_flag_ignores_masked_rows(cuda):
    """The only real-valued example is masked out: its row is never read, the flag stays down, and the step matches
    the oracle."""
    D, H, Z, B = 64, 40, 8, 19
    X = binary_x(B, D, seed=7)
    X[4] = real_x("uniform", 1, D, seed=8)[0]
    mask = batch_mask(B)
    mask[4] = False
    o, ost, s, st = setup(D, H, Z, X, C=0.5)
    assert check_step("masked real row", o, ost, s, st, X, _dev(X), mask) == 0


@pytest.mark.gpu
def test_vae_flag_is_reset_every_step(cuda):
    """One DPSVI object and workspace through binary -> real-valued -> binary steps: each step's partial rows, norms and
    losses are bit-identical to the same step on a fresh object, and the flag follows the batch."""
    D, H, Z, B = 64, 40, 8, 37
    batches = [binary_x(B, D, seed=1), real_x("k255", B, D, seed=2), binary_x(B, D, seed=3)]
    mask = batch_mask(B)
    o, ost, s, st = setup(D, H, Z, batches[0], C=0.5)
    P = s.family.n_params
    st1, keys = s._split_rng_key(st, 2)
    for i, X in enumerate(batches):
        got = _step_outputs(s, st1, keys[0], (_dev(X),), _dev(mask), B, P)
        assert prep_buffers(s, got[0].numel() // (P + 2), B)[2] == (1 if i == 1 else 0), i
        _, _, fresh, fst = setup(D, H, Z, X, C=0.5)
        want = _step_outputs(fresh, st1, keys[0], (_dev(X),), _dev(mask), B, P)
        for g_, w_ in zip(got, want):
            assert torch.equal(g_, w_), i


# ---- 4. evaluate and run_epoch on real-valued data ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("D,H,Z,B", [(36, 20, 3, 50), (64, 40, 20, 333)])
def test_vae_evaluate_real_valued_x(cuda, D, H, Z, B):
    X = real_x("k255", B, D, seed=B)
    o, ost, s, st = setup(D, H, Z, X, C=10.0)
    want = o.evaluate(ost, X)
    got = float(s.evaluate(st, _dev(X)))
    assert np.isclose(got, want, rtol=REL), (got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", ["subsample", "poisson"])
def test_vae_run_epoch_real_valued_data(cuda, sampler):
    """run_epoch over a grey-level data set (gathered rows; with the Poisson sampler also padding slots) is bit-identical
    to get_batch + update step by step, and the first step matches the oracle."""
    D, H, Z, N, B = 64, 40, 8, 600, 45
    X = real_x("k255", N, D, seed=5).reshape(N, 8, 8)
    Xd = _dev(X)
    C = 2.0
    ofam = ovae.VAE(D, H, Z, N)
    p0 = ofam.init_params(0, 0.1)
    o = osvi.DPSVI(ofam, None, osvi.SGD(1.0), None, C, 0.0)
    fam = models.VAE(D, H, Z)
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.0), models.Trace_ELBO(), C, 0.0, num_obs_total=N)
    if sampler == "subsample":
        init, get = mb.subsample_batchify_data((Xd,), batch_size=B)
    else:
        init, get = mb.poisson_batchify_data((Xd,), B / N, 64)
    key = chacha.PRNGKey(5)
    k_init, k_fetch = chacha.split(key, 3)[1:]
    _, bst = init(k_fetch)
    st0 = s.init(k_init, Xd[:B], params=p0)
    n_steps, first_step = 4, 1
    st, losses = st0, []
    for i in range(first_step, first_step + n_steps):
        out = get(i, bst)
        batch, mask = (out, True) if sampler == "subsample" else out
        st, loss = s.update(st, *batch, mask=mask)
        losses.append(float(loss))
        if i == first_step:
            Xb = batch[0].tensor().cpu().numpy()
            if sampler == "subsample":
                m = np.ones(Xb.shape[0], bool)
            else:
                nv = int(batch[0].num_valid.item())
                m = mask.cpu().numpy().astype(bool) & (np.arange(Xb.shape[0]) < nv)
                assert nv < Xb.shape[0] and np.any(Xb[m] != tf32_hi(Xb[m]))          # padding slots, real values
            ost, oloss = o.update(o.init(k_init, Xb, params=p0), Xb, mask=m)
            assert np.isclose(float(loss), float(oloss), rtol=REL), (float(loss), float(oloss))
            oref, got = o.get_params(ost), s.get_params(st)
            for k in oref:
                assert rel_err(got[k], oref[k]) < REL, (k, rel_err(got[k], oref[k]))
    st_e, stats = s.run_epoch(st0, get, bst, n_steps, first_step=first_step)
    assert np.array_equal(np.asarray(st_e.rng_key), np.asarray(st.rng_key))
    assert torch.equal(st_e.optim_state.flat, st.optim_state.flat), "run_epoch must be bit-identical to stepwise"
    assert np.array_equal(stats[:, 0].cpu().numpy(), np.asarray(losses, np.float32))
    assert bool(torch.isfinite(st_e.optim_state.flat).all())


# ---- 5. saturated decoder logits ------------------------------------------------------------------------------------
# Per pixel a logit centre and the x values it is paired with.  x < 1 stays away from logits of about 3 to 15.5: there
# p is inside the clip but within a few hundred ulps of 1, and log(1 - p) inherits the float32 rounding of p next to 1
# (at a logit of 10, one ulp of p is 1e-3 of 1 - p), so neither the kernel nor a float32 reference is accurate there.
SAT_PIXELS = [(-100.0, (0.0, 0.5, 1.0)), (-40.0, (0.0, 0.5, 1.0)), (-3.0, (0.0, 0.5, 1.0)), (0.0, (0.0, 0.5, 1.0)),
              (3.0, (1.0,)), (40.0, (0.0, 0.5, 1.0)), (100.0, (0.0, 0.5, 1.0))]


def saturated_case(D, H, Z, B, at_bound, seed=0):
    """-> (X, params).  Saturated: W5 = 1e-3 randn, so every logit is within 0.05 of its pixel's centre b5; x = 0
    and x = 1 both at +40 (the clamp zeroes both gradients, the unclamped form gives 1 and 0), x = 1 at -100 (the
    lower bound zeroes -1).  At the bound: W5 = 0, b5 = 16.1, x = 0: 1 + exp(-16.1) rounds to 1 + 2^-23 and p to
    1 - 2^-23 exactly, numpyro's gradient factor is 1/2 and each pixel's loss -log(eps)."""
    rs = np.random.RandomState(seed)
    p = ovae.VAE(D, H, Z, 1).init_params(seed, 0.1)
    if at_bound:
        p[ovae.W5] = np.zeros((H, D), np.float32)
        p[ovae.B5] = np.full(D, 16.1, np.float32)
        return np.zeros((B, D), np.float32), p
    p[ovae.W5] = (rs.randn(H, D) * 1e-3).astype(np.float32)
    kinds = np.arange(D) % len(SAT_PIXELS)
    p[ovae.B5] = np.array([SAT_PIXELS[k][0] for k in kinds], np.float32)
    X = np.empty((B, D), np.float32)
    for j, k in enumerate(kinds):
        xs = SAT_PIXELS[k][1]
        X[:, j] = [xs[(i + j) % len(xs)] for i in range(B)]
    return X, p


@pytest.mark.gpu
@pytest.mark.parametrize("D,H,Z,B", [(36, 20, 3, 19), (64, 40, 8, 37)])
@pytest.mark.parametrize("at_bound", [False, True], ids=["saturated", "at_bound"])
def test_vae_saturated_logits_match_oracle(cuda, D, H, Z, B, at_bound):
    X, p0 = saturated_case(D, H, Z, B, at_bound)
    mask = batch_mask(B)
    o, ost, s, st = setup(D, H, Z, X, C=3.0, params=p0)
    # the oracle's premises, in its own float32 arithmetic
    logits = torch.tensor(np.array([16.1, 40.0, -100.0], np.float32))
    assert torch.sigmoid(logits).tolist() == [1.0 - EPS32, 1.0, 0.0]
    onorm, _, csum = oracle_step(o, ost, X, mask)
    db5 = csum[ovae.B5]
    if at_bound:
        # factor 1/2, neither 0 (outside the clip) nor 1 (inside): db5 is half of p - x = 1 - eps, summed with the
        # examples' clip factors
        c = np.minimum(1.0, 3.0 / onorm[mask])
        np.testing.assert_allclose(db5, 0.5 * (1 - EPS32) * c.sum(), rtol=1e-6)
    else:
        x40 = [j for j in range(D) if SAT_PIXELS[j % len(SAT_PIXELS)][0] >= 40.0]
        assert np.all(db5[x40] == 0)                               # clamped: no gradient whatever x is
        for x in (0.0, 1.0):
            assert np.any(X[mask][:, x40] == x)
        lo = [j for j in range(D) if SAT_PIXELS[j % len(SAT_PIXELS)][0] == -100.0]
        assert np.all(db5[lo] == 0) and np.any(X[mask][:, lo] == 1.0)
    check_step("at bound" if at_bound else "saturated", o, ost, s, st, X, _dev(X), mask)
