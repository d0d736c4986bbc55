"""VAE path (ghost-norm clip + tcgen05 clipped-sum GEMMs, csrc/vae.cu) against the CPU oracle
(oracle/vae.py: literally vmap(grad) of the per-example ELBO + clip + mean + noise + optimizer)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import d3p_b200.random as rng
from d3p_b200 import models, optimizers, svi as dsvi
from helpers.tolerance import l2_err, rel_err as ew_rel_err
from oracle import chacha, svi as osvi, threefry, vae as ovae

pytestmark = pytest.mark.gpu

REL = 1e-5   # BASELINE.json: clipped-sum gradients and final parameters fp32 within 1e-5 relative


def make(D, H, Z, N, B, C, dp_scale, optim="adam", seed=0, init_std=None):
    if init_std is None:     # keep the logits O(1) (the example initialises with std 1e-2, vae.py:80-103): at 0.1,
        # 64-416-32 puts two thirds of them past +-3, where float32 log(1 - p) is not good to 1e-5 (test_gpu_vae_inputs.py)
        init_std = 0.1 if D <= 64 and H <= 400 else 0.03
    rs = np.random.RandomState(seed)
    side = int(np.sqrt(D))
    shape = (B, side, side) if side * side == D else (B, D)
    X = (rs.rand(*shape) < 0.35).astype(np.float32)
    ofam = ovae.VAE(D, H, Z, N)
    p0 = ofam.init_params(seed, init_std)
    oopt = osvi.Adam(1e-3) if optim == "adam" else osvi.SGD(1.0)
    o = osvi.DPSVI(ofam, None, oopt, None, C, dp_scale)
    fam = models.VAE(D, H, Z)
    gopt = optimizers.Adam(1e-3) if optim == "adam" else optimizers.SGD(1.0)
    s = dsvi.DPSVI(fam.model, fam.guide, gopt, models.Trace_ELBO(), C, dp_scale, num_obs_total=N)
    key = chacha.PRNGKey(11)
    return X, o, o.init(key, X, params=p0), s, s.init(key, torch.as_tensor(X).cuda(), params=p0)


def rel_err(got, ref):
    return float(np.max(np.abs(got - ref)) / max(float(np.max(np.abs(ref))), 1e-30))


# Shapes of the warp-MMA thin-layer kernels (vae.cu): H % 8 == 0 and Z % 4 == 0 tile their 8 x 8 blocks exactly; H % 8 == 4
# (36-20-*, 64-44-*), 2Z % 8 != 0 (Z = 1, 3, 30) and Z = 32 are padded; 64-416-32 runs the backward kernel with over
# 48 KB of shared memory.  B is mostly not a multiple of 16 (the kernels' rows per CTA).
@pytest.mark.parametrize("D,H,Z,B", [(36, 24, 4, 16), (36, 20, 3, 19), (64, 40, 20, 37), (784, 400, 20, 48),
                                     (36, 20, 4, 21), (36, 24, 3, 19), (36, 20, 1, 23), (64, 44, 30, 37),
                                     (64, 44, 32, 29), (64, 416, 32, 45)])
def test_vae_ghost_norms_and_losses(cuda, D, H, Z, B):
    X, o, ost, s, st = make(D, H, Z, 1000, B, 10.0, 1.0)
    ost1, okeys = o._split_rng_key(ost, 2)
    _, opx_loss, opx_grads, n, f = o._compute_per_example_gradients(ost1, okeys[0], X)
    onorm = np.sqrt(sum(np.sum(np.square(g.reshape(B, -1)), axis=1) for g in opx_grads.values()))
    st1, keys = s._split_rng_key(st, 2)
    px_norms = torch.zeros(B, device=cuda)
    px_loss = torch.zeros(B, device=cuda)
    s._run_step(st1, keys[0], (torch.as_tensor(X).cuda(),), True, px_norms=px_norms, px_loss=px_loss)
    np.testing.assert_allclose(px_norms.cpu().numpy(), onorm, rtol=REL)
    np.testing.assert_allclose(px_loss.cpu().numpy(), opx_loss, rtol=REL)


def poison_workspace(s, B):
    """Fill the step workspace of a B-row batch, which the next step reuses, with NaN."""
    desc = s.family.desc(s._num_obs_total())
    s._workspace(s.family._step_workspace_bytes(desc, B, ctypes.c_uint32(0))).fill_(float("nan"))


def check_clipped_sum(D, H, Z, B, C, poison=False):
    """dp_scale = 0 and SGD(1): parameters move by exactly the clipped-sum gradient.  poison: every step starts from a
    workspace full of NaN."""
    X, o, ost, s, st = make(D, H, Z, 60000, B, C, 0.0, optim="sgd")
    mask = np.ones(B, dtype=bool)
    mask[B // 3::5] = False
    ost2, oloss = o.update(ost, X, mask=mask)
    if poison:
        poison_workspace(s, B)
    st2, loss = s.update(st, torch.as_tensor(X).cuda(), mask=torch.as_tensor(mask).cuda())
    assert np.isclose(float(loss), float(oloss), rtol=REL)
    oref, got = o.get_params(ost2), s.get_params(st2)
    for k in oref:
        assert ew_rel_err(got[k], oref[k]) < REL, (k, ew_rel_err(got[k], oref[k]))
    # the clipped sum itself (not a difference of rounded parameters): the partial rows of the step kernels
    ost1, okeys = o._split_rng_key(ost, 2)
    _, _, opx, _, _ = o._compute_per_example_gradients(ost1, okeys[0], X, mask=mask)
    _, oclipped = o._clip_gradients(ost1, opx)
    st1, keys = s._split_rng_key(st, 2)
    if poison:
        poison_workspace(s, B)
    ws, n_part, _, P = s._run_step(st1, keys[0], (torch.as_tensor(X).cuda(),), torch.as_tensor(mask).cuda())
    part = ws.view(-1)[: n_part * (P + 2)].view(n_part, P + 2).double().sum(0).cpu().numpy()
    for name, off, shape in s.family.layout():
        size = int(np.prod(shape)) if len(shape) else 1
        ref = oclipped[name].astype(np.float64).sum(0).ravel()
        assert ew_rel_err(part[off:off + size], ref) < REL, (name, ew_rel_err(part[off:off + size], ref))


@pytest.mark.parametrize("D,H,Z,B,C", [(36, 24, 4, 16, 0.5), (36, 20, 3, 19, 0.5), (64, 40, 20, 37, 3.0), (784, 400, 20, 48, 10.0),
                                        (784, 400, 20, 300, 2.0), (36, 20, 4, 21, 0.5), (36, 24, 3, 19, 0.5),
                                        (36, 20, 1, 23, 0.5), (64, 44, 30, 37, 3.0), (64, 44, 32, 29, 3.0),
                                        (64, 416, 32, 45, 3.0)])
def test_vae_clipped_sum_matches_oracle(cuda, D, H, Z, B, C):
    check_clipped_sum(D, H, Z, B, C)


@pytest.mark.parametrize("D,H,Z,B,C", [(36, 20, 3, 19, 0.5), (64, 44, 30, 37, 3.0)])
def test_vae_step_ignores_stale_workspace(cuda, D, H, Z, B, C):
    """The step reads no workspace entry it has not written itself: the padded k-steps of the thin-layer kernels read
    past the real rows and columns of their A operands, and a zero weight does not cancel a NaN."""
    check_clipped_sum(D, H, Z, B, C, poison=True)


def test_vae_step_opts_in_to_shared_memory_in_a_fresh_process(cuda):
    """At H = 320 the backward thin-layer kernel's static and dynamic shared memory come to more than 48 KB, its dynamic
    part alone to less than 24 KB; the opt-in is a per-process attribute, so the step runs in a process of its own."""
    here = os.path.dirname(os.path.abspath(__file__))
    code = (f"import sys; sys.path[:0] = [{os.path.dirname(here)!r}, {here!r}]; import test_gpu_vae as t; "
            "t.check_clipped_sum(64, 320, 8, 37, 3.0); print('OPT_IN_OK')")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "OPT_IN_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_vae_trajectory_matches_oracle(cuda):
    X, o, ost, s, st = make(64, 40, 8, 5000, 33, 1.0, 1.0)
    Xd = torch.as_tensor(X).cuda()
    for _ in range(3):
        ost, oloss = o.update(ost, X)
        st, loss = s.update(st, Xd)
        assert np.isclose(float(loss), float(oloss), rtol=REL)
    oref, got = o.get_params(ost), s.get_params(st)
    for k in oref:
        assert ew_rel_err(got[k], oref[k]) < REL, (k, ew_rel_err(got[k], oref[k]))
    assert np.array_equal(np.asarray(st.rng_key).reshape(-1), np.asarray(ost.rng_key).reshape(-1))


def test_vae_full_shape_properties(cuda):
    """BASELINE config 5 (784-400-20, batch 4096): too slow for the autodiff oracle, so check
    size-independent properties — determinism, linearity of the clipped sum in the batch (two
    half batches of disjoint masks add up to the full batch), and norms <= C after clipping."""
    D, H, Z, B = 784, 400, 20, 4096
    g = torch.Generator(device="cuda").manual_seed(0)
    X = (torch.rand((B, 28, 28), device=cuda, generator=g) < 0.3).float()
    fam = models.VAE(D, H, Z, init_std=0.05)

    def grad(mask):
        s = dsvi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.0), models.Trace_ELBO(), 10.0, 0.0, num_obs_total=60000)
        st = s.init(rng.PRNGKey(0), X)
        p0 = st.optim_state.flat.clone()
        st2, loss = s.update(st, X, mask=mask)
        n = float(mask.sum())
        return (p0 - st2.optim_state.flat) * n, float(loss)      # = obs_scale * sum_i c_i g_i

    full = torch.ones(B, dtype=torch.bool, device=cuda)
    lo = full.clone(); lo[B // 2:] = False
    hi = ~lo
    g_full, l_full = grad(full)
    g_again, _ = grad(full)
    assert torch.equal(g_full, g_again)                           # fixed-order reductions: bitwise repeatable
    g_lo, _ = grad(lo)
    g_hi, _ = grad(hi)
    err = (g_lo + g_hi - g_full).abs().max() / g_full.abs().max()
    assert err < 2e-5, float(err)
    assert np.isfinite(l_full)
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.0), models.Trace_ELBO(), 10.0, 0.0, num_obs_total=60000)
    st = s.init(rng.PRNGKey(0), X)
    st1, keys = s._split_rng_key(st, 2)
    norms = torch.zeros(B, device=cuda)
    s._run_step(st1, keys[0], (X,), True, px_norms=norms)
    assert float(norms.min()) > 0 and torch.isfinite(norms).all()


@pytest.mark.parametrize("init_std,C", [(0.03, 300.0), (0.05, 1200.0)])     # C near the median per-example norm
def test_vae_full_shape_matches_explicit_oracle(cuda, init_std, C):
    """BASELINE config 5 at its real shape (784-400-20, B = 4096: the 4-way batch split and the 144-CTA concurrent
    wave of clipped-sum GEMMs) against oracle.vae.explicit_clipped_sum — forward / backward as float64 matmuls,
    ghost norms, A^T diag(c) Delta — which tests/test_oracle_families.py pins to vmap(grad) of the per-example ELBO.
    Compared: all 4096 per-example norms and losses, and the whole 652 824-element clipped sum, leaf by leaf,
    element-wise (helpers/tolerance.py)."""
    D, H, Z, B, N = 784, 400, 20, 4096, 60000
    rs = np.random.RandomState(0)
    X = (rs.rand(B, 28, 28) < 0.35).astype(np.float32)
    mask = np.ones(B, bool)
    mask[B // 3::5] = False
    ofam = ovae.VAE(D, H, Z, N)
    p0 = ofam.init_params(0, init_std)
    fam = models.VAE(D, H, Z)
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.SGD(1.0), models.Trace_ELBO(), C, 0.0, num_obs_total=N)
    Xd, md = torch.as_tensor(X).cuda(), torch.as_tensor(mask).cuda()
    st = s.init(chacha.PRNGKey(11), Xd, params=p0)
    st1, keys = s._split_rng_key(st, 2)
    norms, loss = torch.zeros(B, device=cuda), torch.zeros(B, device=cuda)
    ws, n_part, _, P = s._run_step(st1, keys[0], (Xd,), md, px_norms=norms, px_loss=loss)
    assert P == 652824 and n_part == 4
    part = ws.view(-1)[: n_part * (P + 2)].view(n_part, P + 2).double().sum(0).cpu().numpy()
    eps = ofam.sample_eps(threefry.split(chacha.convert_to_jax_rng_key(np.asarray(keys[0])), B))["z"]
    ref_loss, ref_norm, ref_sum = ovae.explicit_clipped_sum(p0, X, eps, C, mask, ofam.site_scale, st.observation_scale)
    assert 0.2 < np.mean(ref_norm[mask] > C) < 1.0            # the clip is active for part of the batch
    got_norm, got_loss = norms.cpu().numpy().astype(np.float64), loss.cpu().numpy().astype(np.float64)
    # ghost norms: a 5-layer chain of fp32 GEMMs (forward + delta backward) per example; measured 4e-6 / 1.3e-5
    assert np.max(np.abs(got_norm - ref_norm)[mask] / ref_norm[mask]) < 2e-5
    assert np.max(np.abs(got_loss - ref_loss * st.observation_scale)[mask] / np.abs(ref_loss[mask])) < REL
    assert np.all(got_norm[~mask] == 0) or np.all(np.isfinite(got_norm))
    assert part[P + 1] == mask.sum()
    assert abs(part[P] - ref_loss.sum() * st.observation_scale) < REL * abs(ref_loss.sum())
    for name, off, shape in fam.layout():
        size = int(np.prod(shape)) if len(shape) else 1
        got, ref = part[off:off + size], ref_sum[name].ravel()
        assert l2_err(got, ref) < REL, (name, l2_err(got, ref))
        # element-wise with floor = rms(leaf).  2e-5, not 1e-5: the accumulators of tcgen05.mma truncate (DESIGN.md
        # section 7, scripts/gemm_accuracy.py), ~2^-24 per 8-deep k-step over the 1024-example contraction of a split
        assert ew_rel_err(got, ref) < 2e-5, (name, ew_rel_err(got, ref))


@pytest.mark.parametrize("D,H,Z,B", [(36, 24, 4, 50), (36, 20, 3, 19), (64, 40, 20, 333), (784, 400, 20, 1000),
                                     (36, 20, 4, 50), (36, 24, 3, 45), (36, 20, 1, 77), (64, 44, 30, 333),
                                     (64, 44, 32, 99), (64, 416, 32, 123)])
def test_vae_evaluate_matches_oracle(cuda, D, H, Z, B):
    """DPSVI.evaluate (d3p/svi.py:436-449; examples/vae.py:236-247): one guide draw z [B, Z] for the whole batch,
    scale (N / B) (1 / N)."""
    X, o, ost, s, st = make(D, H, Z, 60000, B, 10.0, 1.0)
    want = o.evaluate(ost, X)
    got = float(s.evaluate(st, torch.as_tensor(X).cuda()))
    assert np.isclose(got, want, rtol=REL), (got, want)
    # evaluate does not touch the state; a second call gives the same number
    assert float(s.evaluate(st, torch.as_tensor(X).cuda())) == got
