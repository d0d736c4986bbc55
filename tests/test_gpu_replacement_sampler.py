"""``subsample_batchify_data(with_replacement=True)`` on the device alone: ``d3p_chacha_randint`` runs the whole
rejection loop of ``randint`` in one launch, and the epoch drivers draw with it (``D3P_SAMPLER_SUBSAMPLE_REPLACE``).

* the one-launch values equal the oracle's ``randint`` and the per-round entry points bit for bit, at every width,
  for awkward spans and sizes, and where some lane needs 20 or more rounds;
* the device-key twin equals the host-key entry; ``rng.randint`` records inside a CUDA graph capture;
* ``run_epoch`` with the with-replacement batchifier takes the C driver and equals the ``update`` loop bit for bit for
  every family, with device keys too, and in a two-rank sharded run;
* the refusals come before any launch."""
import ctypes as C

import numpy as np
import pytest
import torch

import d3p_b200.random as rng
from d3p_b200 import _native as _n, minibatch as mb, models, optimizers, parallel, svi as dsvi
from helpers.tolerance import rel_err
from oracle import chacha

pytestmark = pytest.mark.gpu
U32P = C.POINTER(C.c_uint32)
NP_INT = {8: np.int8, 16: np.int16, 32: np.int32}
TORCH_INT = {8: torch.int8, 16: torch.int16, 32: torch.int32}


def _hp(key):
    a = np.ascontiguousarray(np.asarray(key, dtype=np.uint32).reshape(-1))
    return a, a.ctypes.data_as(U32P)


def _dkey(key):
    return torch.as_tensor(np.ascontiguousarray(np.asarray(key, dtype=np.uint32).reshape(-1)).view(np.int32)).cuda()


def _oracle_mask(nbits, delta):
    # oracle/chacha.py randint, restated: the rejection mask of the per-round loop
    udtype = {8: np.uint8, 16: np.uint16, 32: np.uint32}[nbits]
    delta = udtype(delta)
    log_po2 = min(int(udtype(np.float32(np.log2(np.float32(delta))) + np.float32(1))) if delta > 0 else 0, nbits)
    return int(((1 << log_po2) - 1) & ((1 << nbits) - 1))


def _per_round(key, nbits, lo, hi, n):
    """The rejection loop as the library ran it before the one-launch kernel: one d3p_chacha_randint_round launch and
    one host read per round, then d3p_randint_finish."""
    lib = _n.lib()
    delta = (hi - 1 - lo) & ((1 << nbits) - 1)
    bitmask = _oracle_mask(nbits, delta)
    vals = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    pending = torch.zeros(1, dtype=torch.int32, device="cuda")
    first = 1
    while True:
        ks = rng.split(key, 2)
        key, round_key = ks[0], ks[1]
        _, p = _hp(round_key)
        _n.check(lib.d3p_chacha_randint_round(p, nbits, bitmask, delta, first, _n.ptr(vals), n, _n.ptr(pending),
                                              _n.stream_ptr()), "randint_round")
        first = 0
        if int(pending.item()) == 0:
            break
    out = torch.empty(max(n, 1), dtype=TORCH_INT[nbits], device="cuda")
    lo32 = ((lo + (1 << 31)) & 0xFFFFFFFF) - (1 << 31)
    _n.check(lib.d3p_randint_finish(_n.ptr(vals), lo32, nbits, _n.ptr(out), n, _n.stream_ptr()), "randint_finish")
    return out[:n].cpu().numpy()


def _rounds(key, nbits, lo, hi, n):
    """Per element, the round whose draw the loop of oracle/chacha.py randint keeps (that loop does not report it)."""
    udtype = {8: np.uint8, 16: np.uint16, 32: np.uint32}[nbits]
    delta = udtype((hi - 1 - lo) & ((1 << nbits) - 1))
    bitmask = udtype(_oracle_mask(nbits, int(delta)))
    keys = chacha.split(key, 2)
    key, round_key = keys[0], keys[1]
    uvals = chacha.random_bits(round_key, nbits, (n,)).astype(udtype) & bitmask
    rounds, r = np.ones(n, np.int64), 1
    while np.any(uvals > delta):
        r += 1
        keys = chacha.split(key, 2)
        key, round_key = keys[0], keys[1]
        new = chacha.random_bits(round_key, nbits, (n,)).astype(udtype) & bitmask
        rounds[uvals > delta] = r
        uvals = np.where(uvals > delta, new, uvals)
    return rounds


def _spans(nbits):
    """(minval, maxval) pairs: spans 1, 2, 3, 2^k, 2^k + 1, the full range of the type, a negative minval, and for
    32-bit results the data-set sizes 10 M and 2^31 - 1."""
    k = nbits - 3
    half = 1 << (nbits - 1)
    out = [(0, 1), (5, 7), (-1, 2), (0, 1 << k), (3, 3 + (1 << k) + 1), (-half, half), (-half + 3, -7)]
    if nbits == 32:
        out += [(0, 10_000_000), (0, (1 << 31) - 1)]
    return out


@pytest.mark.parametrize("n", [0, 1, 15, 16, 17, 4097, 100_736])
@pytest.mark.parametrize("nbits", [8, 16, 32])
def test_randint_equals_oracle_and_per_round_loop(cuda, nbits, n):
    for j, (lo, hi) in enumerate(_spans(nbits)):
        key = rng.fold_in(rng.PRNGKey(1000 + nbits), 31 * n + j)
        got = rng.randint(key, (n,), lo, hi, TORCH_INT[nbits]).cpu().numpy()
        assert got.dtype == NP_INT[nbits] and got.shape == (n,)
        want = chacha.randint(key, (n,), lo, hi, NP_INT[nbits])
        assert np.array_equal(got, want), (nbits, n, lo, hi)
        assert np.array_equal(got, _per_round(key, nbits, lo, hi, n)), (nbits, n, lo, hi)


def test_randint_lane_with_many_rounds(cuda):
    """span 2^20 + 1 draws under a 21-bit mask: about half of the draws are rejected, so among ~10^6 elements some
    need 20 or more rounds; the kernel runs each lane to acceptance with no round cap."""
    n, lo, hi = 1_000_000, -5, -5 + (1 << 20) + 1
    key = rng.PRNGKey(1)
    rounds = _rounds(key, 32, lo, hi, n)
    assert rounds.max() >= 20, rounds.max()
    got = rng.randint(key, (n,), lo, hi).cpu().numpy()
    want = chacha.randint(key, (n,), lo, hi, np.int32)
    assert np.array_equal(got, want)
    assert np.array_equal(got, _per_round(key, 32, lo, hi, n))
    assert got.min() >= lo and got.max() < hi


@pytest.mark.parametrize("nbits", [8, 16, 32])
def test_randint_device_key_twin(cuda, nbits):
    lib = _n.lib()
    for n, (lo, hi) in zip((1, 17, 4097, 100_736), _spans(nbits)[2:]):
        key = rng.fold_in(rng.PRNGKey(77), n)
        _, p = _hp(key)
        a = torch.empty(n, dtype=TORCH_INT[nbits], device=cuda)
        b = torch.full((n,), 3, dtype=TORCH_INT[nbits], device=cuda)
        kd = _dkey(key)
        _n.check(lib.d3p_chacha_randint(p, nbits, lo, hi, _n.ptr(a), n, _n.stream_ptr()), "randint")
        _n.check(lib.d3p_chacha_randint_dk(_n.ptr(kd), nbits, lo, hi, _n.ptr(b), n, _n.stream_ptr()), "randint_dk")
        assert torch.equal(a, b), (nbits, n)


def test_randint_in_graph_capture(cuda):
    """No host synchronisation: the call records inside torch.cuda.graph, and a replay writes the same values."""
    key, n, lo, hi = rng.PRNGKey(12), 100_736, 0, 10_000_000
    want = chacha.randint(key, (n,), lo, hi, np.int32)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        rng.randint(key, (n,), lo, hi)            # loads the module outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = rng.randint(key, (n,), lo, hi)
    out.fill_(-1)
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), want)


def test_randint_refusals(cuda):
    lib = _n.lib()
    _, p = _hp(rng.PRNGKey(3))
    out = torch.full((64,), 7, dtype=torch.int32, device=cuda)
    assert lib.d3p_chacha_randint(p, 64, 0, 10, _n.ptr(out), 64, _n.stream_ptr()) == -3
    assert lib.d3p_chacha_randint_dk(_n.ptr(out), 4, 0, 10, _n.ptr(out), 64, _n.stream_ptr()) == -3
    assert lib.d3p_chacha_randint(p, 32, 0, 10, None, 64, _n.stream_ptr()) == -1
    assert lib.d3p_chacha_randint(None, 32, 0, 10, _n.ptr(out), 64, _n.stream_ptr()) == -1
    assert lib.d3p_chacha_randint_dk(None, 32, 0, 10, _n.ptr(out), 64, _n.stream_ptr()) == -1
    assert lib.d3p_chacha_randint(p, 32, 0, 10, _n.ptr(out), 0, _n.stream_ptr()) == 0
    torch.cuda.synchronize()
    assert bool((out == 7).all())


# ---- run_epoch with subsample_batchify_data(with_replacement=True) ------------------------------------------------

def _family(kind, cuda):
    g = torch.Generator(device="cuda").manual_seed(11)
    if kind == "logreg":
        N, d = 3000, 12
        data = (torch.randn((N, d), device=cuda, generator=g), (torch.rand(N, device=cuda, generator=g) < .5).to(torch.int32))
        return models.LogisticRegression(d), data, 1.0, 64
    if kind == "gauss":
        N, d = 3000, 40
        return models.GaussianMean(d), (1 + .1 * torch.randn((N, d), device=cuda, generator=g),), 30.0, 333
    if kind == "gmm":
        N, K, d = 4000, 4, 3
        centers = torch.randn((K, d), device=cuda, generator=g) * 3
        lab = torch.randint(0, K, (N,), device=cuda, generator=g)
        return models.GaussianMixture(K, d), (centers[lab] + torch.randn((N, d), device=cuda, generator=g),), 20.0, 80
    N = 600
    return models.VAE(64, 40, 8, init_std=0.1), ((torch.rand((N, 8, 8), device=cuda, generator=g) < .35).float(),), 2.0, 48


def _setup(kind, cuda, return_mask=False):
    fam, data, clip, B = _family(kind, cuda)
    N = len(data[0])
    s = dsvi.DPSVI(fam.model, fam.guide, optimizers.Adam(1e-2), models.Trace_ELBO(), clip, .7, num_obs_total=N)
    init, get = mb.subsample_batchify_data(data, batch_size=B, with_replacement=True, return_mask=return_mask)
    assert get.spec["kind"] == _n.SAMPLER_SUBSAMPLE_REPLACE
    key, k_init, k_fetch = rng.split(rng.PRNGKey(21), 3)
    _, bst = init(k_fetch)
    out = get(0, bst)
    st0 = s.init(k_init, *(out[0] if return_mask else out))
    return s, get, bst, st0


def _stepwise(s, st, get, bst, first_step, n_steps):
    losses = []
    for i in range(first_step, first_step + n_steps):
        out = get(i, bst)
        batch, mask = out if (isinstance(out, tuple) and len(out) == 2 and isinstance(out[0], tuple)) else (out, True)
        st, loss = s.update(st, *batch, mask=mask)
        losses.append(float(loss))
    return st, losses


def _no_update(monkeypatch):
    """run_epoch must take the C driver: the step-by-step fallback calls DPSVI.update, which now raises."""
    def boom(*a, **k):
        raise AssertionError("run_epoch fell back to the step-by-step loop")
    monkeypatch.setattr(dsvi.DPSVI, "update", boom)


@pytest.mark.parametrize("kind,return_mask", [("logreg", False), ("gauss", True), ("gmm", False), ("vae", True)])
def test_run_epoch_equals_update_loop(cuda, kind, return_mask, monkeypatch):
    s, get, bst, st0 = _setup(kind, cuda, return_mask)
    n_steps, first_step = 6, 3
    ref, losses = _stepwise(s, st0, get, bst, first_step, n_steps)
    with monkeypatch.context() as m:
        _no_update(m)
        st, stats = s.run_epoch(st0, get, bst, n_steps, first_step=first_step)
    assert st.optim_state.step == ref.optim_state.step == n_steps
    assert torch.equal(st.optim_state.flat, ref.optim_state.flat), "run_epoch must be bit-identical to the update loop"
    assert torch.equal(st.optim_state.m, ref.optim_state.m) and torch.equal(st.optim_state.v, ref.optim_state.v)
    assert [float(v) for v in stats[:, 0].cpu()] == losses
    assert np.array_equal(np.asarray(st.rng_key), np.asarray(ref.rng_key))
    B = get.spec["batch"]
    assert bool((stats[:, 1] == B).all()) and bool((stats[:, 2] == 1).all())      # n and f of a full batch


@pytest.mark.parametrize("kind", ["logreg", "gauss", "vae"])
def test_run_epoch_device_keys(cuda, kind, monkeypatch):
    s, get, bst, st0 = _setup(kind, cuda)
    with monkeypatch.context() as m:
        _no_update(m)
        a, sa = s.run_epoch(st0, get, bst, 5, first_step=2)
        b, sb = s.run_epoch(st0, get, bst, 5, first_step=2, device_keys=True)
    assert torch.equal(a.optim_state.flat, b.optim_state.flat)
    assert torch.equal(sa, sb)
    assert np.array_equal(np.asarray(a.rng_key, np.uint32).reshape(-1), np.asarray(b.rng_key, np.uint32).reshape(-1))
    ref, _ = _stepwise(s, st0, get, bst, 2, 5)
    assert torch.equal(a.optim_state.flat, ref.optim_state.flat)


def _sharded(kind, cuda, world, steps=3):
    """`world` logical ranks on one device (PeerWindow.local_group), one run_epoch step per call and rank after rank:
    the only kernel that waits for a peer is then the last one queued on its stream (see test_gpu_comm_loopback.py)."""
    fam0, data, clip, B = _family(kind, cuda)
    N = len(data[0])
    fams = [fam0] + [_family(kind, cuda)[0] for _ in range(world - 1)]
    wins = parallel.PeerWindow.local_group(world, fam0.n_params) if world > 1 else []
    for w in wins:
        w.set_timeout_ms(4000)
    svis = []
    for r in range(world):
        s = dsvi.DPSVI(fams[r].model, fams[r].guide, optimizers.Adam(1e-3), models.Trace_ELBO(), clip, 1.0,
                       num_obs_total=N)
        if world > 1:
            parallel.shard_dpsvi(s, window=wins[r])
        svis.append(s)
    init, get = mb.subsample_batchify_data(data, batch_size=B, with_replacement=True)
    key, k_init, k_fetch = rng.split(rng.PRNGKey(5), 3)
    _, bst = init(k_fetch)
    states = [s.init(k_init, *get(0, bst)) for s in svis]
    streams = [torch.cuda.Stream() for _ in range(world)]
    torch.cuda.synchronize()
    losses = [[] for _ in range(world)]
    for i in range(steps):
        stats = [None] * world
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                states[r], stats[r] = svis[r].run_epoch(states[r], get, bst, 1, first_step=i)
        torch.cuda.synchronize()
        for r in range(world):
            losses[r].append(float(stats[r][0, 0]))
    for w in wins:
        assert w.timeouts() == 0
    flats = [st.optim_state.flat.clone() for st in states]
    keys = [np.asarray(st.rng_key).copy() for st in states]
    for w in wins:
        w.close()
    return flats, losses, keys


@pytest.mark.parametrize("kind", ["logreg", "gauss"])
def test_sharded_run_epoch_on_one_device(cuda, kind, monkeypatch):
    with monkeypatch.context() as m:
        _no_update(m)
        (p1,), (l1,), (k1,) = _sharded(kind, cuda, 1)
        flats, losses, keys = _sharded(kind, cuda, 2)
    for r in range(2):
        assert torch.equal(flats[r], flats[0]), f"replica {r} differs from replica 0"
        assert np.array_equal(keys[r], k1)
        assert losses[r] == losses[0]
    assert rel_err(flats[0], p1) <= 1e-5, rel_err(flats[0], p1)
    assert np.allclose(losses[0], l1, rtol=2e-5), (losses[0], l1)


@pytest.mark.parametrize("device_keys", [False, True])
def test_run_epoch_refuses_empty_replacement_sampler(cuda, device_keys, monkeypatch):
    """A REPLACE descriptor with batch == 0 or n_records == 0: no workspace size, and the driver returns
    D3P_ERR_INVALID_ARGUMENT before its first kernel (parameters, state key and stats stay as they were)."""
    s, get, bst, st0 = _setup("logreg", cuda)
    fam = s.family
    calls = []
    real = type(fam)._epoch

    def spy(self, dk, desc, sampler, x, stride, y, batch_key, rng_key, rest):
        calls.append((desc, x, stride, y, rest))
        return real(self, dk, desc, sampler, x, stride, y, batch_key, rng_key, rest)

    monkeypatch.setattr(type(fam), "_epoch", spy)
    st, _ = s.run_epoch(st0, get, bst, 4, device_keys=device_keys)
    desc, x, stride, y, rest = calls[-1]
    lib = _n.lib()
    N, B = get.spec["n_records"], get.spec["batch"]
    rest = list(rest)
    rest[6] = C.byref(s.optim.desc(st.optim_state.step, st.optim_state.lr, desc.n_params))
    stats = torch.full((4, 3), 5.0, device=cuda)
    rest[10] = _n.ptr(stats)
    flat_before = st.optim_state.flat.clone()
    if device_keys:
        run = lib.d3p_dpsvi_run_epoch_meanfield_dk
        bkey, rkey = _dkey(bst), _dkey(st.rng_key)
        keys = (_n.ptr(bkey), _n.ptr(rkey))
    else:
        run = lib.d3p_dpsvi_run_epoch_meanfield
        (bkey, bp), (rkey, rp) = _hp(bst), _hp(st.rng_key)
        keys = (bp, rp)
    rkey_before = rkey.clone() if device_keys else rkey.copy()
    for n_records, batch in ((N, 0), (0, B)):
        sd = _n.SamplerDesc(_n.SAMPLER_SUBSAMPLE_REPLACE, 0.0, n_records, batch, 0, None)
        assert lib.d3p_dpsvi_epoch_workspace_bytes(C.byref(desc), C.byref(sd)) == 0
        assert run(C.byref(desc), C.byref(sd), x, stride, y, *keys, *rest) == -1
    torch.cuda.synchronize()
    assert torch.equal(st.optim_state.flat, flat_before)
    assert bool((stats == 5.0).all())
    assert (torch.equal(rkey, rkey_before) if device_keys else np.array_equal(rkey, rkey_before))
    # drawn with replacement, a batch may be larger than the data set
    big = _n.SamplerDesc(_n.SAMPLER_SUBSAMPLE_REPLACE, 0.0, 10, 50, 0, None)
    assert lib.d3p_dpsvi_epoch_workspace_bytes(C.byref(desc), C.byref(big)) > 0
