"""Consumer of the ``optraj_*`` keys of a reference dump (baseline/run_reference.py ``OPTIM_CASES``): 3-step
logistic-regression trajectories with numpyro's Momentum / Adagrad / RMSProp / RMSPropMomentum / ClippedAdam and a
scheduled Adam.  The writer / file format / consumer round trip runs with the oracle standing in for the reference;
the comparison with a real reference file runs the oracle and the CUDA path against it."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from baseline import run_reference as rr  # noqa: E402

REF_FILE = os.path.join(ROOT, "tests", "golden", "reference_v1.npz")


def check_optim_trajectories(trajectory, d, rtol):
    """Compares ``trajectory(spec)`` (-> dict as ``OracleImpl.trajectory``) with every ``optraj_*`` case in ``d``;
    returns the case names compared."""
    done = []
    data, mask, N, shape = rr.trajectory_inputs("logreg")
    for name, spec in rr.OPTIM_CASES.items():
        if f"optraj_{name}_loss" not in d.files:
            continue
        tr = trajectory(spec, data, mask, N, shape)
        assert np.allclose(tr["loss"], d[f"optraj_{name}_loss"], rtol=rtol), name
        assert np.array_equal(np.stack(tr["rng_key"]), d[f"optraj_{name}_rng_key"]), name
        for s, leaves in enumerate(tr["params"]):
            for i, leaf in enumerate(leaves):
                want = d[f"optraj_{name}_step{s}_{i}"]
                err = np.max(np.abs(np.asarray(leaf, np.float64) - want) /
                             np.maximum(np.abs(want), np.sqrt(np.mean(np.square(want.astype(np.float64)))) + 1e-30))
                assert err <= rtol, (name, s, i, err)
        done.append(name)
    return done


def _oracle_trajectory(spec, data, mask, N, shape):
    return rr.OracleImpl().trajectory("logreg", data, mask, 3, 7, N, optim=spec, **shape)


def test_writer_round_trip_with_oracle_stand_in(tmp_path):
    path = tmp_path / "oracle_dump.npz"
    keys = rr.dump(rr.OracleImpl(), str(path), families=())
    assert all(f"optraj_{n}_loss" in keys for n in rr.OPTIM_CASES)
    d = np.load(path)
    assert str(d["impl"]) == "oracle" and str(d["skipped"]) == ""
    assert check_optim_trajectories(_oracle_trajectory, d, rtol=0.0) == list(rr.OPTIM_CASES)


def test_oracle_matches_reference_file():
    if not os.path.exists(REF_FILE):
        pytest.skip("tests/golden/reference_v1.npz not generated: writing it needs jax + numpyro + jax-chacha-prng "
                    "(python baseline/run_reference.py tests/golden/reference_v1.npz), none of which is installed here")
    d = np.load(REF_FILE)
    assert str(d["impl"]) == "reference"
    if not any(k.startswith("optraj_") for k in d.files):
        pytest.skip("reference_v1.npz predates the optraj_* keys: regenerate it")
    assert check_optim_trajectories(_oracle_trajectory, d, rtol=1e-5)
