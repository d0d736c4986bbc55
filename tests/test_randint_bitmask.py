"""CPU test of randint's rejection mask in C (``d3p_randint_bitmask``, the rule ``d3p_chacha_randint`` and the epoch
drivers' with-replacement sampler use) against the numpy oracle's rule, including the widening of the mask that the
float32 rounding of delta causes just below powers of two.  No kernel is launched here."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def lib():
    from d3p_b200 import _build, _native
    _build.build()
    return _native.lib()


def _oracle_bitmask(nbits, delta):
    # oracle/chacha.py randint: delta, log_po2 and bitmask in the unsigned result type
    udtype = {8: np.uint8, 16: np.uint16, 32: np.uint32}[nbits]
    with np.errstate(over="ignore"):
        delta = udtype(delta)
        log_po2 = min(int(udtype(np.float32(np.log2(np.float32(delta))) + np.float32(1))) if delta > 0 else 0, nbits)
        return int(udtype(((1 << log_po2) - 1) & ((1 << nbits) - 1)))


def _deltas(nbits):
    full = (1 << nbits) - 1
    near = {p + o for k in range(33) for p in (1 << k,) for o in range(-256, 257)}
    rand = np.random.RandomState(nbits).randint(0, 1 << 32, size=100_000, dtype=np.uint64)
    return sorted({d & full for d in near if d >= 0} | {int(d) & full for d in rand})


@pytest.mark.parametrize("nbits", [8, 16, 32])
def test_bitmask_rule_matches_oracle(lib, nbits):
    bad = [d for d in _deltas(nbits) if lib.d3p_randint_bitmask(nbits, d) != _oracle_bitmask(nbits, d)]
    assert not bad, (nbits, bad[:10])


def test_bitmask_rule_keeps_the_float32_widening(lib):
    # 2^25 - 1 rounds to 2^25 in float32, and log2(2^24 - 1) rounds to 24 in float32: each mask gets one bit more
    # than the span needs.  Further below the power of two the mask is the tight one.
    assert lib.d3p_randint_bitmask(32, (1 << 25) - 1) == (1 << 26) - 1
    assert lib.d3p_randint_bitmask(32, (1 << 24) - 1) == (1 << 25) - 1
    assert lib.d3p_randint_bitmask(32, 10_000_000 - 1) == (1 << 24) - 1
    assert lib.d3p_randint_bitmask(32, 0) == 0
    assert lib.d3p_randint_bitmask(8, 255) == 255
    assert lib.d3p_randint_bitmask(32, 0xFFFFFFFF) == 0xFFFFFFFF


def test_randint_refusals_before_any_launch(lib):
    import ctypes as C
    key = np.zeros(16, np.uint32)
    kp = key.ctypes.data_as(C.POINTER(C.c_uint32))
    assert lib.d3p_chacha_randint(kp, 64, 0, 10, None, 5, None) == -3          # D3P_ERR_UNSUPPORTED
    assert lib.d3p_chacha_randint(kp, 12, 0, 10, None, 0, None) == -3
    assert lib.d3p_chacha_randint(kp, 32, 0, 10, None, 5, None) == -1          # D3P_ERR_INVALID_ARGUMENT
    assert lib.d3p_chacha_randint(None, 32, 0, 10, C.c_void_p(256), 5, None) == -1
    assert lib.d3p_chacha_randint_dk(None, 16, 0, 10, C.c_void_p(256), 5, None) == -1
    assert lib.d3p_chacha_randint(None, 32, 0, 10, None, 0, None) == 0        # n == 0: nothing to do
    assert lib.d3p_chacha_randint_dk(None, 8, 0, 10, None, 0, None) == 0
