"""ChaCha20 rng suite — the module-as-interface of ``d3p/random/__init__.py:28-155``
(``PRNGState, PRNGKey, split, fold_in, random_bits, uniform, normal, randint,
convert_to_jax_rng_key``) on top of the CUDA keystream kernels of libd3p_b200.

Keys are host-side ``numpy.uint32`` arrays of shape (4, 4) (RFC 8439 state, like
jax-chacha-prng's ``RNGState``); generated arrays are torch CUDA tensors.  Key derivation
(``split`` / ``fold_in``) runs in the library's host functions and costs no device work.
"""
import ctypes as C
import secrets
from typing import Optional, Sequence, Union

import numpy as np
import torch

from .. import _native as _n

PRNGState = np.ndarray
STATE_SHAPE = (4, 4)
ChaChaKeySizeInBytes = 32


def _state(key):
    a = np.ascontiguousarray(np.asarray(key, dtype=np.uint32).reshape(16))
    return a, a.ctypes.data_as(C.POINTER(C.c_uint32))


def _shape(shape):
    if isinstance(shape, (int, np.integer)):
        return (int(shape),)
    return tuple(int(s) for s in shape)


def _device():
    if not torch.cuda.is_available():
        raise _n.D3PNativeError("d3p_b200 needs a CUDA device (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def PRNGKey(seed: Optional[Union[np.ndarray, int, bytes]] = None) -> PRNGState:
    """``d3p/random/__init__.py:35-47``: ``None`` draws 32 bytes from ``secrets``."""
    if seed is None:
        seed = secrets.token_bytes(ChaChaKeySizeInBytes)
    if isinstance(seed, (int, np.integer)):
        seed = (int(seed) % (1 << 256)).to_bytes(32, byteorder="big", signed=False)
    if isinstance(seed, (bytes, bytearray)):
        if len(seed) > 32:
            raise ValueError("seed must be at most 256 bit long")
        raw = bytes(seed)
    else:
        words = np.asarray(seed, dtype=np.uint32).ravel()
        if words.size > 8:
            raise ValueError("seed must be at most 256 bit long")
        raw = words.astype("<u4").tobytes()
    out = np.zeros(16, dtype=np.uint32)
    buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw) if raw else None
    _n.check(_n.lib().d3p_chacha_key_from_seed_h(C.cast(buf, C.c_void_p) if buf is not None else None, len(raw),
                                                 out.ctypes.data_as(C.POINTER(C.c_uint32))), "PRNGKey")
    return out.reshape(STATE_SHAPE)


def split(key: PRNGState, num: int = 2) -> np.ndarray:
    a, p = _state(key)
    out = np.zeros((int(num), 16), dtype=np.uint32)
    _n.check(_n.lib().d3p_chacha_split_h(p, int(num), out.ctypes.data_as(C.POINTER(C.c_uint32))), "split")
    return out.reshape((int(num),) + STATE_SHAPE)


def fold_in(key: PRNGState, data: int) -> PRNGState:
    a, p = _state(key)
    out = np.zeros(16, dtype=np.uint32)
    _n.check(_n.lib().d3p_chacha_fold_in_h(p, int(data) & 0xFFFFFFFF, out.ctypes.data_as(C.POINTER(C.c_uint32))),
             "fold_in")
    return out.reshape(STATE_SHAPE)


def random_bits_host(key: PRNGState, n_words: int) -> np.ndarray:
    """First ``n_words`` keystream words on the host (tiny outputs: key conversion, Feistel constants)."""
    a, p = _state(key)
    out = np.zeros(int(n_words), dtype=np.uint32)
    _n.check(_n.lib().d3p_chacha_random_bits_h(p, 0, out.ctypes.data_as(C.POINTER(C.c_uint32)), int(n_words)),
             "random_bits_host")
    return out


def random_bits(key: PRNGState, bit_width: int, shape: Sequence[int]) -> torch.Tensor:
    if bit_width not in (8, 16, 32, 64):
        raise ValueError("requires bit field width in (8, 16, 32, 64)")
    shape = _shape(shape)
    size = int(np.prod(shape)) if len(shape) else 1
    n_words = (size * bit_width + 31) // 32
    a, p = _state(key)
    buf = torch.empty(max(n_words, 1), dtype=torch.int32, device=_device())
    _n.check(_n.lib().d3p_chacha_random_bits(p, 0, _n.ptr(buf), n_words, _n.stream_ptr()), "random_bits")
    words = buf[:n_words].view(torch.uint32)
    if bit_width == 32:
        out = words
    elif bit_width == 64:
        out = words.view(torch.uint64)
    else:
        out = words.view({8: torch.uint8, 16: torch.uint16}[bit_width])
    return out[:size].reshape(shape)


def uniform(key: PRNGState, shape: Sequence[int] = (), dtype=torch.float32, minval=0.0, maxval=1.0) -> torch.Tensor:
    if dtype not in (torch.float32, np.float32, "float32"):
        if dtype in (torch.float64, torch.float16, torch.bfloat16, np.float64, np.float16):
            raise TypeError("d3p_b200 implements the float32 path of rng_suite.uniform only")
        raise ValueError(f"dtype argument to `uniform` must be a float dtype, got {dtype}")
    shape = _shape(shape)
    size = int(np.prod(shape)) if len(shape) else 1
    a, p = _state(key)
    out = torch.empty(max(size, 1), dtype=torch.float32, device=_device())
    _n.check(_n.lib().d3p_chacha_uniform_f32(p, 0, float(minval), float(maxval), _n.ptr(out), size,
                                             _n.stream_ptr()), "uniform")
    return out[:size].reshape(shape)


def normal(key: PRNGState, shape: Sequence[int] = (), dtype=torch.float32) -> torch.Tensor:
    """``d3p/random/__init__.py:50-81``."""
    if dtype not in (torch.float32, np.float32, "float32"):
        if dtype in (torch.float64, torch.float16, torch.bfloat16, np.float64, np.float16):
            raise TypeError("d3p_b200 implements the float32 path of rng_suite.normal only")
        raise ValueError(f"dtype argument to `normal` must be a float dtype, got {dtype}")
    shape = _shape(shape)
    size = int(np.prod(shape)) if len(shape) else 1
    a, p = _state(key)
    out = torch.empty(max(size, 1), dtype=torch.float32, device=_device())
    _n.check(_n.lib().d3p_chacha_normal_f32(p, 0, _n.ptr(out), size, _n.stream_ptr()), "normal")
    return out[:size].reshape(shape)


_INT_DTYPES = {torch.int8: (8, torch.int8), np.int8: (8, torch.int8), "int8": (8, torch.int8),
               torch.int16: (16, torch.int16), np.int16: (16, torch.int16), "int16": (16, torch.int16),
               torch.int32: (32, torch.int32), np.int32: (32, torch.int32), "int32": (32, torch.int32), int: (32, torch.int32),
               # jax.dtypes.canonicalize_dtype with x64 disabled (the default the reference runs under): int64 -> int32
               torch.int64: (32, torch.int32), np.int64: (32, torch.int32), "int64": (32, torch.int32)}


def randint(key: PRNGState, shape: Sequence[int], minval, maxval, dtype=torch.int32) -> torch.Tensor:
    """``d3p/random/__init__.py:84-146``: power-of-two mask + rejection on ``random_bits(round_key, nbits, shape)`` with
    nbits the width of the result type, one fresh key pair per round.  The whole rejection loop is one launch
    (``d3p_chacha_randint``), so the call never synchronises with the host and can be captured in a CUDA graph."""
    try:
        np_dt = np.dtype(dtype) if not isinstance(dtype, torch.dtype) else None
    except TypeError:
        np_dt = None
    if dtype not in _INT_DTYPES and not (np_dt is not None and np_dt.type in _INT_DTYPES):
        raise TypeError(f"dtype argument to `randint` must be an integer dtype, got {dtype}")
    nbits, out_dtype = _INT_DTYPES[dtype] if dtype in _INT_DTYPES else _INT_DTYPES[np_dt.type]
    shape = _shape(shape)
    size = int(np.prod(shape)) if len(shape) else 1
    # only the low nbits of the bounds matter (the arithmetic wraps in the result type); int64 carries them to C
    lo, hi = (((int(v) + (1 << 63)) & ((1 << 64) - 1)) - (1 << 63) for v in (minval, maxval))
    a, p = _state(key)
    out = torch.empty(max(size, 1), dtype=out_dtype, device=_device())
    _n.check(_n.lib().d3p_chacha_randint(p, nbits, lo, hi, _n.ptr(out), size, _n.stream_ptr()), "randint")
    return out[:size].reshape(shape)


def convert_to_jax_rng_key(rng_key: PRNGState) -> np.ndarray:
    """``d3p/random/__init__.py:149-155``: the first two keystream words (a Threefry key)."""
    return random_bits_host(rng_key, 2)
