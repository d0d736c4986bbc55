"""Batchifiers of ``d3p/minibatch.py`` on the CUDA samplers of libd3p_b200.

``subsample_batchify_data`` (:136-239), ``poisson_batchify_data`` (:42-133) and
``split_batchify_data`` (:242-312) keep the reference signatures and return
``(init, get_batch)``; ``init(rng_key) -> (num_batches, state)``; ``get_batch(i, state)`` ->
``batch`` or ``(batch, mask)``.

Data set arrays live in HBM as torch CUDA tensors (host arrays are uploaded once).  Batches are
returned as ``BatchView`` objects: the index list produced by the sampler plus a reference to the
resident data set array.  ``DPSVI.update`` consumes the view directly, so each selected row is
read from HBM exactly once by the fused gradient kernel; anything else that needs the rows calls
``.tensor()`` (the masked row-gather kernel, ``mask * take(a, idxs)`` of minibatch.py:126-131).
"""
import ctypes as C

import numpy as np
import scipy.stats
import torch

from . import _native as _n
from . import random as strong_rng
from .util import example_count, sample_indices

__all__ = ["subsample_batchify_data", "split_batchify_data", "poisson_batchify_data",
           "q_to_batch_size", "batch_size_to_q", "BatchView", "gather_rows"]


def _device():
    if not torch.cuda.is_available():
        raise _n.D3PNativeError("d3p_b200 needs a CUDA device (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


def gather_rows(src: torch.Tensor, idx: torch.Tensor, num_valid: torch.Tensor = None) -> torch.Tensor:
    """``mask * take(src, idx, axis=0)`` with rows >= num_valid zero-filled (K4)."""
    src = src.contiguous()
    b = int(idx.shape[0])
    row_bytes = src[0].numel() * src.element_size() if src.shape[0] else 0
    out = torch.empty((b,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
    if b == 0 or row_bytes == 0:
        return out
    _n.check(_n.lib().d3p_gather_rows_masked(_n.ptr(src), row_bytes, _n.ptr(idx), _n.ptr(num_valid), b,
                                             _n.ptr(out), _n.stream_ptr()), "gather_rows_masked")
    return out


class BatchView:
    """A lazily gathered minibatch of one data set array: ``source[idx[:B]]`` with rows at
    positions >= ``num_valid`` (if given) replaced by zeros."""

    def __init__(self, source, idx, num_valid=None):
        self.source, self.idx, self.num_valid = source, idx, num_valid
        self._tensor = None

    @property
    def shape(self):
        return (int(self.idx.shape[0]),) + tuple(self.source.shape[1:])

    @property
    def dtype(self):
        return self.source.dtype

    @property
    def ndim(self):
        return len(self.shape)

    def __len__(self):
        return self.shape[0]

    def tensor(self) -> torch.Tensor:
        if self._tensor is None:
            self._tensor = gather_rows(self.source, self.idx, self.num_valid)
        return self._tensor

    def __getitem__(self, item):
        return self.tensor()[item]

    def __array__(self, dtype=None, copy=None):
        a = self.tensor().cpu().numpy()
        return a.astype(dtype) if dtype is not None else a

    def cpu(self):
        return self.tensor().cpu()

    def numpy(self):
        return self.tensor().cpu().numpy()


class LocalRows:
    """Rows ``[first, first + len(tensor))`` of a batch of ``batch_size`` examples whose other rows
    are handled by other ranks.  A sharded ``DPSVI.update`` (``parallel.shard_dpsvi``) accepts these
    in place of full batch arrays (and of the mask), so that with host-resident batches every rank
    uploads only the slice it processes; ``first`` must be the start of this rank's position range
    (``parallel.position_range``).  Keys stay addressed by the global batch position."""

    def __init__(self, tensor, first, batch_size):
        self.tensor, self.first, self.batch_size = tensor, int(first), int(batch_size)
        if self.first < 0 or self.first + tensor.shape[0] > self.batch_size:
            raise ValueError("LocalRows: the slice does not fit the batch")

    @property
    def shape(self):
        return (self.batch_size,) + tuple(self.tensor.shape[1:])

    def __len__(self):
        return self.batch_size


def _to_device(a):
    if isinstance(a, torch.Tensor):
        return a.to(_device()).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a)).to(_device())


def _validate(dataset):
    if not dataset:
        raise ValueError("The data set must not be empty")
    num_records = example_count(dataset[0])
    for arr in dataset:
        if num_records != example_count(arr):
            raise ValueError("All arrays constituting the data set must have the same number of records")
    return num_records


def q_to_batch_size(q, N):
    return int(N * q)


def batch_size_to_q(batch_size, N):
    return batch_size / N


def poisson_sample_idxs(rng_key, q, N, rng_suite=strong_rng, cutoff_size=None, suppress=False, workspace=None):
    """``d3p/minibatch.py:29-39`` (+ the truncate/suppress/mask logic of :119-124).

    Returns ``(idxs[cutoff] int32, counts[2] int32 = (num_selected, effective), mask[cutoff] bool)``
    as CUDA tensors; no host synchronisation."""
    if rng_suite is not strong_rng:
        raise NotImplementedError("d3p_b200 samplers are built on the ChaCha20 suite (d3p_b200.random)")
    if cutoff_size is None or cutoff_size > N:
        cutoff_size = N
    dev = _device()
    need = _n.lib().d3p_poisson_workspace_bytes(int(N))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    idx = torch.empty(max(cutoff_size, 1), dtype=torch.int32, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    mask = torch.empty(max(cutoff_size, 1), dtype=torch.uint8, device=dev)
    a = np.ascontiguousarray(np.asarray(rng_key, dtype=np.uint32).reshape(16))
    _n.check(_n.lib().d3p_poisson_sample(a.ctypes.data_as(C.POINTER(C.c_uint32)), float(np.float32(q)), int(N),
                                         int(cutoff_size), 1 if suppress else 0, _n.ptr(idx), _n.ptr(counts),
                                         _n.ptr(mask), _n.ptr(workspace), need, _n.stream_ptr()), "poisson_sample")
    return idx[:cutoff_size], counts, mask[:cutoff_size].view(torch.bool)


def poisson_batchify_data(dataset, q, max_batch_size, handle_oversized_batch="truncate", rng_suite=strong_rng):
    """``d3p/minibatch.py:42-133``."""
    if not dataset:
        raise ValueError("The data set must not be empty")
    if not isinstance(dataset, tuple):
        raise ValueError("Parameter dataset must be a tuple containing arrays of equal length.")
    if q < 0 or q > 1:
        raise ValueError("Parameter q must be >=0 and <=1.")
    num_records = _validate(dataset)
    if max_batch_size < 0:
        raise ValueError("max_batch_size must be a positive integer denoting the maximum batch size,"
                         " or a float between 0 and 1 denoting the maximum batch size in terms of Poisson"
                         " probability mass.")
    if not isinstance(max_batch_size, int):
        max_batch_size = int(scipy.stats.poisson(num_records * q).ppf(max_batch_size))
    dataset = tuple(_to_device(a) for a in dataset)
    suppress = handle_oversized_batch == "suppress"
    ws = torch.empty(_n.lib().d3p_poisson_workspace_bytes(int(num_records)), dtype=torch.uint8, device=_device())

    def init(rng_key):
        return num_records // int(q * num_records), rng_key

    def get_batch(i, batchifier_state):
        rng_key = rng_suite.fold_in(batchifier_state, i)
        idxs, counts, mask = poisson_sample_idxs(rng_key, q, num_records, rng_suite, cutoff_size=max_batch_size,
                                                 suppress=suppress, workspace=ws)
        num_valid = counts[1:2]
        return tuple(BatchView(a, idxs, num_valid) for a in dataset), mask

    # what DPSVI.run_epoch needs to drive this batchifier from C (d3p_dpsvi_run_epoch_meanfield)
    get_batch.spec = dict(kind=_n.SAMPLER_POISSON, q=float(np.float32(q)), n_records=num_records,
                          batch=int(max_batch_size), suppress=suppress, dataset=dataset, rng_suite=rng_suite)
    return init, get_batch


def subsample_batchify_data(dataset, batch_size=None, q=None, with_replacement=False, rng_suite=strong_rng,
                            return_mask=False):
    """``d3p/minibatch.py:136-239``."""
    if batch_size is None and q is None:
        raise ValueError("Either batch_size or batch ratio q must be given")
    if batch_size is not None and q is not None:
        raise ValueError("Only one of batch_size and batch ratio q must be given")
    num_records = _validate(dataset)
    if batch_size is None:
        batch_size = q_to_batch_size(q, num_records)
    dataset = tuple(_to_device(a) for a in dataset)

    def init(rng_key):
        return num_records // batch_size, rng_key

    def get_batch(i, batchifier_state):
        batch_rng_key = rng_suite.fold_in(batchifier_state, i)
        if with_replacement:
            ret_idx = rng_suite.randint(batch_rng_key, (batch_size,), 0, num_records)
        else:
            ret_idx = sample_indices(batch_rng_key, num_records, batch_size, rng_suite)
        batch = tuple(BatchView(a, ret_idx) for a in dataset)
        if return_mask:
            return batch, torch.ones(batch_size, dtype=torch.bool, device=ret_idx.device)
        return batch

    get_batch.spec = dict(kind=_n.SAMPLER_SUBSAMPLE_REPLACE if with_replacement else _n.SAMPLER_SUBSAMPLE, q=0.0,
                          n_records=num_records, batch=int(batch_size), suppress=False, dataset=dataset,
                          rng_suite=rng_suite)
    return init, get_batch


def split_batchify_data(dataset, batch_size=None, q=None, rng_suite=strong_rng, return_mask=False):
    """``d3p/minibatch.py:242-312``: one Feistel shuffle of all records per epoch."""
    if batch_size is None and q is None:
        raise ValueError("Either batch_size or batch ratio q must be given")
    if batch_size is not None and q is not None:
        raise ValueError("Only one of batch_size and batch ratio q must be given")
    num_records = _validate(dataset)
    if batch_size is None:
        batch_size = q_to_batch_size(q, num_records)
    dataset = tuple(_to_device(a) for a in dataset)

    def init(rng_key):
        return num_records // batch_size, sample_indices(rng_key, num_records, num_records, rng_suite)

    def get_batch(i, idxs):
        if not isinstance(idxs, torch.Tensor) or idxs.dtype != torch.int32 or not idxs.is_cuda:
            idxs = torch.as_tensor(np.asarray(idxs.cpu() if isinstance(idxs, torch.Tensor) else idxs)).to(
                device=_device(), dtype=torch.int32)           # any permutation the caller built itself
        ret_idx = idxs[i * batch_size:(i + 1) * batch_size]
        batch = tuple(BatchView(a, ret_idx) for a in dataset)
        if return_mask:
            return batch, torch.ones(batch_size, dtype=torch.bool, device=ret_idx.device)
        return batch

    # DPSVI.run_epoch: the epoch's shuffle (the state `init` returns) is the index list of every step
    get_batch.spec = dict(kind=_n.SAMPLER_SPLIT, q=0.0, n_records=num_records, batch=int(batch_size), suppress=False,
                          dataset=dataset, rng_suite=rng_suite)
    return init, get_batch
