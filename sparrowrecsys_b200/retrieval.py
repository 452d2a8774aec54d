"""Candidate retrieval on the device: exact top-k dot / cosine search over an item index in HBM.

The recall stage in front of the rankers: `SimilarMovieProcess.retrievalCandidatesByEmbedding`
(`online/recprocess/SimilarMovieProcess.java:91-112`) scores the whole catalog by embedding cosine,
and `RecForYouProcess.getRecList` (`:34-35`) starts from a fixed candidate list.  `ItemIndex` holds the
catalog once (`srs_index_create`) and answers a batch of queries per call (`srs_index_search_*`); the
positions it returns feed `CTRModel.rank_user`.  Results are the most similar first (the reference's
`retrievalCandidatesByEmbedding` sorts ascending; see INTEGRATION.md).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

METRICS = {"dot": _lib.SRS_DOT, "cosine": _lib.SRS_COSINE}


class ItemIndex:
    """Exact top-k index over `items` [n, dim] float32 (dim <= 128).  A numpy array is copied to the
    device; a contiguous float32 CUDA tensor is used in place (it must stay alive with the index)."""

    def __init__(self, items, metric: str = "dot", device: int = 0):
        if metric not in METRICS:
            raise ValueError("metric must be 'dot' or 'cosine'")
        self._h = None
        self._lib = _lib.load()
        self.metric = metric
        if isinstance(items, np.ndarray):
            a = np.ascontiguousarray(items, np.float32)
            ptr, loc, self._items = a.ctypes.data, _lib.SRS_HOST, None
            self.device = int(device)
        else:
            if str(items.dtype) != "torch.float32" or not items.is_cuda or not items.is_contiguous():
                raise ValueError("a device item table must be a contiguous float32 CUDA tensor")
            a = items
            ptr, loc, self._items = items.data_ptr(), _lib.SRS_DEVICE_BORROWED, items
            self.device = items.device.index or 0
        if a.ndim != 2:
            raise ValueError("items [n, dim] expected")
        self.n, self.dim = int(a.shape[0]), int(a.shape[1])
        h = C.c_void_p()
        _lib.check(self._lib.srs_index_create(ptr, self.n, self.dim, METRICS[metric], loc, self.device, C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._lib.srs_index_destroy(self._h)
            self._h = None
        self._items = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def search(self, queries, k: int, exclude=None):
        """`queries` [q, dim] (or [dim]) -> (positions int32 [q, k], scores float32 [q, k]) as numpy, best
        first; `exclude` [q] positions to leave out (-1 = none).  Unused slots: position -1, score 0."""
        q = np.ascontiguousarray(queries, np.float32)
        q = q.reshape(1, -1) if q.ndim == 1 else q
        nq, k = q.shape[0], int(k)
        pos = np.empty((nq, max(k, 0)), np.int32)
        top = np.empty((nq, max(k, 0)), np.float32)
        ex = None if exclude is None else np.ascontiguousarray(np.broadcast_to(exclude, (nq,)), np.int32)
        _lib.check(self._lib.srs_index_search_host(self._h, q.ctypes.data, nq, q.shape[1], k,
                                                   None if ex is None else ex.ctypes.data,
                                                   pos.ctypes.data, top.ctypes.data))
        return pos, top

    def search_device(self, queries, k: int, exclude=None, stream=None):
        """Device variant: `queries` a float32 CUDA tensor [q, dim], `exclude` an int32 CUDA tensor [q] or
        None; returns (positions, scores) CUDA tensors [q, k] queued on `stream` (default: current)."""
        import torch
        if queries.dtype != torch.float32 or not queries.is_cuda or queries.dim() != 2 \
                or not queries.is_contiguous():
            raise ValueError("queries must be a contiguous [q, dim] float32 CUDA tensor")
        if exclude is not None and (exclude.dtype != torch.int32 or not exclude.is_cuda
                                    or not exclude.is_contiguous()):
            raise ValueError("exclude must be a contiguous int32 CUDA tensor")
        nq, k = queries.shape[0], int(k)
        pos = torch.empty((nq, max(k, 0)), dtype=torch.int32, device=queries.device)
        top = torch.empty((nq, max(k, 0)), dtype=torch.float32, device=queries.device)
        if stream is None:
            stream = torch.cuda.current_stream(queries.device)
        _lib.check(self._lib.srs_index_search_device(self._h, queries.data_ptr(), nq, queries.shape[1], k,
                                                     None if exclude is None else exclude.data_ptr(),
                                                     pos.data_ptr(), top.data_ptr(), stream.cuda_stream))
        return pos, top
