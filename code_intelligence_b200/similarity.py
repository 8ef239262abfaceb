"""Similar-issue search on the B200: exact cosine k-nearest neighbours over an index of issue embeddings.

The reference finds the issues closest to a given one by brute force on the host: the one-shot labeler of
Issue_Embeddings/notebooks/scratch/Kubeflow-FewShotLearning.ipynb (cell 46, ``CosineSimilarity`` against every labelled
issue, then ``argsort(descending=True)``) and ``KNeighborsClassifier(n_neighbors=2, weights='distance',
metric='cosine')`` (cell 77).  ``SimilarityIndex`` answers the same question with the interface of
``sklearn.neighbors.NearestNeighbors(metric='cosine', algorithm='brute').kneighbors`` through ``ie_knn_*``
(include/issue_emb_b200.h, csrc/knn.cu): one fused tensor-core GEMM + top-k pass over the index per 128 queries.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import check

MAX_NEIGHBORS = 32
SELF_CHUNK = 1 << 16     # rows per ie_knn_search call of a self-join (bounds the host-side result staging)


class SimilarityIndex:
    """Index of ``vectors`` (n, d) float32 -- an ndarray or a CUDA tensor, e.g. the output of ``encode_id_list`` or
    ``features[:, :1600]`` -- for exact cosine-distance neighbour queries.  1 <= d <= 4096; zero rows are allowed (cosine
    0 with everything, as in sklearn)."""

    def __init__(self, vectors, device: int = 0):
        self._lib = _lib.load()
        self._h = None
        h = C.c_void_p()
        if _is_cuda_tensor(vectors):
            import torch
            if vectors.dtype != torch.float32 or vectors.dim() != 2:
                raise ValueError(f"vectors must be a 2-d float32 tensor, got {vectors.dtype} {tuple(vectors.shape)}")
            v = vectors.contiguous()
            s = torch.cuda.current_stream(v.device)
            check(self._lib.ie_knn_create(v.data_ptr(), v.shape[0], v.shape[1], v.device.index, _lib.IE_FLAG_DEVICE_PTRS,
                                          C.c_void_p(s.cuda_stream), C.byref(h)))
            self.device = v.device.index
        else:
            v = np.ascontiguousarray(np.asarray(vectors), dtype=np.float32)
            if v.ndim != 2:
                raise ValueError(f"vectors must be (n, d), got shape {v.shape}")
            check(self._lib.ie_knn_create(v.ctypes.data, v.shape[0], v.shape[1], device, 0, None, C.byref(h)))
            self.device = device
        self._h = h
        self.n, self.d = int(v.shape[0]), int(v.shape[1])

    def kneighbors(self, X=None, n_neighbors: int = 5, return_distance: bool = True):
        """sklearn ``NearestNeighbors.kneighbors``: X (m, d) -> (dist (m, k) float32, ind (m, k) int64), cosine distance
        1 - cos ascending, ties by the smaller index.  ``X=None`` queries every index row against the others (a row is
        not its own neighbour)."""
        k = int(n_neighbors)
        if X is None:
            dist = np.empty((self.n, k), dtype=np.float32)
            ind = np.empty((self.n, k), dtype=np.int64)
            for r0 in range(0, self.n, SELF_CHUNK):
                m = min(SELF_CHUNK, self.n - r0)
                check(self._lib.ie_knn_search(self._h, None, r0, m, k, dist[r0:].ctypes.data, ind[r0:].ctypes.data,
                                              0, None))
        else:
            Q = np.ascontiguousarray(np.asarray(X), dtype=np.float32)
            if Q.ndim != 2 or Q.shape[1] != self.d:
                raise ValueError(f"X must be (m, {self.d}), got shape {Q.shape}")
            dist = np.empty((Q.shape[0], k), dtype=np.float32)
            ind = np.empty((Q.shape[0], k), dtype=np.int64)
            if Q.shape[0]:
                check(self._lib.ie_knn_search(self._h, Q.ctypes.data, 0, Q.shape[0], k, dist.ctypes.data,
                                              ind.ctypes.data, 0, None))
        return (dist, ind) if return_distance else ind

    def kneighbors_device(self, X=None, n_neighbors: int = 5, stream=None):
        """Asynchronous device-resident variant: X cuda float32 (m, d), or None for the self-join, -> (dist cuda float32
        (m, k), ind cuda int64 (m, k)) on `stream` (default: torch's current stream)."""
        import torch
        k = int(n_neighbors)
        dev = torch.device("cuda", self.device)
        if X is None:
            m, qptr = self.n, None
        else:
            if not (X.is_cuda and X.dtype == torch.float32 and X.dim() == 2 and X.shape[1] == self.d):
                raise ValueError(f"X must be a cuda float32 tensor of shape (m, {self.d})")
            X = X.contiguous()
            m, qptr, dev = X.shape[0], X.data_ptr(), X.device
        dist = torch.empty((m, k), dtype=torch.float32, device=dev)
        ind = torch.empty((m, k), dtype=torch.int64, device=dev)
        s = stream if stream is not None else torch.cuda.current_stream(dev)
        if m:
            check(self._lib.ie_knn_search(self._h, qptr, 0, m, k, dist.data_ptr(), ind.data_ptr(),
                                          _lib.IE_FLAG_DEVICE_PTRS, C.c_void_p(s.cuda_stream)))
        return dist, ind

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ie_knn_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _is_cuda_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False)
