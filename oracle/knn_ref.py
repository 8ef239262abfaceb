"""CPU oracle of the similar-issue search (csrc/knn.cu): f64 brute-force cosine k-NN, a numpy restatement of the
device arithmetic (centred split-bf16), the plain scorings it replaces, and the rank-wise error the tests measure.

Conventions are sklearn ``NearestNeighbors(metric='cosine', algorithm='brute').kneighbors``: distance = 1 - cos,
ascending, ties by the smaller index; a zero vector has cosine 0 with everything; ``Q=None`` queries every index row
against the others.
"""
from __future__ import annotations

import numpy as np


def unit64(X) -> np.ndarray:
    X = np.asarray(X, dtype=np.float64)
    nrm = np.sqrt(np.einsum("ij,ij->i", X, X))
    return X / np.where(nrm > 0, nrm, 1.0)[:, None]


def _select(scores: np.ndarray, k: int, exclude: np.ndarray | None):
    """Top-k of each row of `scores` by (score descending, column ascending); `exclude[i]` = column row i skips."""
    s = scores.copy()
    if exclude is not None:
        s[np.arange(len(s)), exclude] = -np.inf
    ids = np.broadcast_to(np.arange(s.shape[1]), s.shape)
    order = np.lexsort((ids, -s), axis=1)[:, :k]
    return order


def cosines64(Q, X, chunk: int = 4096) -> np.ndarray:
    """f64 cosine matrix (m, n), chunked over the queries."""
    Xu = unit64(X)
    Qu = unit64(Q)
    out = np.empty((Qu.shape[0], Xu.shape[0]), dtype=np.float64)
    for q0 in range(0, Qu.shape[0], chunk):
        out[q0:q0 + chunk] = Qu[q0:q0 + chunk] @ Xu.T
    return out


def brute_force(X, Q=None, k: int = 5):
    """f64 truth -> (dist (m, k) f64, ind (m, k) int64, cos (m, k) f64).  Q=None: self-join without self."""
    self_join = Q is None
    cos = cosines64(X if self_join else Q, X)
    ind = _select(cos, k, np.arange(len(cos)) if self_join else None)
    c = np.take_along_axis(cos, ind, axis=1)
    return 1.0 - c, ind.astype(np.int64), c


def bf16(x) -> np.ndarray:
    """Round f32 to bf16 (nearest even), returned as f32."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def _split_gemm(A, B) -> np.ndarray:
    """Split-bf16 product [A_hi | A_lo | A_hi] x [B_hi | B_hi | B_lo]^T (exact products, sum rounded to f32)."""
    Ah = bf16(A)
    Al = bf16(A - Ah)
    Bh = bf16(B)
    Bl = bf16(B - Bh)
    Ah, Al, Bh, Bl = (v.astype(np.float64) for v in (Ah, Al, Bh, Bl))
    return (Ah @ Bh.T + Al @ Bh.T + Ah @ Bl.T).astype(np.float32)


def emulate_centred_split(X, Q=None, k: int = 5):
    """The device arithmetic of csrc/knn.cu restated in numpy -> (dist (m, k) f32, ind (m, k) int64).
    mu = mean of the f64 unit vectors; r = f32(x^ - mu), b = f32(mu . r), c = x^ . mu (f64); score t = f32(split-bf16
    GEMM of s_q and r_x) + b_x in f32; ranking by (t desc, id asc); distance = f32((1 - c_q) - t) in f64."""
    self_join = Q is None
    Xu = unit64(X)
    mu = Xu.mean(axis=0)
    r = (Xu - mu).astype(np.float32)
    b = (r.astype(np.float64) @ mu).astype(np.float32)
    if self_join:
        s, c = r, Xu @ mu
    else:
        Qu = unit64(Q)
        s, c = (Qu - mu).astype(np.float32), Qu @ mu
    t = _split_gemm(s, r) + b[None, :]
    ind = _select(t, k, np.arange(len(t)) if self_join else None)
    tk = np.take_along_axis(t, ind, axis=1).astype(np.float64)
    dist = ((1.0 - c)[:, None] - tk).astype(np.float32)
    return dist, ind.astype(np.int64)


def plain_scores(X, Q=None, k: int = 5, mode: str = "f32"):
    """What a plain search would return: dot products of unit vectors rounded to f32 ("f32") or bf16 ("bf16")
    operands with an f32 result -> ind (m, k)."""
    self_join = Q is None
    Xu = unit64(X).astype(np.float32)
    Qu = Xu if self_join else unit64(Q).astype(np.float32)
    if mode == "bf16":
        t = (bf16(Qu).astype(np.float64) @ bf16(Xu).astype(np.float64).T).astype(np.float32)
    else:
        t = Qu @ Xu.T
    return _select(t, k, np.arange(len(t)) if self_join else None).astype(np.int64)


def encoder_like(base, n: int, d: int, seed: int, noise: float = 1e-3) -> np.ndarray:
    """Seeded (n, d) float32 set crowded like encoder outputs: each row a convex mix of three rows of `base` (golden
    encoder outputs) plus Gaussian noise of `noise` x the base's RMS; columns taken cyclically from the base's."""
    rng = np.random.default_rng(seed)
    B = np.asarray(base, dtype=np.float32)[:, np.arange(d) % base.shape[1]]
    pick = rng.integers(0, len(B), size=(n, 3))
    w = rng.dirichlet(np.ones(3), size=n).astype(np.float32)
    out = np.einsum("nj,njd->nd", w, B[pick]) if n * d <= (1 << 22) else None
    if out is None:
        out = np.empty((n, d), dtype=np.float32)
        for r0 in range(0, n, 4096):
            out[r0:r0 + 4096] = np.einsum("nj,njd->nd", w[r0:r0 + 4096], B[pick[r0:r0 + 4096]])
    rms = float(np.sqrt(np.mean(B.astype(np.float64) ** 2)))
    out += rng.standard_normal((n, d), dtype=np.float32) * np.float32(noise * rms)
    return out


def rankwise_error(X, Q, ind, true_cos) -> float:
    """max over queries and ranks j of |cos64(q, X[ind[j]]) - true_cos[j]| (Q=None: the rows of X)."""
    Qu = unit64(X if Q is None else Q)
    Xu = unit64(X)
    got = np.einsum("md,mkd->mk", Qu, Xu[ind])
    return float(np.abs(got - true_cos).max())
