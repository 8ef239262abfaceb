"""Similar-issue search throughput (code_intelligence_b200.similarity, csrc/knn.cu): one JSON line per configuration.

    python tools/knn_bench.py [--rows 1000000] [--self-rows 100000] [--warmup 2] [--reps 5] [--out FILE]

Workloads (seeded, encoder-like: convex mixes of the golden R4 encoder outputs plus small noise, built on the device):
  * an index of --rows x 2400 (1 M rows = 9.7 GB of split-bf16 residuals, far above the 126 MB L2), m in {1, 128, 1024}
    queries, k = 10;
  * a self-join (kneighbors(X=None)) of --self-rows rows, k = 10.
Timing: CUDA events around --reps calls after --warmup calls.  Each line reports ms per call, queries/s, index rows
scanned/s, the algorithmic bytes (index read once per 128-query pass: 4 * k_pad bytes a row) and tensor FLOPs (three
split-bf16 passes over the padded tiles) against the project's measured peaks (6.57 TB/s HBM, 1437 TFLOP/s bf16
sustained), the bound that binds, and the rank-wise cosine error against an f64 brute force on the device (first
128 queries).  A CPU numpy-f64 brute force on a subset of the index gives the host baseline.  The card name and power
limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import usable_cpus  # noqa: E402
from code_intelligence_b200.similarity import SimilarityIndex  # noqa: E402

HBM_TBS = 6.57
TFLOPS = 1437.0
D = 2400


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return {"gpu": name, "power_limit_w": pl}


def encoder_like(base, n, seed, noise=1e-3):
    """Device version of oracle.knn_ref.encoder_like (same recipe, torch RNG): (n, D) float32 cuda."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty((n, D), dtype=torch.float32, device="cuda")
    rms = float(base.double().pow(2).mean().sqrt())
    for r0 in range(0, n, 65536):
        m = min(65536, n - r0)
        pick = torch.randint(0, base.shape[0], (m, 3), generator=g, device="cuda")
        w = -torch.rand((m, 3), generator=g, device="cuda").log()
        w = w / w.sum(1, keepdim=True)
        out[r0:r0 + m] = torch.einsum("nj,njd->nd", w, base[pick])
        out[r0:r0 + m] += torch.randn((m, D), generator=g, device="cuda") * (noise * rms)
    return out


def rankwise_error(X, Q, ind, k, self_join=False):
    """Max |cos64(q, X[ind[j]]) - true j-th cos| on the device in f64."""
    Xu = torch.nn.functional.normalize(X.double(), dim=1)
    Qu = torch.nn.functional.normalize(Q.double(), dim=1)
    cos = Qu @ Xu.T
    if self_join:
        cos[torch.arange(len(Q)), torch.arange(len(Q))] = -2.0
    true = cos.topk(k, dim=1).values
    got = cos.gather(1, ind.to(cos.device))
    return float((got - true).abs().max())


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def line(kind, n, m, k, ms, info, err=None):
    k_pad = (D + 63) // 64 * 64
    n_pad = (n + 255) // 256 * 256
    passes = (m + 127) // 128
    byt = passes * n_pad * 4 * k_pad
    flop = 2.0 * 3 * passes * 128 * n_pad * k_pad
    t_mem = byt / (HBM_TBS * 1e12) * 1e3
    t_mma = flop / (TFLOPS * 1e12) * 1e3
    rec = {"kind": kind, "rows": n, "queries": m, "k": k, "d": D, "ms_per_call": round(ms, 4),
           "queries_per_s": round(m / ms * 1e3, 1), "rows_scanned_per_s": passes * n / ms * 1e3,
           "alg_bytes": byt, "hbm_tbs": round(byt / ms / 1e9, 3), "hbm_share": round(t_mem / ms, 3),
           "tensor_tflops": round(flop / ms / 1e9, 1), "tensor_share": round(t_mma / ms, 3),
           "bound_ms_hbm": round(t_mem, 4), "bound_ms_tensor": round(t_mma, 4),
           "binding_bound": "hbm" if t_mem >= t_mma else "tensor", **info}
    if err is not None:
        rec["rankwise_cos_error_vs_f64"] = err
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--self-rows", type=int, default=100_000)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu-rows", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("knn_bench.py measures the B200 path: no CUDA device")
    info = card()
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    base = torch.from_numpy(np.load(os.path.join(ROOT, "tests", "golden", "encoder_r4_b256_t512.npz"))["expected"]).cuda()
    X = encoder_like(base, a.rows, seed=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    index = SimilarityIndex(X)
    build_s = time.perf_counter() - t0
    emit({"kind": "build", "rows": a.rows, "d": D, "s": round(build_s, 3), "rows_per_s": round(a.rows / build_s, 1),
          "index_bytes": index.n * 4 * ((D + 63) // 64 * 64), **info})
    Qall = encoder_like(base, 1024, seed=2)
    for m in (1, 128, 1024):
        Q = Qall[:m].contiguous()
        ms = timed(lambda: index.kneighbors_device(Q, 10), a.warmup, a.reps)
        _, ind = index.kneighbors_device(Q[:128], 10)
        torch.cuda.synchronize()
        emit(line("query", a.rows, m, 10, ms, info, rankwise_error(X, Q[:128], ind, 10)))

    # CPU baseline: numpy f64 brute force of 128 queries against a subset of the index
    nc = min(a.cpu_rows, a.rows)
    Xc = X[:nc].cpu().numpy().astype(np.float64)
    Qc = Qall[:128].cpu().numpy().astype(np.float64)
    t0 = time.perf_counter()
    Xu = Xc / np.linalg.norm(Xc, axis=1, keepdims=True)
    Qu = Qc / np.linalg.norm(Qc, axis=1, keepdims=True)
    cos = Qu @ Xu.T
    np.argpartition(-cos, 10, axis=1)[:, :10]
    cpu_s = time.perf_counter() - t0
    emit({"kind": "cpu_baseline_numpy_f64", "rows": nc, "queries": 128, "k": 10, "d": D, "s": round(cpu_s, 3),
          "rows_scanned_per_s": round(128 * nc / cpu_s / 128, 1), "query_rows_per_s": round(128 * nc / cpu_s, 1),
          "usable_cpus": usable_cpus(), **info})
    del index, X
    torch.cuda.empty_cache()

    Xs = encoder_like(base, a.self_rows, seed=3)
    sidx = SimilarityIndex(Xs)
    ms = timed(lambda: sidx.kneighbors_device(None, 10), 1, max(1, a.reps // 2))
    _, ind = sidx.kneighbors_device(None, 10)
    torch.cuda.synchronize()
    err = rankwise_error(Xs, Xs[:128], ind[:128], 10, self_join=True)
    emit(line("self_join", a.self_rows, a.self_rows, 10, ms, info, err))
    sidx.close()
    if out:
        out.close()


if __name__ == "__main__":
    main()
