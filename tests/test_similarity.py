"""Similar-issue search (code_intelligence_b200.similarity, csrc/knn.cu): exact cosine k-NN.

CPU: the f64 oracle against sklearn, and the precision design -- on the golden encoder outputs the numpy restatement of
the device arithmetic (centred split-bf16) meets the rank-wise tolerance while plain bf16 and plain f32 scoring do not.
GPU: parity with the f64 oracle, the reference notebook's one-shot labeler, bit-exact structural properties, edges.
"""
import os

import numpy as np
import pytest
import torch

from oracle import knn_ref as K

# Rank-wise tolerance in cosine: the emulation of the device arithmetic gives <= 2.5e-9 on the goldens, plain f32
# scoring >= 8e-8; 20x headroom for the tensor cores' accumulation order.
EPS = 5e-8
GOLDEN_SELF = ["encoder_r4_b256_t512", "encoder_n3_b64_t512", "encoder_r4_t1024", "encoder_r4_t2048", "encoder_n3"]


def golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))["expected"]


def assert_parity(X, Q, dist, ind, k):
    """|cos64(q, ids[j]) - oracle_cos[j]| <= EPS and |dist[j] - (1 - cos64(q, ids[j]))| <= EPS + 1.2e-7 dist[j]."""
    _, _, true_cos = K.brute_force(X, Q, k)
    assert dist.shape == ind.shape == true_cos.shape
    if Q is None:
        assert not (ind == np.arange(len(X))[:, None]).any(), "a self-query returned itself"
    assert ((ind >= 0) & (ind < len(X))).all()
    Qu = K.unit64(X if Q is None else Q)
    got_cos = np.einsum("md,mkd->mk", Qu, K.unit64(X)[ind])
    err = np.abs(got_cos - true_cos).max()
    assert err <= EPS, f"rank-wise cosine error {err:.3g}"
    derr = np.abs(dist.astype(np.float64) - (1.0 - got_cos)) - 1.2e-7 * np.abs(dist)
    assert derr.max() <= EPS, f"distance error {derr.max():.3g}"
    assert (np.diff(dist, axis=1) >= 0).all(), "distances not ascending"


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_matches_sklearn():
    from sklearn.neighbors import NearestNeighbors
    rng = np.random.default_rng(3)
    X = rng.standard_normal((300, 40))
    X[[5, 77]] = 0.0                                 # zero rows: cosine 0, distance 1
    X[10] = X[11]                                    # a duplicate pair
    Q = rng.standard_normal((17, 40))
    Q[3] = 0.0
    nn = NearestNeighbors(metric="cosine", algorithm="brute").fit(X)
    for q, k in [(None, 7), (Q, 7), (None, 299), (Q, 300)]:
        d_sk, i_sk = nn.kneighbors(q, n_neighbors=k)
        d, i, c = K.brute_force(X, q, k)
        np.testing.assert_allclose(d, d_sk, rtol=0, atol=1e-12)
        np.testing.assert_allclose(c, 1.0 - d, rtol=0, atol=1e-15)
        # equal distances may come in any order from sklearn; ours are in index order
        tie = np.isclose(d[:, 1:], d[:, :-1], rtol=0, atol=1e-12)
        assert (i[:, 1:][tie] > i[:, :-1][tie]).all()
        assert (i == i_sk)[~np.isclose(d, np.roll(d, 1, axis=1), rtol=0, atol=1e-12)
                           & ~np.isclose(d, np.roll(d, -1, axis=1), rtol=0, atol=1e-12)].all()
    d, i, _ = K.brute_force(X, None, 299)
    assert (d[5] == 1.0).all() and (d[77] == 1.0).all()
    assert i[10, 0] == 11 and i[11, 0] == 10
    dq, _, _ = K.brute_force(X, Q, 5)
    assert (dq[3] == 1.0).all()


@pytest.mark.parametrize("cols", [2400, 1600])
@pytest.mark.parametrize("name", GOLDEN_SELF)
def test_centred_split_emulation_meets_tolerance_where_plain_scoring_fails(golden_dir, name, cols):
    X = golden(golden_dir, name)[:, :cols]
    k = min(10, len(X) - 1)
    _, _, true_cos = K.brute_force(X, None, k)
    dist, ind = K.emulate_centred_split(X, None, k)
    assert K.rankwise_error(X, None, ind, true_cos) <= EPS
    np.testing.assert_allclose(dist, 1.0 - true_cos, rtol=1.2e-7, atol=EPS)
    assert K.rankwise_error(X, None, K.plain_scores(X, None, k, "f32"), true_cos) > EPS
    assert K.rankwise_error(X, None, K.plain_scores(X, None, k, "bf16"), true_cos) > EPS


def test_centred_split_emulation_out_of_distribution_queries(golden_dir):
    X = golden(golden_dir, "encoder_r4_b256_t512")
    Q = golden(golden_dir, "encoder_r4_varlen")
    _, _, true_cos = K.brute_force(X, Q, 10)
    _, ind = K.emulate_centred_split(X, Q, 10)
    assert K.rankwise_error(X, Q, ind, true_cos) <= EPS


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_similarity_index_has_no_cpu_fallback():
    from code_intelligence_b200.similarity import SimilarityIndex
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        SimilarityIndex(np.ones((4, 3), np.float32))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _index(X):
    from code_intelligence_b200.similarity import SimilarityIndex
    return SimilarityIndex(X)


@pytest.mark.gpu
@pytest.mark.parametrize("cols", [2400, 1600])
def test_parity_on_goldens(golden_dir, cols):
    for name in GOLDEN_SELF:
        X = golden(golden_dir, name)[:, :cols]
        k = min(10, len(X) - 1)
        idx = _index(X)
        dist, ind = idx.kneighbors(None, k)
        assert_parity(X, None, dist, ind, k)
        idx.close()
    X = golden(golden_dir, "encoder_r4_b256_t512")[:, :cols]
    idx = _index(X)
    for qname in ["encoder_r4_varlen", "encoder_r4", "encoder_n3_b64_t512"]:
        Q = golden(golden_dir, qname)[:, :cols]
        dist, ind = idx.kneighbors(Q, 10)
        assert_parity(X, Q, dist, ind, 10)
    idx.close()


@pytest.fixture(scope="module")
def crowded(golden_dir):
    base = golden(golden_dir, "encoder_r4_b256_t512")
    X = K.encoder_like(base, 150_000, 2400, seed=11)
    Q = K.encoder_like(base, 300, 2400, seed=12)
    return X, Q


@pytest.mark.gpu
def test_parity_encoder_like_150k(crowded):
    X, Q = crowded
    idx = _index(X)
    for k in (1, 2, 10, 32):
        dist, ind = idx.kneighbors(Q, k)
        assert_parity(X, Q, dist, ind, k)
    dist, ind = idx.kneighbors(X[1000:1300], 10)      # index rows as outside queries
    assert_parity(X, X[1000:1300], dist, ind, 10)
    idx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("d", [100, 800, 2401])
def test_parity_other_widths(golden_dir, d):
    base = golden(golden_dir, "encoder_r4_b256_t512")
    X = K.encoder_like(base, 20_000, d, seed=d)
    Q = K.encoder_like(base, 130, d, seed=d + 1)
    idx = _index(X)
    dist, ind = idx.kneighbors(Q, 10)
    assert_parity(X, Q, dist, ind, 10)
    sub = X[:700]
    idx2 = _index(sub)
    dist, ind = idx2.kneighbors(None, 5)
    assert_parity(sub, None, dist, ind, 5)
    idx.close()
    idx2.close()


@pytest.mark.gpu
def test_top1_matches_the_reference_one_shot_labeler(golden_dir):
    """tests/golden/similarity_ref.npz: the row the notebook's own oneshotlabeler.query chose (cosine scored in f32)."""
    z = np.load(os.path.join(golden_dir, "similarity_ref.npz"))
    X = np.load(os.path.join(golden_dir, str(z["index_source"])))["expected"]
    Q = np.concatenate([np.load(os.path.join(golden_dir, str(q)))["expected"] for q in z["query_sources"]])
    idx = _index(X)
    _, ind = idx.kneighbors(Q, 1)
    idx.close()
    cos = np.einsum("md,md->m", K.unit64(Q), K.unit64(X)[ind[:, 0]])
    ref_cos = np.einsum("md,md->m", K.unit64(Q), K.unit64(X)[z["top1"]])
    ok = (ind[:, 0] == z["top1"]) | (np.abs(cos - ref_cos) <= 1e-6)
    assert ok.all(), np.flatnonzero(~ok)
    assert (cos >= ref_cos - 1e-6).all()


@pytest.mark.gpu
def test_structural_bit_exact(crowded):
    import torch
    X, Q = crowded
    X = X[:40_000]
    Q = Q[:200]
    idx = _index(X)
    d_all, i_all = idx.kneighbors(Q, 10)
    for r in (0, 57, 128, 199):                      # independent of the other queries of the call
        d1, i1 = idx.kneighbors(Q[r:r + 1], 10)
        assert np.array_equal(d1[0], d_all[r]) and np.array_equal(i1[0], i_all[r])
    d2, i2 = idx.kneighbors(Q, 10)                   # repeated call
    assert np.array_equal(d2, d_all) and np.array_equal(i2, i_all)
    idx_b = _index(X)                                # separately built index
    d3, i3 = idx_b.kneighbors(Q, 10)
    assert np.array_equal(d3, d_all) and np.array_equal(i3, i_all)
    idx_b.close()
    idx_dev = _index(torch.from_numpy(X).cuda())     # built from a device tensor, queried with device pointers
    dd, di = idx_dev.kneighbors_device(torch.from_numpy(Q).cuda(), 10)
    torch.cuda.synchronize()
    assert np.array_equal(dd.cpu().numpy(), d_all) and np.array_equal(di.cpu().numpy(), i_all)
    ds, dsi = idx_dev.kneighbors_device(None, 4)
    hs, hsi = idx.kneighbors(None, 4)
    torch.cuda.synchronize()
    assert np.array_equal(ds.cpu().numpy(), hs) and np.array_equal(dsi.cpu().numpy(), hsi)
    idx_dev.close()
    # X=None with k equals the index rows queried from outside with k + 1, self removed (no duplicates in X)
    rows = X[:300]
    d_out, i_out = idx.kneighbors(rows, 6)
    assert (i_out[:, 0] == np.arange(300)).all()
    assert np.array_equal(hsi[:300], i_out[:, 1:5]) and np.array_equal(hs[:300], d_out[:, 1:5])
    idx.close()


@pytest.mark.gpu
def test_duplicates_come_back_in_id_order(crowded):
    X, _ = crowded
    X = X[:5000].copy()
    X[[100, 2000, 4999]] = X[7]
    idx = _index(X)
    dist, ind = idx.kneighbors(X[7:8], 4)
    assert list(ind[0]) == [7, 100, 2000, 4999]
    assert (dist[0] == dist[0, 0]).all()
    dist, ind = idx.kneighbors(None, 3)
    assert list(ind[100]) == [7, 2000, 4999] and (dist[100] == dist[100, 0]).all()
    idx.close()


@pytest.mark.gpu
def test_edges(golden_dir):
    rng = np.random.default_rng(5)
    base = golden(golden_dir, "encoder_r4_b256_t512")
    one = _index(rng.standard_normal((1, 30)).astype(np.float32))
    d, i = one.kneighbors(rng.standard_normal((3, 30)).astype(np.float32), 1)
    assert (i == 0).all()
    with pytest.raises(ValueError):
        one.kneighbors(None, 1)                      # a self-query of a one-row index has no candidate
    one.close()
    X = K.encoder_like(base, 20, 2400, seed=20)
    idx = _index(X)
    Q = K.encoder_like(base, 5, 2400, seed=21)
    d, i = idx.kneighbors(Q, 20)                     # k = n
    assert sorted(i[0]) == list(range(20))
    assert_parity(X, Q, d, i, 20)
    for bad_k in (21, 0, 33):
        with pytest.raises(ValueError):
            idx.kneighbors(Q, bad_k)
    with pytest.raises(ValueError):
        idx.kneighbors(None, 20)
    Qn = Q.copy()
    Qn[2, 3] = np.nan
    with pytest.raises(ValueError):
        idx.kneighbors(Qn, 3)
    d, i = idx.kneighbors(np.zeros((2, 2400), np.float32), 20)
    np.testing.assert_allclose(d, 1.0, rtol=0, atol=EPS)
    idx.close()
    Xn = X.copy()
    Xn[4, 4] = np.inf
    with pytest.raises(ValueError):
        _index(Xn)
    with pytest.raises(ValueError):
        _index(np.ones((3, 4097), np.float32))
    # zero index rows (a few in a realistic index; mu is the mean over all rows, so a large share of zero rows would
    # shrink it and widen the residuals): cosine 0 with everything, as queries and as neighbours
    Xz = K.encoder_like(base, 2000, 2400, seed=22)
    Xz[[3, 9]] = 0.0
    idx = _index(Xz)
    d, i = idx.kneighbors(None, 5)
    assert_parity(Xz, None, d, i, 5)
    np.testing.assert_allclose(d[[3, 9]], 1.0, rtol=0, atol=EPS + 1.2e-7)
    assert not np.isin(i[np.setdiff1d(np.arange(2000), [3, 9])], [3, 9]).any()
    idx.close()
