"""Pins the CPU oracle against the reference's own known-answer tests (SURVEY §8c).

Each case re-types the fixed vectors of a reference unit test and asserts what that test asserts
(SIMD tier == scalar tier, exactly), plus the hand-computable value.  Sources:
  f32 : lib/segment/src/spaces/simple_avx.rs:218-256, simple_sse.rs:206-..., simple.rs:248-277
  u8  : lib/segment/src/spaces/metric_uint/avx2/{dot.rs:77-106,cosine.rs:112-170,euclid.rs,manhattan.rs}
  topk: lib/segment/src/spaces/tools.rs:64-75
  SQ8/BQ inner loops: the reference's C kernels compiled verbatim (oracle/_ref/libsimd_utils.so); their results on the
        seeded inputs below are stored in tests/golden/ref_kernels_kat.npz (tests/golden/make_golden.py)
"""
import ctypes as C
import os

import numpy as np

REF_KAT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels_kat.npz")


def f32_kat():
    base = list(range(10, 26))
    v1 = base * 4 + [26, 27, 28, 29, 30, 31]
    v2 = list(range(40, 56)) + base * 3 + [56, 57, 58, 59, 60, 61]
    return np.array(v1, np.float32), np.array(v2, np.float32)


def u8_kat():
    a = [255, 255, 0] + list(range(1, 18))
    v1 = a * 5
    b0 = [255, 255, 0] + list(range(254, 237, -1))
    b = [255, 255, 255] + list(range(254, 237, -1))
    v2 = b0 + b * 4
    assert len(v1) == 100 and len(v2) == 100
    return np.array(v1, np.uint8), np.array(v2, np.uint8)


def test_f32_avx_equals_scalar_kat(oracle):
    v1, v2 = f32_kat()
    assert v1.size == 70
    for name in ("euclid", "manhattan", "dot"):
        assert oracle.raw_f32(name, "avx", v1, v2) == oracle.raw_f32(name, "scalar", v1, v2), name
    # hand-computable: first 16 differ by 30, last 6 by 30 -> 22 * 900 ; manhattan 22 * 30
    assert oracle.raw_f32("euclid", "avx", v1, v2) == np.float32(-22 * 900)
    assert oracle.raw_f32("manhattan", "avx", v1, v2) == np.float32(-22 * 30)
    assert oracle.raw_f32("dot", "avx", v1, v2) == np.float32(np.dot(v1.astype(np.float64), v2.astype(np.float64)))
    np.testing.assert_array_equal(oracle.raw_cosine_preprocess("avx", v1), oracle.raw_cosine_preprocess("scalar", v1))


def test_f32_sse_equals_scalar_kat(oracle):
    v1, v2 = f32_kat()
    for name in ("euclid", "manhattan", "dot"):
        assert oracle.raw_f32(name, "sse", v1, v2) == oracle.raw_f32(name, "scalar", v1, v2), name
    np.testing.assert_array_equal(oracle.raw_cosine_preprocess("sse", v1), oracle.raw_cosine_preprocess("scalar", v1))


def test_cosine_preprocess_zero_and_stable(oracle):
    # simple.rs:248-252
    z = np.zeros(4, np.float32)
    np.testing.assert_array_equal(oracle.preprocess_f32(oracle.COSINE, z), z)
    # simple.rs:256-277: re-normalising a normalised vector is a fixed point (100 x 1500-d)
    rng = np.random.default_rng(1)
    for _ in range(100):
        v = rng.uniform(-1, 1, 1500).astype(np.float32)
        p1 = oracle.preprocess_f32(oracle.COSINE, v)
        p2 = oracle.preprocess_f32(oracle.COSINE, p1)
        np.testing.assert_array_equal(p1, p2)


def test_dispatch_tiers(oracle):
    rng = np.random.default_rng(5)
    for dim, tier in ((8, "scalar"), (15, "scalar"), (16, "sse"), (31, "sse"), (32, "avx"), (70, "avx"), (768, "avx")):
        a, b = rng.standard_normal(dim).astype(np.float32), rng.standard_normal(dim).astype(np.float32)
        assert oracle.similarity_f32(oracle.DOT, a, b) == oracle.raw_f32("dot", tier, a, b)
        assert oracle.similarity_f32(oracle.COSINE, a, b) == oracle.raw_f32("dot", tier, a, b)
        assert oracle.similarity_f32(oracle.EUCLID, a, b) == oracle.raw_f32("euclid", tier, a, b)
        assert oracle.similarity_f32(oracle.MANHATTAN, a, b) == oracle.raw_f32("manhattan", tier, a, b)


def test_postprocess(oracle):
    assert oracle.postprocess_f32(oracle.EUCLID, -9.0) == np.float32(3.0)
    assert oracle.postprocess_f32(oracle.MANHATTAN, -9.0) == np.float32(9.0)
    assert oracle.postprocess_f32(oracle.DOT, -9.0) == np.float32(-9.0)


def test_u8_avx_equals_scalar_kat(oracle):
    v1, v2 = u8_kat()
    for name in ("dot", "cosine", "euclid", "manhattan"):
        assert oracle.raw_u8(name, "avx", v1, v2) == oracle.raw_u8(name, "scalar", v1, v2), name
    d = int(np.dot(v1.astype(np.int64), v2.astype(np.int64)))
    assert oracle.raw_u8("dot", "avx", v1, v2) == np.float32(d)


def test_u8_cosine_zero(oracle):
    # metric_uint/avx2/cosine.rs:148-166 and simple_cosine.rs:80-87
    v1 = np.zeros(8, np.uint8)
    v2 = np.array([255, 255, 0, 254, 253, 252, 251, 250], np.uint8)
    for tier in ("avx", "scalar"):
        assert oracle.raw_u8("cosine", tier, v1, v2) == 0.0
        assert oracle.raw_u8("cosine", tier, v2, v1) == 0.0
        assert oracle.raw_u8("cosine", tier, v1, v1) == 0.0


def test_peek_top_kat(oracle):
    # tools.rs:64-75
    data = np.array([10, 20, 40, 5, 100, 33, 84, 65, 20, 43, 44, 42], np.float32)
    res = oracle.topk(data, 3)
    assert list(res["score"]) == [100.0, 84.0, 65.0]
    assert list(res["idx"]) == [4, 6, 7]
    res = oracle.topk(-data, 3)
    assert list(-res["score"]) == [5.0, 10.0, 20.0]
    assert oracle.topk(data, 0).size == 0
    assert oracle.topk(data, 100).size == data.size  # fewer points than top


def test_topk_matches_sort(oracle):
    rng = np.random.default_rng(3)
    s = rng.standard_normal(5000).astype(np.float32)
    res = oracle.topk(s, 17)
    order = np.argsort(-s, kind="stable")[:17]
    np.testing.assert_array_equal(res["score"], s[order])
    np.testing.assert_array_equal(res["idx"], order.astype(np.uint32))


def sq8_kat_codes():
    """(dim, query code, row code): random and extreme 7-bit codes, seeded."""
    rng = np.random.default_rng(42)
    for dim in (16, 32, 48, 64, 80, 768, 784, 1536, 4096):
        for trial in range(20):
            q = rng.integers(0, 128, dim, dtype=np.uint8)
            v = rng.integers(0, 128, dim, dtype=np.uint8)
            if trial == 0:
                q[:] = 127; v[:] = 127
            if trial == 1:
                q[:] = 0
            yield dim, q, v


def bq_kat_vectors():
    """(dim, 4 stored f32 vectors, f32 query), seeded."""
    rng = np.random.default_rng(9)
    for dim in (1, 127, 128, 129, 768, 1000, 1536):
        data = rng.standard_normal((4, dim)).astype(np.float32)
        q = rng.standard_normal(dim).astype(np.float32)
        yield dim, data, q


def test_sq8_inner_loops_match_reference_c(oracle):
    """oracle restatement == the reference's own avx2.c / sse.c compiled verbatim, on random + extreme codes."""
    R = np.load(REF_KAT)
    L = oracle.lib()
    u8p = C.POINTER(C.c_uint8)
    for c, (dim, q, v) in enumerate(sq8_kat_codes()):
        qp, vp = q.ctypes.data_as(u8p), v.ctypes.data_as(u8p)
        assert L.qo_sq8_dot_avx(qp, vp, dim) == R["sq8_dot_avx"][c], (c, dim)
        assert L.qo_sq8_l1_avx(qp, vp, dim) == R["sq8_l1_avx"][c], (c, dim)
        # the SSE tier is the same integers for dims whose sums stay < 2^24 (exactness window)
        if dim <= 1040:
            assert R["sq8_dot_sse"][c] == R["sq8_dot_avx"][c]
            assert R["sq8_dot_avx"][c] == np.float32(int(np.dot(q.astype(np.int64), v.astype(np.int64)))), (c, dim)
    assert R["sq8_dot_avx"].size == c + 1


def test_bq_popcount_matches_reference_c(oracle):
    R = np.load(REF_KAT)
    for c, (dim, data, q) in enumerate(bq_kat_vectors()):
        for qenc, bits, tag in ((oracle.BQQ_SCALAR8, 8, "s8"), (oracle.BQQ_SCALAR4, 4, "s4")):
            bq = oracle.BQ.encode(data, oracle.BQ_ONE, qenc, oracle.QD_DOT, False)
            qe = bq.encode_query(q)
            for i in range(data.shape[0]):
                x = int(R["bq_xor_" + tag][c, i])      # impl_xor_popcnt_scalar{8,4}_avx_uint128(query, row i)
                xf = np.float32(x) / np.float32((1 << bits) - 1)
                zeros = np.float32(dim) - xf
                assert bq.score(qe, i) == zeros - xf
        bq = oracle.BQ.encode(data, oracle.BQ_ONE, oracle.BQQ_SAME, oracle.QD_DOT, False)
        qe = bq.encode_query(q)
        for i in range(data.shape[0]):
            x = int(R["bq_xor_bin"][c, i])              # impl_xor_popcnt_sse_uint128(query, row i)
            assert bq.score(qe, i) == np.float32(dim - x) - np.float32(x)
            bits_q = (q > 0)
            bits_v = (data[i] > 0)
            assert x == int(np.sum(bits_q != bits_v))
    assert R["bq_xor_bin"].shape[0] == c + 1


def test_f16_avx_vs_scalar_tolerance(oracle):
    # metric_f16/avx/dot.rs:82-124: 256-element vectors in [1, 8], |simd - scalar| / |scalar| < 5e-4
    rng = np.random.default_rng(16)
    v1 = (rng.integers(10, 80, 256) / 10.0).astype(np.float32).astype(np.float16)
    v2 = (rng.integers(10, 80, 256) / 10.0).astype(np.float32).astype(np.float16)
    simd = oracle.raw_f16("dot_avx", v1, v2)
    scalar = oracle.raw_f16("dot_scalar", v1, v2)
    assert abs(simd - scalar) / abs(scalar) < 0.0005
    exact = float(np.dot(v1.astype(np.float64), v2.astype(np.float64)))
    assert abs(simd - exact) / exact < 1e-5
    assert oracle.similarity_f16(oracle.DOT, v1, v2) == simd
    assert oracle.similarity_f16(oracle.COSINE, v1, v2) == simd  # f16 cosine == dot (simple_cosine.rs:28-58)


# ------------------------------------------------------------------------------------------------ custom queries
def test_reco_best_score_reference_table(oracle):
    """reco_query.rs:150-185 `score_query` rstest table (dummy similarity = the example itself)."""
    cases = [([42], [4], "P", 42.0), ([4], [42], "N", 42.0), ([-1], [0], "N", 0.0), ([0], [-1], "P", 0.0), ([-42], [-84], "P", -42.0),
             ([-84], [-42], "N", -42.0), ([1, 2, 3], [4, 5, 6], "N", 6.0), ([10, 2, 3], [4, 5, 6], "P", 10.0)]
    for pos, neg, chosen, expected in cases:
        got = oracle.custom_score(oracle.RECO_BEST_SCORE, len(pos), len(neg), np.array(pos + neg, np.float32))
        want = oracle.scaled_fast_sigmoid(expected) if chosen == "P" else -oracle.scaled_fast_sigmoid(expected)
        assert got == want, (pos, neg)
    # math.rs:7-18
    assert oracle.fast_sigmoid(3.0) == np.float32(3.0) / np.float32(4.0)
    assert oracle.scaled_fast_sigmoid(-1.0) == np.float32(0.25)


def test_reco_best_score_order_properties(oracle):
    """reco_query.rs:204-262 proptests: negatives invert the order, positives keep it, positive-chosen >= negative-chosen."""
    rng = np.random.default_rng(0)
    for _ in range(500):
        a, b = (np.float32(x) for x in rng.uniform(-100, 100, 2))
        pa, pb = (oracle.custom_score(oracle.RECO_BEST_SCORE, 1, 0, np.array([x], np.float32)) for x in (a, b))
        na, nb = (oracle.custom_score(oracle.RECO_BEST_SCORE, 0, 1, np.array([x], np.float32)) for x in (a, b))
        if a < b:
            assert pa <= pb and na >= nb
        assert pa >= nb and pb >= na


def test_discover_rank_reference_table(oracle):
    """discover_query.rs:100-125 `context_ranking` rstest table; score = rank + scaled_fast_sigmoid(target) (:66-76)."""
    cases = [([], 0), ([(10, 4)], 1), ([(4, 10)], -1), ([(11, 11)], 0), ([(10, 4), (4, 10)], 0), ([(10, 4), (4, 2)], 2), ([(4, 10), (2, 4)], -2),
             ([(1, 0), (2, 0), (3, 0), (4, 0), (5, 0), (0, 4)], 4)]
    for pairs, rank in cases:
        sims = np.array([42.0] + [x for p in pairs for x in p], np.float32)
        got = oracle.custom_score(oracle.DISCOVER, len(pairs), 0, sims)
        assert got == np.float32(rank) + oracle.scaled_fast_sigmoid(42.0), pairs


def test_context_loss_bounds_and_sum(oracle):
    """context_query.rs:146-160: per-pair loss in (-1, 0]; :111-119: the score is the sequential f32 sum of the losses."""
    rng = np.random.default_rng(1)
    for _ in range(1000):
        p, n = (np.float32(x) for x in rng.uniform(-100, 100, 2))
        s = oracle.custom_score(oracle.CONTEXT, 1, 0, np.array([p, n], np.float32))
        assert -1.0 < s <= 0.0
        if p > n + np.float32(1e-3):
            assert s == 0.0
    sims = np.array([1.0, 3.0, 5.0, 2.0, -2.0, 0.5], np.float32)  # pairs (1,3) (5,2) (-2,0.5)
    eps = np.float32(np.finfo(np.float32).eps)
    want = np.float32(0.0)
    for p, n in [(1.0, 3.0), (5.0, 2.0), (-2.0, 0.5)]:
        d = min(np.float32(np.float32(p) - np.float32(n)) - eps, np.float32(0.0))
        want = np.float32(want + np.float32(d / np.float32(np.float32(1.0) + abs(d))))
    assert oracle.custom_score(oracle.CONTEXT, 3, 0, sims) == want


def test_reco_sum_scores(oracle):
    sims = np.array([0.1, 0.2, 0.7, 0.05], np.float32)
    want = np.float32(np.float32(np.float32(0.0) + sims[0]) + sims[1]) - np.float32(np.float32(np.float32(0.0) + sims[2]) + sims[3])
    assert oracle.custom_score(oracle.RECO_SUM_SCORES, 2, 2, sims) == np.float32(want)
    m = np.stack([sims, sims[::-1]], axis=1)  # two candidates
    out = oracle.custom_combine(oracle.RECO_SUM_SCORES, 2, 2, m)
    assert out[0] == np.float32(want) and out.shape == (2,)


def test_maxsim_reference_kat(oracle):
    """query_scorer/mod.rs:168-184 test_score_multi_euclidean: score(a, a) == -0.0 and score(a, b) == -19."""
    a = np.array([[1.0, 2.0, 3.0], [3.0, 3.0, 3.0], [4.0, 5.0, 6.0]], np.float32)
    b = np.array([[3.0, 3.0, 3.0], [4.0, 2.0, 1.0]], np.float32)
    assert oracle.maxsim_f32(oracle.EUCLID, a, a) == np.float32(-0.0)
    assert oracle.maxsim_f32(oracle.EUCLID, a, b) == np.float32(-19.0)
    # the fold over a precomputed similarity matrix agrees with the direct form
    rows = np.concatenate([a, b])
    sims = np.stack([oracle.score_rows_f32(oracle.EUCLID, rows, q) for q in a])
    np.testing.assert_array_equal(oracle.maxsim_fold(sims, [0, 3, 5]), np.array([-0.0, -19.0], np.float32))
