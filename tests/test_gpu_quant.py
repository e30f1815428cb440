"""GPU parity: SQ8 / PQ / BQ scorers through the C ABI vs the CPU oracle — bit-exact (assert_array_equal).

Test shapes follow lib/quantization/tests/integration (129 vectors x dim 65, seed 42: dim not a multiple of 16
exercises padding; test_simple.rs / test_avx2.rs / test_pq.rs / test_binary.rs) plus the BASELINE.json dims.
Quantizer *training* is RNG-dependent in the reference (SURVEY §8c), so both sides are fed the SAME metadata
and codes (produced by the oracle's restatement of encode) and only scoring / query encoding is compared.
"""
import numpy as np
import pytest

from tests.util import assert_topk_equal, pack_bitmap

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def qb():
    from qdrant_b200 import scorer

    return scorer


def qparams(qb, dist):
    dt, inv = qb.construct_vector_parameters(dist)
    return int(dt), bool(inv)


def gen(oracle, qb, dist, n, dim, seed=42, nq=3):
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((n, dim)).astype(np.float32)
    if dist == qb.Distance.Cosine:
        base = oracle.preprocess_rows_f32(oracle.COSINE, base)
    queries = rng.standard_normal((nq, dim)).astype(np.float32)
    return base, queries


# ------------------------------------------------------------------------------------------------ SQ8
@pytest.mark.parametrize("dist", ["Cosine", "Dot", "Euclid", "Manhattan"])
@pytest.mark.parametrize("n,dim", [(129, 65), (500, 16), (400, 768), (300, 1536), (200, 2000)])
def test_sq8_scores_bit_exact(qb, oracle, dist, n, dim):
    d = getattr(qb.Distance, dist)
    dt, inv = qparams(qb, d)
    base, queries = gen(oracle, qb, d, n, dim)
    sq = oracle.SQ8.encode(base, dt, inv)
    st = qb.ScalarQuantizedVectors(sq.rows, dim, sq.meta.alpha, sq.meta.offset, sq.meta.multiplier, d)
    ids = np.arange(n, dtype=np.uint32)
    for q in queries:
        qp = oracle.preprocess_f32(int(d), q)
        code, off = sq.encode_query(qp)
        want = np.array([sq.score(code, off, i) for i in range(n)], np.float32)
        sc = st.raw_scorer(q)
        np.testing.assert_array_equal(sc.score_points(ids), want)
        assert sc.score_point(7) == want[7]
        sc.close()
    # internal scorer: stored point as query (encode_internal_vector, encoded_vectors_u8.rs:715-728)
    isc = st.raw_internal_scorer(5)
    want = np.array([sq.score_internal(5, j) for j in range(n)], np.float32)
    np.testing.assert_array_equal(isc.score_points(ids), want)
    assert isc.score_internal(11, 3) == sq.score_internal(11, 3)
    isc.close()
    st.close()


def test_sq8_matches_reference_c_kernel(qb, oracle):
    """End-to-end against the reference's OWN impl_score_dot_avx + postprocess_score: its scores of these queries and rows,
    multiplier * raw + query offset + row offset, are stored in tests/golden/ref_kernels_kat.npz."""
    from tests.test_oracle_kat import REF_KAT

    want = np.load(REF_KAT)["sq8_e2e_scores"]
    d = qb.Distance.Cosine
    base, queries = gen(oracle, qb, d, 256, 768)
    sq = oracle.SQ8.encode(base, oracle.QD_DOT, False)
    st = qb.ScalarQuantizedVectors(sq.rows, 768, sq.meta.alpha, sq.meta.offset, sq.meta.multiplier, d)
    assert want.shape == (queries.shape[0], 256)
    for qi, q in enumerate(queries):
        got = st.raw_scorer(q).score_points(np.arange(256, dtype=np.uint32))
        for i in range(256):
            assert got[i] == want[qi, i], (qi, i)
    st.close()


@pytest.mark.parametrize("dist", ["Cosine", "Euclid", "Manhattan"])
def test_sq8_search_batch(qb, oracle, dist):
    d = getattr(qb.Distance, dist)
    dt, inv = qparams(qb, d)
    base, queries = gen(oracle, qb, d, 80_000, 64, nq=5)
    sq = oracle.SQ8.encode(base, dt, inv)
    st = qb.ScalarQuantizedVectors(sq.rows, 64, sq.meta.alpha, sq.meta.offset, sq.meta.multiplier, d)
    enc = [sq.encode_query(oracle.preprocess_f32(int(d), q)) for q in queries]
    codes = np.stack([e[0] for e in enc]); offs = np.array([e[1] for e in enc], np.float32)
    deleted = np.random.default_rng(2).random(base.shape[0]) < 0.1
    for top, dl in ((10, None), (100, deleted)):
        got = st.search_batch(queries, top, point_deleted=dl)
        want = sq.scan(codes, offs, top, deleted=None if dl is None else pack_bitmap(dl))
        for i in range(len(queries)):
            assert_topk_equal(got[i], want[i], None, f"sq8 {dist} top={top} q={i}")
    st.close()


# ------------------------------------------------------------------------------------------------ PQ
@pytest.mark.parametrize("dist", ["Cosine", "Dot", "Euclid", "Manhattan"])
@pytest.mark.parametrize("n,dim,chunk", [(129, 65, 2), (300, 128, 8), (200, 1536, 16), (150, 70, 16)])
def test_pq_scores_bit_exact(qb, oracle, dist, n, dim, chunk):
    d = getattr(qb.Distance, dist)
    dt, inv = qparams(qb, d)
    base, queries = gen(oracle, qb, d, n, dim)
    cents = oracle.kmeans_pq_centroids(base, chunk, n_centroids=256 if n >= 256 else 64, iters=3)
    pq = oracle.PQ.encode(base, chunk, cents, dt, inv)
    st = qb.ProductQuantizedVectors(pq.codes, cents, chunk, dim, d)
    ids = np.arange(n, dtype=np.uint32)
    for q in queries:
        lut = pq.encode_query(oracle.preprocess_f32(int(d), q))
        want = np.array([pq.score(lut, i) for i in range(n)], np.float32)
        sc = st.raw_scorer(q)
        np.testing.assert_array_equal(sc.score_points(ids), want)
        # score_internal decodes both codes through the centroids (encoded_vectors_pq.rs:574-618)
        assert sc.score_internal(2, 9) == pq.score_internal(2, 9)
        sc.close()
    from qdrant_b200._capi import QbError, QB_ERR_UNSUPPORTED

    with pytest.raises(QbError) as ei:  # encode_internal_vector = None (encoded_vectors_pq.rs:624-627)
        st.raw_internal_scorer(0)
    assert ei.value.status == QB_ERR_UNSUPPORTED
    st.close()


def test_pq_search_batch(qb, oracle):
    d = qb.Distance.Dot
    base, queries = gen(oracle, qb, d, 70_000, 96, nq=4)
    cents = oracle.kmeans_pq_centroids(base, 8, iters=2)
    pq = oracle.PQ.encode(base, 8, cents, oracle.QD_DOT, False)
    st = qb.ProductQuantizedVectors(pq.codes, cents, 8, 96, d)
    luts = np.stack([pq.encode_query(q) for q in queries])
    got = st.search_batch(queries, 10)
    want = pq.scan(luts, 10)
    for i in range(len(queries)):
        assert_topk_equal(got[i], want[i], None, f"pq q={i}")
    st.close()


@pytest.mark.parametrize("dist,n,dim,chunk,nq", [("Dot", 70_000, 128, 4, 5), ("Euclid", 66_000, 128, 2, 8), ("Cosine", 70_001, 1536, 16, 7), ("Manhattan", 131_000, 64, 2, 3),
                                                 ("Euclid", 140_000, 256, 2, 20), ("Cosine", 70_001, 1536, 16, 33)])
def test_pq_batched_four_query_cluster_kernel(qb, oracle, dist, n, dim, chunk, nq):
    """pq_scan4_kernel (m % 32 == 0: CTA pair, float4-interleaved LUT halves, partial sums handed over through distributed shared
    memory) == oracle score_point_sse order, bit-exact, for every queries-per-pass variant, with deletions and several row blocks."""
    d = getattr(qb.Distance, dist)
    dt, inv = qparams(qb, d)
    rng = np.random.default_rng(dim + nq)
    base = rng.standard_normal((n, dim)).astype(np.float32)
    if d == qb.Distance.Cosine:
        base = oracle.preprocess_rows_f32(oracle.COSINE, base)
    queries = rng.standard_normal((nq, dim)).astype(np.float32)
    cents = (rng.standard_normal((256, dim)) * 0.3).astype(np.float32)
    codes = rng.integers(0, 256, (n, dim // chunk), dtype=np.uint8)          # scoring parity does not depend on how codes were chosen
    pq = oracle.PQ(dim, chunk, cents, codes, dt, inv)
    st = qb.ProductQuantizedVectors(codes, cents, chunk, dim, d)
    luts = np.stack([pq.encode_query(oracle.preprocess_f32(int(d), q)) for q in queries])
    deleted = rng.random(n) < 0.02
    want = pq.scan(luts, 10, deleted=pack_bitmap(deleted))
    for qpp in (0, 16, 8, 4, 2, 1):
        qb.set_option("pq_queries_per_pass", qpp)
        try:
            got = st.search_batch(queries, 10, point_deleted=deleted)
        finally:
            qb.set_option("pq_queries_per_pass", 0)
        for i in range(nq):
            assert_topk_equal(got[i], want[i], None, f"pq4 {dist} qpp={qpp} q={i}")
    assert st.search_stats()[1] == 0
    st.close()


@pytest.mark.parametrize("qpp", [16, 8])
@pytest.mark.parametrize("case", ["plain", "ties", "wide_range", "nan_centroid", "cancelling", "flat_tables"])
def test_pq_prefilter_kernels_are_exact(qb, oracle, case, qpp):
    """pq_scan8_kernel scores eight queries per gather through bf16 tables and keeps every row within (2^-9 + 2^-15) * sum_j max|lut_j| of
    the threshold; pq_scan16_kernel sixteen per gather through u8 tables with an integer threshold (quantisation step * m / 2 + roundings);
    pq_rescore_kernel re-scores the survivors in score_point_sse's order.  The result must be the single-query kernel's,
    bit for bit: partial last group (19 queries), boundary ties, tables whose entries span 12 orders of magnitude, sums that cancel
    (margin >> score spread: nearly everything survives -> overflow -> exact rerun), and a NaN centroid (no finite margin)."""
    rng = np.random.default_rng(sum(map(ord, case)))
    n, dim, chunk, nq, top = 150_000, 128, 4, 19, 10
    d = qb.Distance.Dot
    queries = rng.standard_normal((nq, dim)).astype(np.float32)
    cents = (rng.standard_normal((256, dim)) * 0.3).astype(np.float32)
    codes = rng.integers(0, 256, (n, dim // chunk), dtype=np.uint8)
    if case == "ties":
        codes = codes[rng.integers(0, 40, n)]                 # 40 distinct rows: every score value occurs thousands of times
    elif case == "wide_range":
        cents *= (10.0 ** rng.uniform(-6, 6, (1, dim))).astype(np.float32)
    elif case == "nan_centroid":
        cents[7, 5] = np.nan
    elif case == "flat_tables":
        cents[:] = cents[0]                                     # every centroid the same: all rows score alike, quantisation step 0
    elif case == "cancelling":
        cents[:, :64] *= 1.0e4                                  # huge table entries ...
        queries[:, 32:64] = -queries[:, :32]                    # ... that cancel pairwise in most rows' sums
        cents[:, 32:64] = cents[:, :32]
        codes[:, 8:16] = codes[:, :8]
    pq = oracle.PQ(dim, chunk, cents, codes, oracle.QD_DOT, False)
    st = qb.ProductQuantizedVectors(codes, cents, chunk, dim, d)
    qb.set_option("pq_queries_per_pass", 1)
    try:
        want = st.search_batch(queries, top)
    finally:
        qb.set_option("pq_queries_per_pass", 0)
    st.search_stats(reset=True)
    qb.set_option("pq_queries_per_pass", qpp)
    try:
        got = st.search_batch(queries, top)
    finally:
        qb.set_option("pq_queries_per_pass", 0)
    searches, reruns = st.search_stats(reset=True)
    if case in ("plain", "wide_range"):
        assert reruns == 0, "the prefilter's margin admitted too many rows on an ordinary table"
    if case != "nan_centroid":                                  # the oracle's heap order among NaN scores is not the id order
        luts = np.stack([pq.encode_query(q) for q in queries])
        ref = pq.scan(luts, top)
        for i in range(nq):
            assert_topk_equal(got[i], ref[i], None, f"pq{qpp} {case} vs oracle q={i}")
    for i in range(nq):
        np.testing.assert_array_equal(got[i]["idx"], want[i]["idx"], err_msg=f"pq{qpp} {case} q={i}")
        np.testing.assert_array_equal(got[i]["score"].view(np.uint32), want[i]["score"].view(np.uint32), err_msg=f"pq{qpp} {case} q={i}")
    st.close()


# ------------------------------------------------------------------------------------------------ BQ
@pytest.mark.parametrize("dist", ["Cosine", "Dot", "Euclid", "Manhattan"])
@pytest.mark.parametrize("enc", ["OneBit", "TwoBits", "OneAndHalfBits"])
@pytest.mark.parametrize("qenc", ["SameAsStorage", "Scalar4bits", "Scalar8bits"])
@pytest.mark.parametrize("n,dim", [(129, 65), (200, 768), (100, 1000)])
def test_bq_scores_bit_exact(qb, oracle, dist, enc, qenc, n, dim):
    d = getattr(qb.Distance, dist)
    dt, inv = qparams(qb, d)
    base, queries = gen(oracle, qb, d, n, dim)
    e, qe = int(getattr(qb.BQEncoding, enc)), int(getattr(qb.BQQueryEncoding, qenc))
    ms = oracle.bq_mean_std(base) if e != oracle.BQ_ONE else None
    bq = oracle.BQ.encode(base, e, qe, dt, inv, ms)
    st = qb.BinaryQuantizedVectors(bq.rows, dim, d, qb.BQEncoding(e), qb.BQQueryEncoding(qe), ms)
    ids = np.arange(n, dtype=np.uint32)
    for q in queries:
        qenc_bytes = bq.encode_query(oracle.preprocess_f32(int(d), q))
        want = np.array([bq.score(qenc_bytes, i) for i in range(n)], np.float32)
        sc = st.raw_scorer(q)
        np.testing.assert_array_equal(sc.score_points(ids), want)
        sc.close()
    # internal scoring always compares two stored binary vectors (calculate_metric(.., 1), :892-917)
    isc = st.raw_internal_scorer(4)
    binq = oracle.BQ(dim, e, oracle.BQQ_SAME, bq.rows, dt, inv, ms)
    want = np.array([binq.score(bq.rows[4], j) for j in range(n)], np.float32)
    np.testing.assert_array_equal(isc.score_points(ids), want)
    isc.close()
    st.close()


def test_bq_search_batch_and_rescore(qb, oracle):
    """BQ defaults to rescoring with the original vectors (accessors.rs:16-38): oversample -> rescore -> truncate."""
    d = qb.Distance.Dot
    base, queries = gen(oracle, qb, d, 90_000, 128, nq=3)
    bq = oracle.BQ.encode(base, oracle.BQ_ONE, oracle.BQQ_SAME, oracle.QD_DOT, False)
    st = qb.BinaryQuantizedVectors(bq.rows, 128, d)
    orig = qb.DenseVectorStorage(base, d)
    qencs = np.stack([bq.encode_query(q) for q in queries])
    top = qb.get_oversampled_top(10, True, 3.0)
    assert top == 30
    got = st.search_batch(queries, top)
    want = bq.scan(qencs, top)
    for i in range(len(queries)):
        # integer scores tie massively: compare score lists exactly, ids only through their scores
        all_sc = np.array([bq.score(qencs[i], int(j)) for j in got[i]["idx"]], np.float32)
        np.testing.assert_array_equal(got[i]["score"], want[i]["score"])
        np.testing.assert_array_equal(all_sc, got[i]["score"])
        res = qb.postprocess_search_result(got[i], orig, queries[i], 10, rescore=True)
        exact = oracle.score_points_f32(oracle.DOT, base, queries[i], got[i]["idx"])
        order = np.argsort(-exact, kind="stable")[:10]
        np.testing.assert_array_equal(res["score"], exact[order])
    st.close(); orig.close()


# ------------------------------------------------------------------------------------------------ SQ8 tensor-core batch path
@pytest.mark.parametrize("dist,n,dim,nq", [("Cosine", 100_000, 768, 300), ("Euclid", 70_000, 128, 64), ("Dot", 80_000, 65, 33),
                                           ("Cosine", 70_000, 1536, 40), ("Cosine", 66_000, 768, 256)])
def test_sq8_batched_tensor_core_path(qb, oracle, dist, n, dim, nq):
    """Batched SQ8 search (tcgen05 kind::i8 GEMM + fused epilogue/filter) == oracle peek_top_iter, bit-exact, and
    == the CUDA-core path (option disable_mma)."""
    d = getattr(qb.Distance, dist)
    dt, inv = qparams(qb, d)
    base, queries = gen(oracle, qb, d, n, dim, nq=nq)
    sq = oracle.SQ8.encode(base, dt, inv)
    st = qb.ScalarQuantizedVectors(sq.rows, dim, sq.meta.alpha, sq.meta.offset, sq.meta.multiplier, d)
    enc = [sq.encode_query(oracle.preprocess_f32(int(d), q)) for q in queries]
    codes = np.stack([e[0] for e in enc]); offs = np.array([e[1] for e in enc], np.float32)
    deleted = np.random.default_rng(4).random(n) < 0.05
    qb.set_option("disable_mma", 0)
    st.search_stats(reset=True)
    got = st.search_batch(queries, 10, point_deleted=deleted)
    searches, reruns = st.search_stats(reset=True)
    # the tensor-core fast path itself produced the answer: no "assumption broken" rerun on the exact CUDA-core / full-materialisation paths
    # (only dim > 1040 can leave the f32-exact window: flag 2 -> lane-exact kernel)
    assert searches == 1 and (reruns == 0 or dim > 1040), (searches, reruns)
    qb.set_option("disable_mma", 1)
    try:
        got_cc = st.search_batch(queries, 10, point_deleted=deleted)
    finally:
        qb.set_option("disable_mma", 0)
    want = sq.scan(codes, offs, 10, deleted=pack_bitmap(deleted))
    for i in range(nq):
        np.testing.assert_array_equal(got[i], got_cc[i])
        assert_topk_equal(got[i], want[i], None, f"sq8-mma {dist} q={i}")
    st.close()


def test_sq8_batched_fallbacks_on_mass_ties(qb, oracle):
    """Every row identical: the per-(query, CTA) segments overflow, then the global candidate buffer overflows, and the
    search must still end on the exact full-materialisation path with the right answer."""
    d = qb.Distance.Dot
    rng = np.random.default_rng(12)
    base = np.tile(rng.standard_normal((1, 64)).astype(np.float32), (70_000, 1))
    queries = rng.standard_normal((40, 64)).astype(np.float32)
    sq = oracle.SQ8.encode(base, oracle.QD_DOT, False)
    st = qb.ScalarQuantizedVectors(sq.rows, 64, sq.meta.alpha, sq.meta.offset, sq.meta.multiplier, d)
    got = st.search_batch(queries, 10)
    for i, q in enumerate(queries):
        code, off = sq.encode_query(q)
        s0 = sq.score(code, off, 0)
        assert got[i].size == 10 and np.all(got[i]["score"] == s0)
        assert sorted(got[i]["idx"].tolist()) == list(range(10))
    st.close()
