"""Generates tests/golden/simd_utils_r01.npz: outputs of the REFERENCE'S OWN C kernels (lib/quantization/cpp/{avx2,sse}.c,
compiled verbatim into oracle/_ref/libsimd_utils.so by oracle/Makefile) on seeded inputs.

/root/reference does not exist on the GPU box, so the vectors are committed; this script is how they were made:

    python tests/golden/make_golden.py        # needs /root/reference (or a prebuilt oracle/_ref/libsimd_utils.so)

Contents
    sq8_dim[c], sq8_q[c, 4096], sq8_v[c, 4096]   random / extreme 7-bit codes (only the first sq8_dim[c] bytes are used)
    sq8_dot_avx[c], sq8_l1_avx[c], sq8_dot_sse[c], sq8_l1_sse[c]   impl_score_{dot,l1}_{avx,sse}(q, v, dim)
    e2e_*                                            a 256 x 768 SQ8 cosine segment, 3 f32 queries, and the scores
                                                     postprocess_score(impl_score_dot_avx(query code, row code)) of every (query, row)
    bq_*                                             one-bit rows, scalar-8/4-bit and binary queries, impl_xor_popcnt_* outputs

and tests/golden/ref_kernels_kat.npz: the same kernels' results on the seeded inputs the tests regenerate themselves
    sq8_{dot_avx,l1_avx,dot_sse}[c]     impl_score_* on case c of tests.test_oracle_kat.sq8_kat_codes()
    bq_xor_{s8,s4,bin}[c, row]          impl_xor_popcnt_{scalar8_avx,scalar4_avx,sse}_uint128 on tests.test_oracle_kat.bq_kat_vectors()
    sq8_e2e_scores[query, row]          postprocess_score(impl_score_dot_avx) on test_gpu_quant.test_sq8_matches_reference_c_kernel's segment
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def main():
    from oracle import oracle as o

    R = o.ref()
    assert R is not None, "oracle/_ref/libsimd_utils.so is needed to generate the golden vectors"
    u8p = C.POINTER(C.c_uint8)
    rng = np.random.default_rng(20260922)
    dims, qs, vs = [], [], []
    for dim in (16, 32, 48, 64, 80, 768, 784, 1536, 2000, 4096):
        for trial in range(8):
            q = rng.integers(0, 128, 4096, dtype=np.uint8)
            v = rng.integers(0, 128, 4096, dtype=np.uint8)
            if trial == 0:
                q[:] = 127; v[:] = 127
            if trial == 1:
                q[:] = 0
            if trial == 2:
                v[:] = 0; q[:] = 127
            dims.append(dim); qs.append(q); vs.append(v)
    dims = np.array(dims, np.uint32); qs = np.stack(qs); vs = np.stack(vs)
    out = {"sq8_dim": dims, "sq8_q": qs, "sq8_v": vs}
    for name in ("dot_avx", "l1_avx", "dot_sse", "l1_sse"):
        fn = getattr(R, "impl_score_" + name)
        out["sq8_" + name] = np.array([fn(qs[c].ctypes.data_as(u8p), vs[c].ctypes.data_as(u8p), int(dims[c])) for c in range(len(dims))], np.float32)

    # end to end: EncodedVectorsU8 rows (oracle encode; metadata fixed) scored with the reference's kernel + postprocess_score
    base = o.preprocess_rows_f32(o.COSINE, rng.standard_normal((256, 768)).astype(np.float32))
    queries = rng.standard_normal((3, 768)).astype(np.float32)
    sq = o.SQ8.encode(base, o.QD_DOT, False)
    scores = np.zeros((3, 256), np.float32)
    codes, offs = [], []
    for qi, q in enumerate(queries):
        code, off = sq.encode_query(o.preprocess_f32(o.COSINE, q))
        codes.append(code); offs.append(off)
        for i in range(256):
            row = np.ascontiguousarray(sq.rows[i])
            raw = np.float32(R.impl_score_dot_avx(code.ctypes.data_as(u8p), row[4:].ctypes.data_as(u8p), 768))
            voff = row[:4].view(np.float32)[0]
            scores[qi, i] = np.float32(np.float32(np.float32(sq.meta.multiplier) * raw) + off) + voff   # encoded_vectors_u8.rs:101-103
    out.update(e2e_rows=np.asarray(sq.rows), e2e_meta=np.array([sq.meta.alpha, sq.meta.offset, sq.meta.multiplier], np.float32), e2e_queries=queries,
               e2e_query_codes=np.stack(codes), e2e_query_offs=np.array(offs, np.float32), e2e_scores=scores)

    # BQ: one-bit rows vs scalar-8 / scalar-4 / binary queries
    bq_dim = 1000
    data = rng.standard_normal((16, bq_dim)).astype(np.float32)
    q = rng.standard_normal(bq_dim).astype(np.float32)
    out["bq_dim"] = np.array([bq_dim], np.uint32)
    for tag, qenc, fn in (("s8", o.BQQ_SCALAR8, R.impl_xor_popcnt_scalar8_avx_uint128), ("s4", o.BQQ_SCALAR4, R.impl_xor_popcnt_scalar4_avx_uint128),
                          ("bin", o.BQQ_SAME, R.impl_xor_popcnt_sse_uint128)):
        bq = o.BQ.encode(data, o.BQ_ONE, qenc, o.QD_DOT, False)
        qe = bq.encode_query(q)
        words = bq.rows.shape[1] // 16
        out["bq_rows"] = np.asarray(bq.rows)
        out["bq_query_" + tag] = np.asarray(qe)
        out["bq_xor_" + tag] = np.array([fn(qe.ctypes.data_as(u8p), np.ascontiguousarray(bq.rows[i]).ctypes.data_as(u8p), words) for i in range(16)], np.uint32)
    out["bq_data"] = data
    out["bq_query_f32"] = q
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "simd_utils_r01.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


def ref_kernels_kat():
    from oracle import oracle as o
    from qdrant_b200 import scorer as qb
    from tests.test_gpu_quant import gen
    from tests.test_oracle_kat import REF_KAT, bq_kat_vectors, sq8_kat_codes

    R = o.ref()
    assert R is not None, "oracle/_ref/libsimd_utils.so is needed to generate the golden vectors"
    u8p = C.POINTER(C.c_uint8)
    out = {"sq8_" + name: [] for name in ("dot_avx", "l1_avx", "dot_sse")}
    for dim, q, v in sq8_kat_codes():
        for name in ("dot_avx", "l1_avx", "dot_sse"):
            out["sq8_" + name].append(getattr(R, "impl_score_" + name)(q.ctypes.data_as(u8p), v.ctypes.data_as(u8p), dim))
    out = {k: np.array(x, np.float32) for k, x in out.items()}

    xor = {"s8": [], "s4": [], "bin": []}
    for dim, data, q in bq_kat_vectors():
        for tag, qenc, fn in (("s8", o.BQQ_SCALAR8, R.impl_xor_popcnt_scalar8_avx_uint128), ("s4", o.BQQ_SCALAR4, R.impl_xor_popcnt_scalar4_avx_uint128),
                              ("bin", o.BQQ_SAME, R.impl_xor_popcnt_sse_uint128)):
            bq = o.BQ.encode(data, o.BQ_ONE, qenc, o.QD_DOT, False)
            qe = bq.encode_query(q)
            words = bq.rows.shape[1] // 16
            xor[tag].append([fn(qe.ctypes.data_as(u8p), np.ascontiguousarray(bq.rows[i]).ctypes.data_as(u8p), words) for i in range(data.shape[0])])
    out.update({"bq_xor_" + tag: np.array(x, np.uint32) for tag, x in xor.items()})

    base, queries = gen(o, qb, qb.Distance.Cosine, 256, 768)
    sq = o.SQ8.encode(base, o.QD_DOT, False)
    scores = np.zeros((queries.shape[0], 256), np.float32)
    for qi, q in enumerate(queries):
        code, off = sq.encode_query(o.preprocess_f32(o.COSINE, q))
        for i in range(256):
            row = np.ascontiguousarray(sq.rows[i])
            raw = np.float32(R.impl_score_dot_avx(code.ctypes.data_as(u8p), row[4:].ctypes.data_as(u8p), 768))
            voff = row[:4].view(np.float32)[0]
            scores[qi, i] = np.float32(np.float32(np.float32(sq.meta.multiplier) * raw) + off) + voff   # encoded_vectors_u8.rs:101-103
    out["sq8_e2e_scores"] = scores
    np.savez_compressed(REF_KAT, **out)
    print(REF_KAT, os.path.getsize(REF_KAT), "bytes")


if __name__ == "__main__":
    main()
    ref_kernels_kat()
