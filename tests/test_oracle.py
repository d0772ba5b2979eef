"""not-gpu: pins the CPU oracle (oracle/) against the answers of the UNMODIFIED reference.

  * tests/golden/synthetic.npz was produced by the reference + the oracle stand-in (oracle/make_golden.py);
    the oracle's own restatement of fit() (oracle/pipeline.py) must reproduce it exactly;
  * tests/golden/standin_calls.npz holds every distinct call the reference's own unittest suite made into the
    stand-in, with the stand-in's answers, recorded while that suite passed (oracle/record_standin_calls.py): every
    hot-path test passed (the add_match tests fail on pandas 3's removed Series._append, off the hot path —
    SURVEY.md §0 fact 4).  Replaying the calls must give the same answers bit for bit.
"""
import json
import os

import numpy as np
from scipy.sparse import csc_matrix, csr_matrix

from oracle import pipeline as P
from oracle.sdt import sp_matmul_topn, zip_sp_matmul_topn
from synth_corpus import make_names

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "synthetic.npz"), allow_pickle=True)


def test_pipeline_restatement_reproduces_reference_self_match():
    names = make_names(3000, seed=11)
    ml, true_max = P.fit(names, min_similarity=0.8)
    assert np.array_equal(ml.master_side.to_numpy(), GOLD["self3000_master_side"])
    assert np.array_equal(ml.dupe_side.to_numpy(), GOLD["self3000_dupe_side"])
    np.testing.assert_array_equal(ml.similarity.to_numpy(), GOLD["self3000_similarity"])
    assert true_max == int(GOLD["self3000_true_max"][0])
    ml2, _ = P.fit(names, min_similarity=0.8, fast_symmetrize=True)
    assert np.array_equal(ml2.dupe_side.to_numpy(), GOLD["self3000_dupe_side"])
    np.testing.assert_allclose(ml2.similarity.to_numpy(), GOLD["self3000_similarity"], atol=1e-15)


def test_pipeline_restatement_reproduces_reference_two_series():
    master = make_names(2000, seed=12)
    dupes = make_names(1200, seed=12)[:600] + make_names(200, seed=13)
    ml, _ = P.fit(master, dupes, min_similarity=0.7, max_n_matches=5)
    assert np.array_equal(ml.master_side.to_numpy(), GOLD["two2000_master_side"])
    assert np.array_equal(ml.dupe_side.to_numpy(), GOLD["two2000_dupe_side"])
    np.testing.assert_array_equal(ml.similarity.to_numpy(), GOLD["two2000_similarity"])


def test_tfidf_restatement_reproduces_reference_matrix():
    texts = make_names(500, seed=14) + ["", "ab", "abc", "A.B,C-D/E F\tG", "ÀbracâDABRÀ", "ﬁ½① İstanbul",
                                        "x" * 300 + " inc", "aaa aaa aaa aaaa"]
    m, _, vec = P.tf_idf_matrices(texts)
    assert np.array_equal(m.indptr, GOLD["tfidf_indptr"]) and np.array_equal(m.indices, GOLD["tfidf_indices"])
    np.testing.assert_array_equal(m.data, GOLD["tfidf_data"])
    assert sorted(vec.vocabulary_, key=vec.vocabulary_.get) == GOLD["tfidf_vocab"].tolist()


def test_analyzer_known_answers():
    # reference tests test_n_grams_* (test_string_grouper.py:495-517) and docs/references/sg_class.md:54-57
    assert P.n_grams('McDonalds') == ['mcd', 'cdo', 'don', 'ona', 'nal', 'ald', 'lds']
    assert P.n_grams('McDonalds', ignore_case=False) == ['McD', 'cDo', 'Don', 'ona', 'nal', 'ald', 'lds']
    assert P.n_grams('ÀbracâDABRÀ') == ['abr', 'bra', 'rac', 'aca', 'cad', 'ada', 'dab', 'abr', 'bra']
    assert P.n_grams('ab') == []


def test_topn_semantics_strict_threshold_and_zip():
    A = csr_matrix(np.array([[1.0, 0.0], [0.6, 0.8], [0.0, 1.0]]))
    C = sp_matmul_topn(A, A.T.tocsr(), top_n=2, threshold=0.6, sort=True)
    # row 0: {0:1.0} (0.6 is NOT > 0.6); row 1: {1:1.0, 2:0.8}; row 2: {2:1.0, 1:0.8}
    assert C[0].indices.tolist() == [0] and C[1].indices.tolist() == [1, 2] and C[2].indices.tolist() == [2, 1]
    blocks = [sp_matmul_topn(A, A[r].T.tocsr(), top_n=2, threshold=0.1, sort=True) for r in ([0], [1, 2])]
    Z = zip_sp_matmul_topn(2, blocks)
    full = sp_matmul_topn(A, A.T.tocsr(), top_n=2, threshold=0.1, sort=True)
    assert (Z != full).nnz == 0 and Z.shape == (3, 3)


def test_block_invariance_of_the_oracle():
    names = make_names(1500, seed=21)
    m, d, _ = P.tf_idf_matrices(names)
    base = P.build_matches(m, d, (1, 1), 20, 0.6)
    for nb in [(1, 4), (2, 3), (3, 7)]:
        other = P.build_matches(m, d, nb, 20, 0.6)
        assert abs(base - other).max() < 1e-12 or (base != other).nnz <= 4   # top-n ties may swap


def test_reference_own_suite_passes_with_the_oracle_standin():
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "standin_calls.npz"), allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    values, ints = z["values"], z["ints"]
    suite = meta["suite"]
    # only the pandas-3 `Series._append` removals failed (add_match, off the hot path)
    assert all("add_match" in t or "prior_matches" in t for t in suite["failed"]), suite
    assert suite["passed"] >= 49, suite

    def load(rec):
        v0, nv = rec["values"]
        i0, ni = rec["indices"]
        p0, npp = rec["indptr"]
        parts = (values[v0:v0 + nv].astype(rec["dtype"]), ints[i0:i0 + ni].astype(rec["index_dtype"]),
                 ints[p0:p0 + npp].astype(rec["index_dtype"]))
        return (csr_matrix if rec["format"] == "csr" else csc_matrix)(parts, shape=tuple(rec["shape"]))

    assert len(meta["calls"]) > 100 and {c["fn"] for c in meta["calls"]} == {"sp_matmul_topn", "zip_sp_matmul_topn"}
    for i, c in enumerate(meta["calls"]):
        if c["fn"] == "sp_matmul_topn":
            got = sp_matmul_topn(load(c["A"]), load(c["B"]), *c["args"], **c["kwargs"])
        else:
            got = zip_sp_matmul_topn(top_n=c["top_n"], C_mats=[load(m) for m in c["C_mats"]])
        want = load(c["out"])
        label = "call %d (%s)" % (i, c["fn"])
        assert got.format == "csr" and got.shape == want.shape and got.dtype == want.dtype, label
        assert got.indices.dtype == want.indices.dtype, label
        assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices), label
        assert np.array_equal(got.data, want.data), label
