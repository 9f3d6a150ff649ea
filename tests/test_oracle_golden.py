"""Pins the CPU oracle against fixtures produced by the reference's own unmodified code
(oracle/gen_golden.py).  CPU-only."""
import os

import numpy as np
import pytest

from oracle import oracle, ref_import, synth


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def test_cosine_kat_bit_exact(golden_dir):
    g = _load(golden_dir, "cosine_kat.npz")
    for i in range(len(g["out"])):
        a, b = g["a"][i, :g["len_a"][i]], g["b"][i, :g["len_b"][i]]
        for col, variant in enumerate(("injector", "retriever", "utils")):
            got = oracle.cosine(a, b, variant)
            assert got == g["out"][i, col], (i, variant, got, g["out"][i, col])


def test_sum_mode_naive_differs_only_in_rounding():
    rng = np.random.default_rng(0)
    a, b = rng.uniform(-1, 1, 384), rng.uniform(-1, 1, 384)
    n, c = oracle.cosine(a, b, "injector", oracle.SUM_NAIVE), oracle.cosine(a, b, "injector", oracle.SUM_NEUMAIER)
    assert abs(n - c) < 1e-14
    # naive mode is the plain left-to-right binary64 recurrence (CPython < 3.12)
    dot = 0.0
    for x, y in zip(a, b):
        dot = dot + x * y
    n1 = 0.0
    for x in a:
        n1 = n1 + x * x
    n2 = 0.0
    for y in b:
        n2 = n2 + y * y
    assert n == dot / (np.sqrt(n1) * np.sqrt(n2))


@pytest.mark.parametrize("k", [3, 10, 200])
def test_batch_small_matches_reference(golden_dir, k):
    g = _load(golden_dir, "batch_small.npz")
    got = oracle.batch_similarities(g["Q"], g["X"], k, query_ok=g["query_ok"], row_ok=g["row_ok"])
    for qi, lst in enumerate(got):
        cnt = int(g[f"count_k{k}"][qi])
        assert len(lst) == cnt
        assert [r for r, _ in lst] == list(g[f"idx_k{k}"][qi, :cnt])
        assert [s for _, s in lst] == list(g[f"score_k{k}"][qi, :cnt])  # bit-exact binary64


def test_batch_small_edge_semantics(golden_dir):
    g = _load(golden_dir, "batch_small.npz")
    got = oracle.batch_similarities(g["Q"], g["X"], 10, query_ok=g["query_ok"], row_ok=g["row_ok"])
    assert got[3] == []                                   # Exception-valued query
    assert [r for r, _ in got[1]][:3] == [5, 17, 99]       # exact duplicates: lowest row first
    assert all(s == 0.0 for _, s in got[4])                # zero query
    assert [r for r, _ in got[4]] == [0, 1, 2, 3, 4, 5, 6, 7, 9, 10]  # store order, falsy row 8 skipped


def test_batch_c1_matches_reference(golden_dir):
    g = _load(golden_dir, "batch_c1.npz")
    n, d, q, k = int(g["n"]), int(g["d"]), int(g["q"]), int(g["k"])
    X = synth.synth_rows(int(g["store_seed"]), 0, n, d)
    Q = synth.synth_queries(int(g["query_seed"]), q, d, int(g["store_seed"]), n)
    got = oracle.batch_similarities(Q, X, k)
    assert np.array_equal(np.array([[r for r, _ in l] for l in got]), g["idx"])
    assert np.array_equal(np.array([[s for _, s in l] for l in got]), g["score"])
    # the blocked large-N tier must agree with the straight restatement
    bi, bs, bc = oracle.topk_blocked(Q, X, k, block=1024)
    assert np.array_equal(bi, g["idx"]) and np.array_equal(bs, g["score"]) and (bc == k).all()


@pytest.mark.parametrize("k,k2", [(3, 2), (10, 4), (10, 25)])
def test_merge_matches_reference(golden_dir, k, k2):
    g = _load(golden_dir, "merge.npz")
    per_query = oracle.batch_similarities(g["Q"], g["X"], k)
    got = oracle.merge_max_by_id(per_query, k2)
    assert [r for r, _ in got] == list(g[f"idx_{k}_{k2}"])
    assert [s for _, s in got] == list(g[f"score_{k}_{k2}"])


def test_prune_matches_reference(golden_dir):
    g = _load(golden_dir, "prune.npz")
    for name in "abcd":
        E = g[f"E_{name}"]
        rep, _ = oracle.representative(E)
        assert rep == int(g[f"rep_{name}"])
        for thr in (0.8, 0.9):
            same = bool(g[f"same_{name}_{int(thr * 10)}"])
            i, j, s = oracle.pairs_above(E, thr)
            assert (len(i) > 0) == same
    E = synth.synth_rows(int(g["pairs_seed"]), 0, int(g["pairs_n"]), int(g["pairs_d"]), int(g["pairs_dup"]))
    E[50] = 0.0
    for thr in (0.8, 0.9):
        i, j, s = oracle.pairs_above(E, thr)
        t = int(thr * 10)
        assert np.array_equal(i, g[f"pairs_i_{t}"]) and np.array_equal(j, g[f"pairs_j_{t}"])
        np.testing.assert_allclose(s, g[f"pairs_s_{t}"], rtol=1e-5)  # BLAS order unspecified -> tolerance
        # the streamed tier (BLAS pre-scoring + the same decision arithmetic) is the same set, bit for bit
        si, sj, ss = oracle.pairs_above_streamed(E, thr, block=64)
        assert np.array_equal(si, i) and np.array_equal(sj, j) and np.array_equal(ss, s)


def test_streamed_pair_tier_equals_the_scalar_tier():
    """oracle.pairs_above_streamed (used where the O(N^2 D) loop takes hours) against oracle.pairs_above: ragged last
    blocks, one block, zero rows, a threshold low enough for ~10^6 hits, thresholds at / around an attained score."""
    for n, d, thr, dup, block in [(3000, 768, 0.9, 20, 1024), (5000, 96, 0.5, 7, 4096), (2049, 384, 0.05, 0, 512),
                                  (1, 8, 0.5, 0, 8), (2, 8, -1.0, 0, 8), (700, 64, 0.3, 3, 8192)]:
        E = oracle.synth_rows_c(44, 0, n, d, dup)
        if n > 100:
            E[17] = 0.0
        a = oracle.pairs_above(E, thr)
        b = oracle.pairs_above_streamed(E, thr, block=block)
        assert all(np.array_equal(x, y) for x, y in zip(a, b)), (n, d, thr)
    E = oracle.synth_rows_c(45, 0, 600, 128, 5)
    _, _, s = oracle.pairs_above(E, 0.6)
    for thr in (float(s[3]), float(np.nextafter(s[3], np.float32(0))), float(np.nextafter(s[3], np.float32(2)))):   # strict >
        a, b = oracle.pairs_above(E, thr), oracle.pairs_above_streamed(E, thr, block=256)
        assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_vector_search_semantics():
    # PARITY UNPINNED (Neo4j server not runnable here): checks the documented convention only.
    X = synth.synth_rows(9, 0, 64, 32)
    q = X[7].copy()
    got = oracle.vector_search(q, X, 5, 0.3)
    assert got[0] == (7, 1.0)
    raw = oracle.batch_similarities(q[None], X, 64)[0]
    expect = [(r, (1.0 + s) / 2.0) for r, s in raw if (1.0 + s) / 2.0 > 0.3][:5]
    assert got == expect


def test_threshold_filter_inclusive():
    X = synth.synth_rows(9, 0, 16, 32)
    q = X[3]
    s3 = oracle.cosine(q, X[3], "retriever")
    kept = oracle.threshold_filter_ge(q, X, s3, 10)
    assert (3, s3) in kept  # `>=` keeps the boundary (retriever_hybrid.py:499)


def test_synth_numpy_equals_c():
    for dup in (0, 7):
        assert np.array_equal(synth.synth_rows(5, 1000, 300, 384, dup), oracle.synth_rows_c(5, 1000, 300, 384, dup))
    v = synth.synth_rows(5, 0, 64, 768) * 128
    assert np.array_equal(v, np.round(v)) and np.abs(v).max() <= 127


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present (see oracle/ref_import.py)")
def test_oracle_against_live_reference():
    X = synth.synth_rows(77, 0, 120, 96)
    Q = synth.synth_queries(78, 3, 96, 77, 120)
    store = {f"c{i}": [float(v) for v in X[i]] for i in range(len(X))}
    ref = ref_import.run_batch_similarities([[float(v) for v in q] for q in Q], store, 5)
    got = oracle.batch_similarities(Q, X, 5)
    assert [[(int(c[1:]), s) for c, s in l] for l in ref] == got
