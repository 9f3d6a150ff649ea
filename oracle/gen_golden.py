"""Generate tests/golden/*.npz by running the UNMODIFIED reference functions.

Needs a checkout of the reference project (see oracle/ref_import.py):  python -m oracle.gen_golden
The reference ships no golden vectors for this path (SURVEY.md section 4), so these
fixtures -- outputs of the reference's own code on seeded synthetic inputs -- are what pins
the oracle (tests/test_oracle_golden.py) and, through it, the CUDA path.
Interpreter that produced the committed fixtures: CPython 3.12.3 (Neumaier `sum`), numpy 2.3,
scikit-learn 1.9.0.
"""
from __future__ import annotations

import contextlib
import io
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_import, synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _lists(a):
    return [[float(v) for v in row] for row in a]


def gen_cosine_kat(ref):
    rng = np.random.default_rng(20261018)
    inj = ref_import.make_injector(3)
    HR, EU = ref["HybridRetriever"], ref["EmbeddingUtils"]
    cases = []
    for t in range(64):
        n1 = int(rng.choice([1, 2, 3, 8, 48, 384]))
        n2 = n1 if t % 5 else int(rng.choice([1, 2, 7, 48]))
        scale = 10.0 ** rng.integers(-3, 4)
        v1 = rng.uniform(-1, 1, n1) * scale
        v2 = rng.uniform(-1, 1, n2)
        if t % 11 == 3:
            v1[:] = 0.0
        if t % 13 == 5:
            v2[:] = 0.0
        if t % 17 == 7:
            v1 *= 1e-170
            v2 *= 1e-170  # magnitude product underflows -> HybridRetriever returns 0.0
        cases.append((v1, v2))
    maxn = max(max(len(a), len(b)) for a, b in cases)
    A = np.zeros((len(cases), maxn))
    B = np.zeros((len(cases), maxn))
    la = np.array([len(a) for a, _ in cases])
    lb = np.array([len(b) for _, b in cases])
    out = np.zeros((len(cases), 3))
    for i, (a, b) in enumerate(cases):
        A[i, :len(a)], B[i, :len(b)] = a, b
        out[i, 0] = inj._cosine_similarity(list(map(float, a)), list(map(float, b)))
        out[i, 1] = HR._cosine_similarity(list(map(float, a)), list(map(float, b)))
        out[i, 2] = EU.cosine_similarity(list(map(float, a)), list(map(float, b)))
    np.savez_compressed(os.path.join(OUT, "cosine_kat.npz"), a=A, b=B, len_a=la, len_b=lb, out=out)


def gen_batch_small(ref):
    n, d, q = 160, 48, 6
    X = synth.synth_rows(101, 0, n, d)
    X[17] = X[5]          # exact duplicate rows -> tie broken by store order
    X[99] = X[5]
    X[33] = 0.0           # zero-norm row -> score 0.0
    X[64] = 2.0 * X[63]   # colinear rows: equal cosine up to rounding
    row_ok = np.ones(n, np.uint8)
    row_ok[[8, 120]] = 0  # falsy embedding (None / []) -> skipped (:363)
    Q = synth.synth_queries(202, q, d, 101, n)
    Q[1] = X[5]           # query equal to the triplicated row
    Q[4] = 0.0            # zero query -> every score 0.0 -> first k rows in store order
    query_ok = np.ones(q, np.uint8)
    query_ok[3] = 0       # Exception-valued embedding -> [] (:357-359)
    store = {}
    for i in range(n):
        store[f"c{i}"] = _lists(X[i:i + 1])[0] if row_ok[i] else (None if i == 8 else [])
    queries = [_lists(Q[i:i + 1])[0] if query_ok[i] else RuntimeError("embed failed") for i in range(q)]
    res = {}
    for k in (3, 10, 200):
        out = ref_import.run_batch_similarities(queries, store, k)
        idx = np.full((q, k), -1, np.int64)
        sc = np.zeros((q, k))
        cnt = np.zeros(q, np.int64)
        for i, lst in enumerate(out):
            cnt[i] = len(lst)
            for j, (cid, s) in enumerate(lst):
                idx[i, j], sc[i, j] = int(cid[1:]), s
        res[f"idx_k{k}"], res[f"score_k{k}"], res[f"count_k{k}"] = idx, sc, cnt
    np.savez_compressed(os.path.join(OUT, "batch_small.npz"), X=X, Q=Q, row_ok=row_ok, query_ok=query_ok, **res)


def gen_batch_c1(ref):
    """Config C1: 5 000 x 384 store, 30 queries, top-10 (inputs re-derived from the seeds)."""
    n, d, q, k = 5000, 384, 30, 10
    X = synth.synth_rows(1, 0, n, d)
    Q = synth.synth_queries(1001, q, d, 1, n)
    store = {f"c{i}": row for i, row in enumerate(_lists(X))}
    out = ref_import.run_batch_similarities(_lists(Q), store, k)
    idx = np.array([[int(c[1:]) for c, _ in lst] for lst in out], np.int64)
    sc = np.array([[s for _, s in lst] for lst in out])
    np.savez_compressed(os.path.join(OUT, "batch_c1.npz"), store_seed=1, query_seed=1001, n=n, d=d, q=q, k=k,
                        idx=idx, score=sc)


def gen_merge(ref):
    """Cross-query merge, pre_llm_injector.py:235-249, executed verbatim on the reference lists."""
    inj = ref_import.make_injector(3, 2)
    n, d, q = 160, 48, 5
    X = synth.synth_rows(101, 0, n, d)
    X[17] = X[5]
    Q = synth.synth_queries(303, q, d, 101, n)
    Q[1] = Q[0]
    store = {f"c{i}": row for i, row in enumerate(_lists(X))}
    res = {}
    for k, k2 in ((3, 2), (10, 4), (10, 25)):
        batch = ref_import.run_batch_similarities(_lists(Q), store, k)
        # ---- verbatim semantics of :238-249 ----
        final_scores = {}
        for chunk_similarities in batch:
            for chunk_id, score in chunk_similarities:
                if chunk_id not in final_scores or score > final_scores[chunk_id]:
                    final_scores[chunk_id] = score
        final = sorted(final_scores.items(), key=lambda x: x[1], reverse=True)[:k2]
        res[f"idx_{k}_{k2}"] = np.array([int(c[1:]) for c, _ in final], np.int64)
        res[f"score_{k}_{k2}"] = np.array([s for _, s in final])
    np.savez_compressed(os.path.join(OUT, "merge.npz"), X=X, Q=Q, **res)


def gen_prune(ref):
    from sklearn.metrics.pairwise import cosine_similarity
    res = {}
    g = ref_import.make_graph(lambda s: np.asarray(s, dtype=np.float32))
    for name, (seed, n, d, dup) in {"a": (3, 6, 768, 2), "b": (4, 9, 384, 0), "c": (5, 2, 768, 1), "d": (6, 1, 64, 0)}.items():
        E = synth.synth_rows(seed, 0, n, d, dup_period=dup)
        if name == "b":
            E[4] = 0.0
        with contextlib.redirect_stdout(io.StringIO()):
            rep = int(g._get_representative_relation(E))
        res[f"E_{name}"] = E
        res[f"rep_{name}"] = rep
        for thr in (0.8, 0.9):
            res[f"same_{name}_{int(thr * 10)}"] = bool(g._are_same_context(E, thr))
    # generalised pair set from sklearn itself (the arithmetic prune.py:76-79 runs)
    n, d = 192, 768
    E = synth.synth_rows(44, 0, n, d, dup_period=4)
    E[50] = 0.0
    S = cosine_similarity(E)
    np.fill_diagonal(S, 0)
    for thr in (0.8, 0.9):
        ii, jj = np.nonzero(np.triu(S > np.float32(thr), 1))
        res[f"pairs_i_{int(thr * 10)}"], res[f"pairs_j_{int(thr * 10)}"] = ii.astype(np.int64), jj.astype(np.int64)
        res[f"pairs_s_{int(thr * 10)}"] = S[ii, jj].astype(np.float32)
    res["pairs_seed"], res["pairs_n"], res["pairs_d"], res["pairs_dup"] = 44, n, d, 4
    np.savez_compressed(os.path.join(OUT, "prune.npz"), **res)


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = ref_import.load()
    gen_cosine_kat(ref)
    gen_batch_small(ref)
    gen_merge(ref)
    gen_prune(ref)
    gen_batch_c1(ref)
    print("wrote", sorted(os.listdir(OUT)))


if __name__ == "__main__":
    main()
