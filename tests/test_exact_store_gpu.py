"""Binary64 stores ("f64": fp32 shadow, "f64+bf16": bf16 shadow): the reference scores Python float lists, i.e.
binary64 values (pre_llm_injector.py:382-388).  The scan reads a rounded shadow copy, every exact step reads the
original rows, so index lists and binary64 scores must equal the oracle's ON THE ORIGINAL float64 INPUTS -- including
rows that are indistinguishable after rounding to fp32."""
import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

EXACT = ["f64", "f64+bf16"]


@pytest.fixture(scope="module")
def vm():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import vidmem_b200
    vidmem_b200._lib.load()
    return vidmem_b200


def _check(idx, score, count, ref):
    for qi, lst in enumerate(ref):
        assert count[qi] == len(lst), (qi, count[qi], len(lst))
        assert list(idx[qi, :len(lst)]) == [r for r, _ in lst], (qi, idx[qi], lst)
        assert list(score[qi, :len(lst)]) == [s for _, s in lst], qi  # bit-exact binary64
        assert (idx[qi, len(lst):] == -1).all()


def _twins(rng, n, d, nq):
    """Rows that are exactly fp32-representable, plus for every query a 'twin pair': row a, and a LATER row b = a moved
    towards the query by 1e-12 per element -- far below half an fp32 ulp, so both round to the same fp32 vector, while in
    binary64 b scores higher than a.  The reference therefore ranks b before a; a store of rounded values sees a tie and
    ranks the earlier row a first."""
    X = rng.standard_normal((n, d)).astype(np.float32).astype(np.float64)
    Q = rng.standard_normal((nq, d))
    pairs = []
    for qi in range(nq):
        a, b = 10 + 37 * qi, n - 5 - 11 * qi
        base = (Q[qi] + 0.3 * rng.standard_normal(d)).astype(np.float32).astype(np.float64)   # a strong match of query qi
        X[a] = base
        mv = np.where(np.abs(base) > 0.05, 1e-12 * Q[qi], 0.0)
        X[b] = base + mv
        assert np.array_equal(X[a].astype(np.float32), X[b].astype(np.float32)) and not np.array_equal(X[a], X[b])
        pairs.append((a, b))
    return X, Q, pairs


@pytest.mark.parametrize("dtype", EXACT)
@pytest.mark.parametrize("n", [3000, 20011])      # dump mode / slab mode of the tcgen05 scan
def test_exact_store_ranks_by_the_original_values(vm, dtype, n):
    d, nq, k = 384, 9, 10
    rng = np.random.default_rng(5 + n)
    X, Q, pairs = _twins(rng, n, d, nq)
    ref = oracle.batch_similarities(Q, X, k)
    for qi, (a, b) in enumerate(pairs):
        assert [r for r, _ in ref[qi][:2]] == [b, a]           # the reference prefers the later twin
    st = vm.EmbeddingStore(d, n + 7, dtype)
    st.append(X[:1234]); st.append(X[1234:])
    for flags in (0, vm.VM_FLAG_FORCE_SIMT):
        idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER, flags=flags)
        _check(idx, score, count, ref)
    c = st.counters()
    assert c["bound_violations"] == 0 and c["full_rescans"] == 0       # the twins are told apart by the rescoring itself
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER, flags=vm.VM_FLAG_FORCE_EXACT)
    _check(idx, score, count, ref)
    # the naive recurrence (CPython < 3.12) on the same store
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NAIVE)
    _check(idx, score, count, oracle.batch_similarities(Q, X, k, sum_mode=oracle.SUM_NAIVE))
    # what the binary64 rows buy: an fp32 store of the same inputs cannot tell the twins apart
    s32 = vm.EmbeddingStore(d, n, "f32")
    s32.append(X)
    i32, _, _ = s32.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
    assert all(list(i32[qi, :2]) == [a, b] for qi, (a, b) in enumerate(pairs))
    s32.close()
    # upsert of a twin with its sibling's value -> a true tie -> earliest row wins again; skipped rows vanish
    st.update(pairs[0][1], X[pairs[0][0]][None, :])
    st.invalidate([pairs[1][1]])
    X2 = X.copy(); X2[pairs[0][1]] = X[pairs[0][0]]
    ok = np.ones(n, np.uint8); ok[pairs[1][1]] = 0
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
    ref2 = oracle.batch_similarities(Q, X2, k, row_ok=ok)
    _check(idx, score, count, ref2)
    assert [r for r, _ in ref2[0][:2]] == [pairs[0][0], pairs[0][1]]
    st.close()


@pytest.mark.parametrize("dtype", EXACT)
def test_exact_store_general_float64_values(vm, dtype):
    """Values with full 53-bit mantissas, a near-duplicate cluster (cosines within 1e-7 of each other: one fp32 ulp),
    duplicates, a zero row, device-side queries."""
    import torch
    d, n, nq, k = 384, 40_000, 33, 10
    rng = np.random.default_rng(77)
    X = rng.standard_normal((n, d)) * np.exp(rng.uniform(-3, 3, (n, 1)))
    centre = rng.standard_normal(d)
    X[5000:5064] = centre + 1e-7 * rng.standard_normal((64, d))        # 64 rows, all within ~1e-13 in cosine
    X[7000] = X[6000]; X[7001] = 3.5 * X[6000]                          # exact duplicate, positive multiple
    X[123] = 0.0
    Q = rng.standard_normal((nq, d))
    Q[0] = centre + 1e-3 * rng.standard_normal(d)
    Q[1] = X[6000]
    st = vm.EmbeddingStore(d, n, dtype)
    st.append(torch.from_numpy(X).cuda())                               # binary64 device source
    ref = oracle.batch_similarities(Q, X, k)
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
    _check(idx, score, count, ref)
    di, ds, dc = st.topk_device(torch.from_numpy(Q).cuda(), k, sum_mode=vm.VM_SUM_NEUMAIER, flags=vm.VM_FLAG_ASYNC)
    torch.cuda.synchronize()
    _check(di.cpu().numpy(), ds.cpu().numpy(), dc.cpu().numpy(), ref)
    c = st.counters()
    assert c["bound_violations"] == 0 and c["full_rescans"] == 0        # settled by the scan + band, no fallback
    st.close()


def test_exact_store_rows_the_shadow_cannot_hold(vm):
    """A row of 1e-60s (flushes to zero in fp32) and a row of 1e60s (overflows fp32) are ordinary vectors for the
    reference; the store counts them as out of range and answers every query through the binary64 pass."""
    d, n, k = 64, 5000, 5
    rng = np.random.default_rng(3)
    X = rng.standard_normal((n, d))
    Q = rng.standard_normal((4, d))
    X[100] = 1e-60 * Q[0]
    X[200] = 1e60 * Q[1]
    ref = oracle.batch_similarities(Q, X, k)
    assert ref[0][0][0] == 100 and ref[1][0][0] == 200
    st = vm.EmbeddingStore(d, n, "f64")
    st.append(X)
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
    _check(idx, score, count, ref)
    assert st.counters()["full_rescans"] == 4
    st.close()


def test_exact_store_wide_rows_take_the_fused_rescoring(vm):
    """1536-d binary64 rows: 32 whole candidate rows do not fit shared memory, so the rescoring kernel streams them through
    its window of column chunks."""
    d, n, k = 1536, 12_000, 10
    rng = np.random.default_rng(8)
    X = rng.standard_normal((n, d))
    Q = rng.standard_normal((5, d))
    Q[0] = X[4242] + 0.05 * rng.standard_normal(d)
    st = vm.EmbeddingStore(d, n, "f64")
    st.append(X)
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
    _check(idx, score, count, oracle.batch_similarities(Q, X, k))
    assert idx[0, 0] == 4242
    st.close()


@pytest.mark.parametrize("dtype", EXACT)
def test_exact_store_sidecar_and_prefix_view(vm, dtype, tmp_path):
    d, n, k = 96, 3000, 4
    rng = np.random.default_rng(12)
    X = rng.standard_normal((n, d))
    Q = rng.standard_normal((3, d))
    st = vm.EmbeddingStore(d, n, dtype)
    st.append(X)
    st.invalidate([17])
    p = str(tmp_path / "side")
    st.save(p, ids=[f"c{i}" for i in range(n)])
    st2, ids = vm.EmbeddingStore.load(p)
    assert st2.exact and st2.dtype_code == st.dtype_code and ids[5] == "c5"
    a, b = st.topk(Q, k), st2.topk(Q, k)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    ok = np.ones(n, np.uint8); ok[17] = 0
    _check(*a, oracle.batch_similarities(Q, X, k, row_ok=ok))
    v = st.prefix_view(1000)
    _check(*v.topk(Q, k), oracle.batch_similarities(Q, X[:1000], k, row_ok=ok[:1000]))
    v.close(); st.close(); st2.close()


@pytest.mark.parametrize("dtype", EXACT)
@pytest.mark.parametrize("n,d,nq,k", [(1, 8, 1, 1), (7, 24, 3, 10), (1000, 384, 5, 10), (4097, 768, 8, 3), (20000, 100, 2, 24),
                                      (3000, 384, 17, 10), (30000, 384, 64, 40), (9473, 200, 33, 10)])
def test_exact_store_every_path_vs_oracle(vm, dtype, n, d, nq, k):
    """Shapes x paths (tcgen05 scan incl. dump mode / slabs / 64-candidate lists, CUDA-core scan, binary64 scan) x both
    summation orders on float64 values; duplicates, a zero row, a query equal to a row."""
    rng = np.random.default_rng(n * 31 + d)
    X = rng.standard_normal((n, d)) * (1.0 + rng.random((n, 1)))
    Q = rng.standard_normal((nq, d))
    if n > 10:
        X[3] = X[1]; X[n - 1] = X[1]; X[5] = 0.0
        Q[0] = X[1]
    st = vm.EmbeddingStore(d, n + 5, dtype)
    st.append(X)
    for sm, osm in ((vm.VM_SUM_NEUMAIER, oracle.SUM_NEUMAIER), (vm.VM_SUM_NAIVE, oracle.SUM_NAIVE)):
        ref = oracle.batch_similarities(Q, X, k, sum_mode=osm)
        for flags in (0, vm.VM_FLAG_FORCE_SIMT, vm.VM_FLAG_FORCE_EXACT):
            if flags == vm.VM_FLAG_FORCE_SIMT and k > 24:
                continue
            idx, score, count = st.topk(Q, k, sum_mode=sm, flags=flags)
            _check(idx, score, count, ref)
    assert st.counters()["bound_violations"] == 0
    st.close()


@pytest.mark.parametrize("dtype", EXACT)
def test_exact_store_mass_duplicates_take_the_fallbacks(vm, dtype):
    """300 exact duplicates at the top (band settlement), 3 000 of them (beyond the band: collect pass), 6 000 of them
    (beyond the collect buffer: binary64 scan of every row) -- each fallback reads the binary64 rows -- and a zero query
    (every row ties at 0.0: store order, answered directly)."""
    d, n, k = 64, 20_000, 10
    rng = np.random.default_rng(5)
    X = rng.standard_normal((n, d))
    X[100:400] = X[100]
    X[5000:8000] = X[5000]
    X[10000:16000] = X[10000]
    Q = np.stack([X[100], X[5000], rng.standard_normal(d), np.zeros(d), X[10000]])
    st = vm.EmbeddingStore(d, n, dtype)
    st.append(X)
    idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
    _check(idx, score, count, oracle.batch_similarities(Q, X, k))
    assert list(idx[0]) == list(range(100, 110)) and list(idx[1]) == list(range(5000, 5010)) and list(idx[3]) == list(range(10))
    assert list(idx[4]) == list(range(10000, 10010))
    c = st.counters()
    assert c["uncertified"] == 3 and c["band_settled"] == 1 and c["collect_settled"] == 1 and c["full_rescans"] == 1
    assert c["bound_violations"] == 0
    st.close()

