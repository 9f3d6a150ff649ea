"""The CUDA-graph fast path of host-buffer top-k calls.  After 16 calls on the legacy default stream without a
mutation in between, a one-batch host-buffer call is captured into a graph (a 4-entry cache keyed on the call's
shape and the store version) and later calls replay it.  These tests drive the branches of that path: the re-run
of a batch with uncertified queries, eviction from the cache, and a mutation between replays."""
import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu

STABLE_CALLS = 17   # calls after which the graph path takes over


@pytest.fixture(scope="module")
def vm():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import vidmem_b200
    vidmem_b200._lib.load()
    return vidmem_b200


def _plain(vm, st, Q, k):
    """The same call through the plain path: a non-default stream never takes the graph path."""
    import torch
    with torch.cuda.stream(torch.cuda.Stream()):
        return st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)


def _same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("scale", [1e-30, 1e25])
def test_uncertified_replay_reruns_the_plain_path(vm, scale):
    """Rows at an extreme scale leave every query uncertified: each replay hands the batch to the plain path,
    which settles it with the binary64 scan."""
    d, n, k = 128, 20000, 10
    rng = np.random.default_rng(11)
    X = rng.standard_normal((n, d)).astype(np.float32)
    X[100:140] = (X[100:140].astype(np.float64) * scale).astype(np.float32)
    Q = rng.standard_normal((6, d)).astype(np.float32)
    Q[0] = (X[120].astype(np.float64) / scale).astype(np.float32)
    st = vm.EmbeddingStore(d, n, "f32")
    st.append(X)
    ref = oracle.batch_similarities(Q, X, k)
    for call in range(STABLE_CALLS + 4):
        idx, score, count = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
        for qi, lst in enumerate(ref):
            assert count[qi] == len(lst), (call, qi)
            assert list(idx[qi, :len(lst)]) == [r for r, _ in lst], (call, qi)
            assert list(score[qi, :len(lst)]) == [s for _, s in lst], (call, qi)
        assert st.last_stats.uncertified == len(Q), call
    assert ref[0][0][0] == 120
    st.close()


def test_graph_cache_eviction(vm):
    """More distinct (nq, k) shapes than the cache holds, cycled twice, each shape called twice in a row (a
    capture, then a replay of the fresh entry): every answer equals the plain path's.  k = 64 is beyond the fast
    scans, so its graph holds the binary64 scan alone."""
    d, n = 128, 5000
    rng = np.random.default_rng(12)
    X = rng.standard_normal((n, d)).astype(np.float32)
    st = vm.EmbeddingStore(d, n, "f32")
    st.append(X)
    Q = rng.standard_normal((40, d)).astype(np.float32)
    shapes = [(1, 5), (3, 10), (8, 1), (16, 16), (30, 24), (40, 48), (5, 64)]
    plain = {s: _plain(vm, st, Q[:s[0]], s[1]) for s in shapes}
    for _ in range(STABLE_CALLS):
        st.topk(Q[:2], 3, sum_mode=vm.VM_SUM_NEUMAIER)
    for rnd in range(2):
        for nq, k in shapes:
            for rep in range(2):
                got = st.topk(Q[:nq], k, sum_mode=vm.VM_SUM_NEUMAIER)
                assert _same(got, plain[(nq, k)]), (rnd, nq, k, rep)
    st.close()


def test_mutation_between_replays(vm):
    """An append bumps the store version: the next call, and every replay after the graph is captured again,
    returns the new row as the top hit."""
    d, n, k = 128, 5000, 8
    rng = np.random.default_rng(13)
    X = rng.standard_normal((n, d)).astype(np.float32)
    st = vm.EmbeddingStore(d, n + 1, "f32")
    st.append(X)
    Q = rng.standard_normal((4, d)).astype(np.float32)
    before = _plain(vm, st, Q, k)
    for _ in range(STABLE_CALLS + 2):
        assert _same(st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER), before)
    new_row = st.append(Q[2:3] * 3.0)   # the same direction as query 2: its best hit
    after = _plain(vm, st, Q, k)
    assert after[0][2, 0] == new_row and not _same(after, before)
    for call in range(STABLE_CALLS + 2):
        got = st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)
        assert got[0][2, 0] == new_row, call
        assert _same(got, after), call
    st.close()
