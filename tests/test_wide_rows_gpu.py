"""Stores whose kp candidate rows do not fit shared memory whole (wide fp32 rows, binary64 stores): the rescoring kernel
streams the rows through a window of column chunks, so these shapes take the same one-launch path as narrow rows --
near-tie band settlement included -- and stay bit-exact against the oracle."""
import numpy as np
import pytest

from oracle import oracle

pytestmark = pytest.mark.gpu


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


def _topk_on_side_stream(st, Q, k, vm):
    import torch
    with torch.cuda.stream(torch.cuda.Stream()):                     # non-default stream: the plain (non-graph) path
        return st.topk(Q, k, sum_mode=vm.VM_SUM_NEUMAIER)


@pytest.mark.parametrize("dtype,d,k", [("f32", 1536, 10), ("f64", 384, 20), ("f64", 1536, 10), ("f32", 3072, 10)])
def test_wide_rows_duplicate_band(vm, dtype, d, k):
    """300 exact duplicates at the top of one query, next to an ordinary query and one close to a single row.  The
    tcgen05 scan's band is complete, so the rescoring kernel settles the duplicates itself: no collect pass, no binary64
    scan.  At 3072-d fp32 the CUDA-core scan runs (the tcgen05 kernel fits fp32 up to ~2816-d); its per-CTA lists bound
    the rows outside them by each list's last key only, so a band wider than the lists goes to the binary64 scan."""
    n = 20_000
    rng = np.random.default_rng(d + k)
    ft = np.float32 if dtype == "f32" else np.float64
    X = rng.standard_normal((n, d)).astype(ft)
    X[100:400] = X[100]
    Q = np.stack([X[100], rng.standard_normal(d).astype(ft), (X[7777] + 0.05 * rng.standard_normal(d)).astype(ft)])
    st = vm.EmbeddingStore(d, n, dtype)
    st.append(X)
    idx, score, count = _topk_on_side_stream(st, Q, k, vm)
    _check(idx, score, count, oracle.batch_similarities(Q, X, k))
    assert list(idx[0]) == list(range(100, 100 + k)) and idx[2, 0] == 7777
    c = st.counters()
    assert c["uncertified"] == 1 and c["collect_settled"] == 0 and c["bound_violations"] == 0
    if d == 3072:
        assert c["band_settled"] == 0 and c["full_rescans"] == 1
    else:
        assert c["band_settled"] == 1 and c["full_rescans"] == 0
    st.close()


def test_widest_rows_parity(vm):
    """4096-d fp32, the largest dimension the store accepts."""
    d, n, k = 4096, 12_000, 10
    rng = np.random.default_rng(4096)
    X = rng.standard_normal((n, d)).astype(np.float32)
    Q = np.stack([rng.standard_normal(d), X[42] + 0.05 * rng.standard_normal(d)]).astype(np.float32)
    st = vm.EmbeddingStore(d, n, "f32")
    st.append(X)
    idx, score, count = _topk_on_side_stream(st, Q, k, vm)
    _check(idx, score, count, oracle.batch_similarities(Q, X, k))
    assert idx[1, 0] == 42
    assert st.counters()["bound_violations"] == 0
    st.close()
