"""The rescoring kernels' staged-row window at the edges of its shapes, against the binary64 oracle on the stored values.

Every exact answer passes through stage_and_chain, which streams candidate rows through three column-chunk slots sized
per shape (csrc/stage_window.h).  The dims come from the host build of that layout (stage_window_lib): the last dim whose
rows are staged whole, the first windowed dim, a windowed dim whose groups do not divide evenly into its chunks, a
windowed dim that is not a multiple of 8 (padding in the last chunk) and 4096.  At each one a query's near-tie band is
made of DISTINCT near-duplicates of one base row: every copy differs from the base in a single column, and the columns
cycle over the first and last column of every chunk (plus column dim-1), so a chunk staged from the wrong row, the
wrong columns or the wrong slot changes some copy's score.  The bands are sized from the shape's band capacity:
kp + 5 rows (first pass + a small band settlement), exactly the capacity (settled from the band) and one row more (the
collect pass, through collect_rescore_kernel's own window); 4096 and 4097 rows on a few shapes (the collect pass at its
capacity, the binary64 scan one row past it).  Runs on a non-default stream, so the plain path runs and the
certification counters are read back."""
import numpy as np
import pytest

from oracle import oracle
from stage_window_lib import SLAB, Harness

pytestmark = pytest.mark.gpu

# store kind -> (bytes per element of the rows the rescoring reads, host dtype of rows and queries)
KINDS = {"f32": (4, np.float32), "bf16": (2, np.float32), "f64": (8, np.float64), "f64+bf16": (8, np.float64)}
FP32_SCAN = ("f32", "f64")          # kinds whose scan reads fp32 rows (the tcgen05 kernel fits them up to ~2816-d)
ROLES = ["last_whole", "first_windowed", "ragged", "unaligned", "widest"]
N_SLAB, N_DUMP = 12_000, 9_000      # 94 tiles: union buffer (slab mode); 71 tiles: every key dumped
PIVOT = 0.1875                      # base value of every perturbed column (small: every copy stays in the band)
XS_CG = 24                          # 16-byte groups per chunk of the binary64 scan (select.cu)


@pytest.fixture(scope="module")
def vm():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import vidmem_b200
    vidmem_b200._lib.load()
    return vidmem_b200


@pytest.fixture(scope="module")
def H(tmp_path_factory):
    return Harness(tmp_path_factory.mktemp("stage_window"))


def _kp(k):
    return 32 if k <= 16 else 64


def _source(H, mode, n):
    return SLAB if mode == "slab" else H.dump_tiles(n)


def _dims(H, eb, kp, source):
    """The five dims of the shape edges for rows of eb bytes per element, kp candidates and this key source."""
    lists, list_len = (0, 0) if source == SLAB else source
    lay = H.select(eb, kp, lists, list_len)
    gpr, chunks = lay[:, 1], lay[:, 3]
    dim = np.arange(1, 4097)
    last_whole = int(dim[chunks == 3].max())
    win = chunks > 3
    ragged = dim[win & (dim > last_whole + 8) & (dim % 8 == 0) & (gpr % np.maximum(chunks, 1) != 0)]
    unaligned = [d for d in (1001, 2001, 3001) if win[d - 1] and d != last_whole + 1]
    return {"last_whole": last_whole, "first_windowed": last_whole + 1, "ragged": int(ragged[0]),
            "unaligned": unaligned[0], "widest": 4096}


def _boundary_columns(H, eb, dim, kp, source):
    """First and last column of every chunk of the select window and of the collect window, plus column dim - 1."""
    epg = 16 // eb
    gpr = ((dim + 7) & ~7) * eb // 16
    cols = {dim - 1}
    for chunks, pitch in (H.stage_regime(eb, dim, kp, source)[:2], H.collect_regime(eb, dim)):
        rc, lo, _ = H.walk(gpr, pitch, chunks)
        assert rc == 0
        for c in range(chunks):
            a, b = int(lo[c]) * epg, min(int(lo[c + 1]) * epg, dim)
            if a < b:
                cols.update((a, b - 1))
    return sorted(cols)


def _values(kind, m):
    """m distinct values of the stored type other than PIVOT, nearest first: bf16 values (steps of whole bf16 ulps),
    fp32 values one ulp apart, binary64 values 2^22 ulps apart (smaller steps would tie in the binary64 scores)."""
    if kind == "bf16":
        v = np.array([2.0 ** e * (1 + j / 128) for e in (-4, -3, -2) for j in range(128)])
        v = v[v != PIVOT]
        v = v[np.argsort(np.abs(v - PIVOT), kind="stable")]
    else:
        step = 2.0 ** -26 if kind == "f32" else 2.0 ** -33
        j = np.arange(1, m // 2 + 2)
        v = np.stack([PIVOT + j * step, PIVOT - j * step], 1).reshape(-1)
    assert len(v) >= m, (kind, m)
    return v[:m]


def _to_stored(kind, a):
    if kind != "bf16":
        return a.astype(KINDS[kind][1])
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).float().numpy()


def _make(H, kind, dim, kp, mode, n, bands, seed):
    """Random rows, plus one band of near-duplicates per entry of `bands` at shuffled row positions.  -> (X, band
    queries, random query, close query, band row lists)."""
    eb, ft = KINDS[kind]
    rng = np.random.default_rng(seed)
    X = _to_stored(kind, rng.standard_normal((n, dim)))
    cols = _boundary_columns(H, eb, dim, kp, _source(H, mode, n))
    pos = rng.permutation(n)
    used, band_rows, band_q = 0, [], []
    for B in bands:
        base = rng.standard_normal(dim)
        base[cols] = PIVOT
        base = _to_stored(kind, base)
        vals = _values(kind, -(-B // len(cols)))
        rows = np.sort(pos[used:used + B])
        rows = rng.permutation(rows)                 # copy i at a shuffled position
        used += B
        for i, r in enumerate(rows):
            X[r] = base
            X[r, cols[i % len(cols)]] = vals[i // len(cols)]
        band_rows.append(rows)
        band_q.append((base + 0.05 * rng.standard_normal(dim)).astype(ft))
    close = int(pos[used])
    rand_q = rng.standard_normal(dim).astype(ft)
    close_q = (X[close] + 0.05 * rng.standard_normal(dim)).astype(ft)
    return X, band_q, rand_q, close_q, band_rows, close


def _stored(st, n, dim):
    """The values the store holds (what the reference would score): binary64 originals or the rows themselves."""
    src = st.rows_exact if st.exact else st.rows
    return src[:n, :dim].double().cpu().numpy()


def _check(idx, score, count, ref, what):
    for qi, lst in enumerate(ref):
        assert count[qi] == len(lst), (what, qi, count[qi], len(lst))
        assert list(idx[qi, :len(lst)]) == [r for r, _ in lst], (what, qi, idx[qi], lst)
        assert list(score[qi, :len(lst)]) == [s for _, s in lst], (what, qi)   # bit-exact binary64
        assert (idx[qi, len(lst):] == -1).all(), what


def _topk(st, Q, k, vm, sum_mode=None, flags=0):
    import torch
    with torch.cuda.stream(torch.cuda.Stream()):   # non-default stream: the plain (non-graph) path
        return st.topk(np.stack(Q), k, sum_mode=vm.VM_SUM_NEUMAIER if sum_mode is None else sum_mode, flags=flags)


def _expected(kernel, B, band_cap, collect_cap):
    """Settlement of a band of B rows (B > kp) by the scan that ran."""
    if kernel == 0:                                 # binary64 scan only: no candidates, no certification
        return {"uncertified": 0, "band_settled": 0, "collect_settled": 0, "full_rescans": 0}
    if kernel == 1:                                 # per-CTA lists bound the outside rows by their last key only
        return {"uncertified": 1, "band_settled": 0, "collect_settled": 0, "full_rescans": 1}
    return {"uncertified": 1, "band_settled": int(B <= band_cap), "collect_settled": int(band_cap < B <= collect_cap),
            "full_rescans": int(B > collect_cap)}


def _check_scan(st, kind, dim, k, mode, what):
    """The scan that ran: tcgen05, except for fp32 rows beyond its reach, where the CUDA-core scan takes k <= 24 and
    the binary64 scan of every row (no rescoring kernel) the rest."""
    s = st.last_stats
    kernel = int(s.scan_kernel)
    assert kernel == (2 if kind not in FP32_SCAN or dim <= 2816 else (1 if k <= 24 else 0)), (what, kernel)
    if kernel == 2:
        assert (int(s.scan_variant) == 1) == (mode == "dump"), (what, int(s.scan_variant))
    return kernel


def _run_bands(vm, H, st, kind, dim, k, mode, n, X, bands, band_q, rand_q, close_q, band_rows, close, ref, what):
    eb = KINDS[kind][0]
    band_cap = H.stage_regime(eb, dim, _kp(k), _source(H, mode, n))[2]
    nb = len(bands)
    for j, B in enumerate(bands):
        w = what + (f"B={B}",)
        top = [r for r, _ in ref[j]]
        assert set(top) <= set(band_rows[j].tolist()), w
        assert top != sorted(band_rows[j].tolist())[:k], w        # the row-id tie-break alone cannot produce the list
        st.counters(reset=True)
        idx, score, count = _topk(st, [band_q[j], rand_q, close_q], k, vm)
        _check(idx, score, count, [ref[j], ref[nb], ref[nb + 1]], w)
        assert idx[2, 0] == close, w
        kernel = _check_scan(st, kind, dim, k, mode, w)
        assert st.counters()["bound_violations"] == 0, w
        # the band query alone: its settlement path, counted
        st.counters(reset=True)
        idx, score, count = _topk(st, [band_q[j]], k, vm)
        _check(idx, score, count, [ref[j]], w)
        assert _check_scan(st, kind, dim, k, mode, w) == kernel
        c = st.counters()
        assert c["bound_violations"] == 0, (w, c)
        assert {n_: c[n_] for n_ in ("uncertified", "band_settled", "collect_settled", "full_rescans")} == \
            _expected(kernel, B, band_cap, H.COLLECT_CAP), (w, kernel, band_cap, c)


CASES = [(kind, k, role, mode) for kind in KINDS for k in (10, 40) for role in ROLES for mode in ("slab", "dump")
         if mode == "slab" or kind.startswith("f64")]


@pytest.mark.parametrize("kind,k,role,mode", CASES, ids=["-".join(map(str, c)) for c in CASES])
def test_band_at_window_edges(vm, H, kind, k, role, mode):
    """Bands of kp + 5, band_cap and band_cap + 1 distinct near-duplicates; bit-exact lists and expected settlement.
    Also, on some shapes: the naive summation order, the CUDA-core scan's lists and the binary64 scan."""
    eb, ft = KINDS[kind]
    kp = _kp(k)
    n = N_SLAB if mode == "slab" else N_DUMP
    dim = _dims(H, eb, kp, _source(H, mode, n))[role]
    band_cap = H.stage_regime(eb, dim, kp, _source(H, mode, n))[2]
    bands = [kp + 5, band_cap, band_cap + 1]
    what = (kind, k, role, mode, dim)
    X, band_q, rand_q, close_q, band_rows, close = _make(H, kind, dim, kp, mode, n, bands, seed=dim * 131 + k + len(kind))
    st = vm.EmbeddingStore(dim, n, kind)
    try:
        st.append(X)
        Xs = _stored(st, n, dim)
        assert np.array_equal(Xs, X.astype(np.float64)), what    # the perturbations survive storage
        Q = band_q + [rand_q, close_q]
        ref = oracle.batch_similarities(np.stack(Q), Xs, k)
        _run_bands(vm, H, st, kind, dim, k, mode, n, X, bands, band_q, rand_q, close_q, band_rows, close, ref, what)

        if role in ("first_windowed", "widest"):
            # the reference's summation order before CPython 3.12, through the first pass and the collect pass
            Qn = [band_q[0], band_q[2], rand_q, close_q]
            refn = oracle.batch_similarities(np.stack(Qn), Xs, k, sum_mode=oracle.SUM_NAIVE)
            st.counters(reset=True)
            _check(*_topk(st, Qn, k, vm, sum_mode=vm.VM_SUM_NAIVE), refn, what + ("naive",))
            assert st.counters()["bound_violations"] == 0, what
        if k == 10 and role != "last_whole" and mode == "slab":
            # the CUDA-core scan: per-CTA lists of kp 24 keys as the key source
            st.counters(reset=True)
            _check(*_topk(st, [band_q[0], rand_q, close_q], k, vm, flags=vm.VM_FLAG_FORCE_SIMT),
                   [ref[0], ref[3], ref[4]], what + ("simt",))
            assert int(st.last_stats.scan_kernel) == 1, what
            assert st.counters()["bound_violations"] == 0, what
        gpr = ((dim + 7) & ~7) * eb // 16
        if k == 10 and gpr % XS_CG != 0 and mode == "slab":
            # the binary64 scan of every row, whose last 24-group chunk is partial here
            _check(*_topk(st, Q, k, vm, flags=vm.VM_FLAG_FORCE_EXACT), ref, what + ("exact",))
    finally:
        st.close()


WIDE_BANDS = [("f32", 10, "first_windowed", "slab"), ("bf16", 40, "widest", "slab"), ("f64+bf16", 40, "widest", "dump"),
              ("f64", 10, "unaligned", "slab")]


@pytest.mark.parametrize("kind,k,role,mode", WIDE_BANDS, ids=["-".join(map(str, c)) for c in WIDE_BANDS])
def test_band_at_collect_capacity(vm, H, kind, k, role, mode):
    """4096 near-duplicates: the collect pass, full to its capacity.  4097: one row past it, the binary64 scan."""
    eb, ft = KINDS[kind]
    kp = _kp(k)
    n = N_SLAB if mode == "slab" else 9472
    dim = _dims(H, eb, kp, _source(H, mode, n))[role]
    bands = [H.COLLECT_CAP, H.COLLECT_CAP + 1]
    what = (kind, k, role, mode, dim)
    X, band_q, rand_q, close_q, band_rows, close = _make(H, kind, dim, kp, mode, n, bands, seed=dim * 7 + k)
    st = vm.EmbeddingStore(dim, n, kind)
    try:
        st.append(X)
        Xs = _stored(st, n, dim)
        assert np.array_equal(Xs, X.astype(np.float64)), what
        ref = oracle.batch_similarities(np.stack(band_q + [rand_q, close_q]), Xs, k)
        _run_bands(vm, H, st, kind, dim, k, mode, n, X, bands, band_q, rand_q, close_q, band_rows, close, ref, what)
    finally:
        st.close()
