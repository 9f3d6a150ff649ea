"""The scans' error bound eps at its edge: stores whose rounding pushes one row's approximate score as far below its
exact score as each scan allows (constructions and host models in scan_eps_lib), against the binary64 oracle.

Each store holds one target row r*, the exact top-1, whose scanned score s~* falls short of s* by a large share of eps;
N_DECOYS (>= kp + 8) decoys at lower and higher row ids whose exact scores sit a few 1e-5 below s* and whose values
the scan reads exactly; and filler rows of low cosine.  The rescoring certifies a list once every key >= s_k - eps has
been rescored, and s_k is a decoy's score, so if the true deviation of r* exceeded eps, r* would never be rescored
and the answer would lack it, with no counter moving (the rescoring audits only the rows it rescored).  Each case runs
in dump mode (every row's key ranked) and slab mode (the union buffer), k = 1 and 10, at 64, 384 and 4096 dims, and
asserts bit-exact parity with the oracle, r* first, zero bound violations and zero binary64 rescans, and which scan
ran.  The host model asserts beforehand that the construction reaches its stated share of eps."""
import functools

import numpy as np
import pytest

from oracle import oracle
from scan_eps_lib import (CUDA_CORE, N_DECOYS, TCGEN05, VM_BF16, VM_F32, Eps, rounding_construction,
                          shadow_construction, to_bf16, tf32_trunc)

pytestmark = pytest.mark.gpu

N = {"dump": 9_000, "slab": 20_011}     # 71 tiles: every key dumped; 157 tiles: union buffer
DIMS = (64, 384, 4096)
KS = (1, 10)
TC_FP32_MAX_DIM = 2816                  # widest fp32 rows the tcgen05 scan takes (wider: the CUDA-core scan, k <= 24)

# variant -> (store kind, scanned dtype, flags, split query, share of eps the modelled deviation must reach or None)
VARIANTS = {
    "f64+bf16-split": ("f64+bf16", VM_BF16, 0, True, 0.6),
    "f64+bf16-single": ("f64+bf16", VM_BF16, "NO_SPLIT", False, None),
    "f64": ("f64", VM_F32, 0, False, 0.9),
    "f32": ("f32", VM_F32, 0, False, 0.9),
    "bf16-single": ("bf16", VM_BF16, "NO_SPLIT", False, 0.8),
}
KINDS = ("f64+bf16", "f64", "f32", "bf16")


@pytest.fixture(scope="module")
def vm():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import vidmem_b200
    vidmem_b200._lib.load()
    return vidmem_b200


@pytest.fixture(scope="module")
def E(tmp_path_factory):
    return Eps(tmp_path_factory.mktemp("scan_eps"))


def _construction(kind, dim):
    if kind == "f64+bf16":
        return shadow_construction(dim)
    return rounding_construction(dim, VM_BF16 if kind == "bf16" else VM_F32, exact=kind == "f64")


@functools.lru_cache(maxsize=1)
def _fillers(n, dim):
    """Rows of negative expected cosine with the (non-negative) queries."""
    return np.random.default_rng(n * 7 + dim).standard_normal((n, dim), dtype=np.float32) - np.float32(0.5)


def _store_values(kind, dim, n, c):
    """-> (rows as given to the store, row of r*, decoy rows).  r* sits mid-store, the decoys on both sides of it."""
    X = _fillers(n, dim).astype(np.float64)
    rng = np.random.default_rng(dim + n)
    target = n // 2 + 3
    others = np.setdiff1d(np.arange(n), [target])
    decoys = np.sort(np.r_[rng.choice(others[others < target], N_DECOYS // 2, replace=False),
                           rng.choice(others[others > target], N_DECOYS - N_DECOYS // 2, replace=False)])
    X[target] = c.target
    X[decoys] = np.stack(c.decoys)
    if kind == "f32":
        X = X.astype(np.float32)
    elif kind == "bf16":
        X = to_bf16(X)
    return X, target, decoys


def _check(idx, score, count, ref, what):
    assert count[0] == len(ref), what
    assert list(idx[0, :len(ref)]) == [r for r, _ in ref], (what, idx[0], ref)
    assert list(score[0, :len(ref)]) == [s for _, s in ref], what      # bit-exact binary64


def _topk(vm, st, q, k, flags):
    import torch
    with torch.cuda.stream(torch.cuda.Stream()):    # non-default stream: the plain path, counters read back
        return st.topk(q[None], k, sum_mode=vm.VM_SUM_NEUMAIER, flags=flags)


def _flags(vm, f):
    return getattr(vm, "VM_FLAG_" + f) if isinstance(f, str) else f


def _model_share(E, c, dtype, dim, split, shadow, share, what):
    """The modelled deviation of r* as a share of the variant's eps; asserts the construction reaches `share`."""
    eps = E.scan(TCGEN05, dtype, dim, split, shadow)
    dev = c.deviation(dtype, split)
    assert dev <= eps, (what, dev, eps)
    if share is not None:
        assert dev >= share * eps, (what, dev / eps)
    if shadow and dtype == VM_BF16 and split:
        # the bound before the bf16 shadow's unit roundoff was corrected (2^-9): r* would fall below the decoys' band
        old = E.stored(TCGEN05, dtype, dim, split) + 2.0 ** -9 * 1.01
        assert dev > old + (c.s_target - c.s_decoys.min()), (what, dev, old)
    return dev / eps


CASES = [(kind, dim, mode) for dim in DIMS for mode in N for kind in KINDS]   # dim-major: the fillers are reused


@pytest.mark.parametrize("kind,dim,mode", CASES, ids=["-".join(map(str, c)) for c in CASES])
def test_row_at_the_error_bound_is_found(vm, E, kind, dim, mode):
    n = N[mode]
    c = _construction(kind, dim)
    X, target, decoys = _store_values(kind, dim, n, c)
    q = c.q.astype(np.float64 if kind.startswith("f64") else np.float32)
    ref = oracle.batch_similarities(q[None], X, max(KS))[0]
    assert ref[0][0] == target and {r for r, _ in ref[1:]} <= set(decoys.tolist())
    tc = kind in ("f64+bf16", "bf16") or dim <= TC_FP32_MAX_DIM
    st = vm.EmbeddingStore(dim, n, kind)
    try:
        st.append(X)
        for name, (vkind, dtype, flags, split, share) in VARIANTS.items():
            if vkind != kind:
                continue
            what = (name, dim, mode)
            if tc:
                print(what, "modelled deviation / eps = %.3f" % _model_share(E, c, dtype, dim, split, kind.startswith("f64"), share, what))
            for k in KS:
                st.counters(reset=True)
                _check(*_topk(vm, st, q, k, _flags(vm, flags)), ref[:k], what + (k,))
                s, cnt = st.last_stats, st.counters()
                assert cnt["bound_violations"] == 0, (what, k, cnt)
                if tc:
                    assert cnt["full_rescans"] == 0 and int(s.full_rescans) == 0, (what, k, cnt)
                    assert int(s.scan_kernel) == TCGEN05, (what, k)
                    assert int(s.scan_variant) == (1 if mode == "dump" else 2), (what, k, int(s.scan_variant))
                else:
                    # the tcgen05 scan cannot take these fp32 rows: this shape is left out of its cases
                    assert int(s.scan_kernel) == CUDA_CORE, (what, k)
        # the CUDA-core scan over the same store (its per-CTA lists bound the other rows only by their last key, so the
        # decoys send it to the fallbacks): parity only
        st.counters(reset=True)
        _check(*_topk(vm, st, q, 10, vm.VM_FLAG_FORCE_SIMT), ref[:10], (kind, dim, mode, "simt"))
        assert int(st.last_stats.scan_kernel) == CUDA_CORE and st.counters()["bound_violations"] == 0
    finally:
        st.close()


def test_pair_below_threshold_in_tf32_is_found(vm, E):
    """All-pairs scorer on fp32 rows: two rows truncated by almost 2^-10 on every element, whose reference score lies
    one fp32 step above the threshold and whose tf32 score lies about 2^-9 below it.  The epilogue's thr - eps filter must stage the
    pair and pairs_finalize_kernel must decide it in binary64: it is in the set."""
    import torch
    from vidmem_b200 import dedup
    dim, n = 384, 512
    B1 = np.ones(dim, np.float32)
    B2 = np.ones(dim, np.float32)
    B2[: dim // 5] = 0.0
    x1, x2 = ((b.view(np.uint32) | np.where(b != 0, np.uint32(0x1FFF), np.uint32(0))).view(np.float32) for b in (B1, B2))
    # the reference's score of the pair (rows normalised in fp32, binary64 dot, rounded to fp32), one fp32 step above thr
    _, _, s = oracle.pairs_above(np.stack([x1, x2]), 0.0)
    thr = float(np.nextafter(s[0], np.float32(0)))
    # the scorer's tf32 score of the pair (fp32 accumulation left out): truncated rows over the fp32 row norms
    inv = [np.float32(1 / np.sqrt(np.dot(x.astype(np.float64), x))) for x in (x1, x2)]
    tf32 = float(np.dot(tf32_trunc(x1).astype(np.float64), tf32_trunc(x2))) * float(inv[0]) * float(inv[1])
    eps = E.pairs(VM_F32, dim)
    assert thr - eps + 1e-4 < tf32 < thr - 1e-3, (tf32, thr, eps)
    X = np.random.default_rng(5).standard_normal((n, dim), dtype=np.float32)
    i1, i2 = 101, 400
    X[i1], X[i2] = x1, x2
    i, j, _ = dedup.pairs_above(torch.from_numpy(X).cuda(), thr)
    oi, oj, _ = oracle.pairs_above(X, thr)
    assert (i1, i2) in set(zip(oi.tolist(), oj.tolist()))
    assert set(zip(i.tolist(), j.tolist())) == set(zip(oi.tolist(), oj.tolist()))
