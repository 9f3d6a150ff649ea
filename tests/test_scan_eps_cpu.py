"""The fast scans' error bound eps (csrc/scan_eps.h), compiled for the host with g++, against a bound derived here
from the unit roundoffs of the types involved (torch.finfo; tf32: truncation 2^-10, rounding 2^-11), for every scan,
store dtype, query form, shadow and dim the API accepts.  Every exact top-k answer rests on |s~ - s| <= eps for every
row: a term that is too small lets the scan drop a true top-k row below the band the rescoring certifies, and no
counter notices (the rescoring audits only the rows it rescored).  Also runs the host models of the adversarial
stores of test_scan_bound_gpu.py and checks that each deviation stays within its term and reaches the stated share of
eps (a store that does not come close to the bound would prove nothing on the GPU)."""
import pytest

from scan_eps_lib import (CUDA_CORE, TCGEN05, VM_BF16, VM_F32, Eps, accumulation, cosine, required, required_pairs,
                          rounding_construction, shadow_construction, shadow_term)

DIMS = range(1, 4097)
SCANS = [(CUDA_CORE, VM_F32, False), (CUDA_CORE, VM_BF16, False), (TCGEN05, VM_F32, False), (TCGEN05, VM_BF16, False),
         (TCGEN05, VM_BF16, True)]
SCAN_IDS = ["simt-f32", "simt-bf16", "tc-tf32", "tc-bf16", "tc-bf16-split"]
CONSTRUCTION_DIMS = (64, 384, 4096)


@pytest.fixture(scope="module")
def E(tmp_path_factory):
    return Eps(tmp_path_factory.mktemp("scan_eps"))


@pytest.mark.parametrize("shadow", [False, True], ids=["stored", "shadow"])
@pytest.mark.parametrize("kernel,dtype,split", SCANS, ids=SCAN_IDS)
def test_eps_covers_every_rounding(E, kernel, dtype, split, shadow):
    bad = [(d, E.scan(kernel, dtype, d, split, shadow), required(kernel, dtype, d, split, shadow)) for d in DIMS
           if not E.scan(kernel, dtype, d, split, shadow) >= required(kernel, dtype, d, split, shadow)]
    assert not bad, bad[:4]
    assert all(E.scan(kernel, dtype, d, split, False) == E.stored(kernel, dtype, d, split) for d in DIMS)


@pytest.mark.parametrize("kernel,dtype,split", SCANS, ids=SCAN_IDS)
def test_shadow_term_covers_its_rounding(E, kernel, dtype, split):
    """A bf16 shadow is binary64 -> fp32 -> bf16: 8 significant bits, rounded twice (2^-8 + 2^-24 of each element)."""
    for d in (1, 64, 384, 4096):
        term = E.scan(kernel, dtype, d, split, True) - E.scan(kernel, dtype, d, split, False)
        assert term >= shadow_term(dtype), (d, term, shadow_term(dtype))


@pytest.mark.parametrize("dtype", [VM_F32, VM_BF16], ids=["f32", "bf16"])
def test_pairs_eps_covers_every_rounding(E, dtype):
    bad = [(d, E.pairs(dtype, d), required_pairs(dtype, d)) for d in DIMS if not E.pairs(dtype, d) >= required_pairs(dtype, d)]
    assert not bad, bad[:4]


@pytest.mark.parametrize("dim", CONSTRUCTION_DIMS)
def test_bf16_shadow_construction(E, dim):
    """cos(q, r*) - cos(q, shadow of r*) is 2.757e-3 at every dim: more than 2^-9 (what a bf16 shadow with 7 significant
    bits would cost), within the shadow term.  With the split query the whole scan error reaches ~0.6-0.7 of eps."""
    c = shadow_construction(dim)
    shadow_dev = c.s_target - cosine(c.q, c.scan_target)
    assert 2.0 ** -9 * 1.01 < shadow_dev <= E.scan(TCGEN05, VM_BF16, dim, True, True) - E.stored(TCGEN05, VM_BF16, dim, True)
    for split in (True, False):
        eps = E.scan(TCGEN05, VM_BF16, dim, split, True)
        dev = c.deviation(VM_BF16, split)
        assert dev <= eps - accumulation(dim, split), (split, dev, eps)
    eps = E.scan(TCGEN05, VM_BF16, dim, True, True)
    assert c.deviation(VM_BF16, True) >= 0.6 * eps
    # the decoys sit between a few 1e-6 and 1e-4 below r*: far closer than the shadow's rounding
    gap = c.s_target - c.s_decoys
    assert (gap > 0).all() and gap.max() < 1e-4 and c.deviation(VM_BF16, True) > E.stored(TCGEN05, VM_BF16, dim, True) + 2.0 ** -9 * 1.01 + gap.max()


@pytest.mark.parametrize("dim", CONSTRUCTION_DIMS)
@pytest.mark.parametrize("dtype,exact", [(VM_F32, False), (VM_F32, True), (VM_BF16, False)], ids=["f32", "f64", "bf16"])
def test_rounding_construction(E, dim, dtype, exact):
    """tf32 scan (fp32 store, binary64 store with fp32 shadow): rows truncated by almost 2^-10 and query elements
    rounded down by almost 2^-11 take r*'s score down by >= 0.9 of eps where the tcgen05 scan serves the shape (up to
    2816-d fp32 rows), >= 0.6 from the rows alone.  bf16 store, single-term query: >= 0.8 of eps from the query."""
    c = rounding_construction(dim, dtype, exact)
    eps = E.scan(TCGEN05, dtype, dim, False, exact)
    dev = c.deviation(dtype)
    assert dev <= eps - accumulation(dim), (dev, eps)
    gap = c.s_target - c.s_decoys
    assert (gap >= 1e-5).all() and gap.max() < 5e-5
    if dtype == VM_F32:
        rows = c.deviation(dtype, round_query=False)
        assert rows <= 2.0 ** -10 + (shadow_term(VM_F32) if exact else 0.0)
        if dim <= 2816:
            assert dev >= 0.9 * eps and rows >= 0.6 * eps, (dev / eps, rows / eps)
    else:
        assert dev >= 0.8 * eps, dev / eps
