"""The scans' error bound eps (csrc/scan_eps.h, host build through tests/native/scan_eps_harness.cpp), a bound derived
independently of it, and host models of the stores that push a row's approximate score as far below its exact score
as each scan allows.  Used by test_scan_eps_cpu.py, which checks eps against the independent bound and the models, and
by test_scan_bound_gpu.py, which builds the stores.

The fast scans compute s~ = (q' . x') * inv, where q' is the normalised query as the scan feeds it (rounded to tf32 /
bf16, or bf16 hi + lo terms), x' the row as the tensor core reads it (fp32 truncated to tf32, bf16 as stored, or the
rounded shadow of a binary64 row) and inv the row's cached fp32 inverse norm.  The models below reproduce those
roundings exactly and leave out only the fp32 accumulation, which the accumulation term of eps covers."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "real-time-brain-inspired-video-memory_b200", "csrc")

VM_F32, VM_BF16 = 0, 1
CUDA_CORE, TCGEN05 = 1, 2                                  # scan kernels (vm_topk_stats.scan_kernel)

U_BF16 = float(torch.finfo(torch.bfloat16).eps) / 2        # unit roundoff: 2^-8 (8 significant bits)
U_F32 = float(torch.finfo(torch.float32).eps) / 2          # 2^-24
TF32_TRUNC = 2.0 ** -10                                     # fp32 operand truncated to tf32 by the tensor core
TF32_ROUND = 2.0 ** -11                                     # fp32 query rounded to nearest tf32 before the scan


class Eps:
    """eps as the library computes it."""

    def __init__(self, out_dir):
        so = os.path.join(str(out_dir), "libscan_eps.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                               os.path.join(ROOT, "tests", "native", "scan_eps_harness.cpp"), "-o", so])
        L = C.CDLL(so)
        L.eps_scan.argtypes = [C.c_int] * 5
        L.eps_scan.restype = C.c_double
        L.eps_scan_stored.argtypes = [C.c_int] * 4
        L.eps_scan_stored.restype = C.c_double
        L.eps_pairs.argtypes = [C.c_int] * 2
        L.eps_pairs.restype = C.c_float
        self.L = L

    def scan(self, kernel, dtype, dim, split=False, shadow=False):
        return self.L.eps_scan(kernel, dtype, dim, int(split), int(shadow))

    def stored(self, kernel, dtype, dim, split=False):
        return self.L.eps_scan_stored(kernel, dtype, dim, int(split))

    def pairs(self, dtype, dim):
        return self.L.eps_pairs(dtype, dim)


# ---- the independent bound ------------------------------------------------------------------------------------------
def accumulation(dim, split=False):
    """fp32 accumulation of the dot product and the normalisations of query and row; the split query's lo MMAs add
    one accumulator rounding per 16-column slice (counted as dim/8 + 16 extra terms).  Same form as the library's."""
    return (dim + dim // 8 + 32 if split else dim + 16) * 2 * U_F32


def shadow_term(dtype):
    """A binary64 row is rounded to its shadow: to nearest fp32 (u = 2^-24); to bf16 through fp32, twice (2^-8 + 2^-24)."""
    return U_F32 if dtype == VM_F32 else U_BF16 + U_F32


def required(kernel, dtype, dim, split=False, shadow=False):
    """Smallest eps the roundings of each scan allow, by Cauchy-Schwarz (every term is relative per element of one
    operand, hence relative in norm, and a unit query times a unit row moves by at most that much)."""
    if kernel == CUDA_CORE:
        r = accumulation(dim)
    elif dtype == VM_F32:
        r = TF32_TRUNC + TF32_ROUND + accumulation(dim)
    elif not split:
        r = U_BF16 + accumulation(dim)
    else:
        r = U_BF16 * U_BF16 + accumulation(dim, True)       # residual of hi + lo: 2^-8 of 2^-8
    return r + (shadow_term(dtype) if shadow else 0.0)


def required_pairs(dtype, dim):
    """All-pairs scorer: both rows truncated to tf32 (fp32 rows), bf16 rows exact; accumulation over dim + 32 terms."""
    return (2 * TF32_TRUNC if dtype == VM_F32 else 0.0) + (dim + 32) * 2 * U_F32


# ---- roundings, as the kernels do them ------------------------------------------------------------------------------
def _bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def tf32_round(v):
    """normalize_queries_kernel's tf32 rounding of the fp32 query (to nearest, ties away)."""
    return ((_bits(v) + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def tf32_trunc(x):
    """The tensor core's reading of an fp32 operand as tf32 (low 13 mantissa bits dropped)."""
    return (_bits(x) & np.uint32(0xFFFFE000)).view(np.float32)


def to_bf16(x):
    """fp32 -> bf16 -> fp32, round to nearest even (__float2bfloat16_rn)."""
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).float().numpy()


def bf16_shadow(x64):
    """convert_rows_kernel's bf16 copy of binary64 rows: binary64 -> fp32 -> bf16, each to nearest."""
    return to_bf16(np.asarray(x64, np.float64).astype(np.float32))


def normalize(q):
    """normalize_queries_kernel for one query whose squares sum exactly (so the warp's summation order does not
    matter): v = fp32(q * (1 / sqrt(sum q^2))), in binary64 up to the last rounding."""
    q = np.asarray(q, np.float64)
    assert np.array_equal(q, np.round(q)) and np.abs(q).max() < 2.0 ** 24    # integers: exact squares, exact in fp32
    sq = q * q
    ss = float(np.sum(sq))
    assert ss == math.fsum(sq.tolist())
    return (q * (1.0 / math.sqrt(ss))).astype(np.float32)


def scan_query(q, dtype, split):
    """The query as the tcgen05 scan multiplies it: tf32-rounded (fp32 store) or bf16 (hi, + lo when split)."""
    v = normalize(q)
    if dtype == VM_F32:
        return tf32_round(v).astype(np.float64)
    hi = to_bf16(v)
    return hi.astype(np.float64) + (to_bf16(v - hi).astype(np.float64) if split else 0.0)


def scan_row(x, dtype):
    """(row as the tensor core reads it, its cached fp32 inverse norm) for a row stored as `x` (fp32 or bf16 values)."""
    x = np.asarray(x, np.float32)
    inv = np.float32(1.0 / math.sqrt(float(np.sum(x.astype(np.float64) ** 2))))
    xe = tf32_trunc(x) if dtype == VM_F32 else x
    return xe.astype(np.float64), float(inv)


def cosine(q, x):
    q, x = np.asarray(q, np.float64), np.asarray(x, np.float64)
    return math.fsum((q * x).tolist()) / (math.sqrt(math.fsum((q * q).tolist())) * math.sqrt(math.fsum((x * x).tolist())))


def model_score(q, x_scan, dtype, split=False, round_query=True):
    """s~ of the tcgen05 scan without its fp32 accumulation.  x_scan: what the scan streams (the row itself, or the
    shadow of a binary64 row).  round_query=False: the query's own rounding left out (rows alone)."""
    qe = scan_query(q, dtype, split) if round_query else normalize(q).astype(np.float64)
    xe, inv = scan_row(x_scan, dtype)
    return math.fsum((qe * xe).tolist()) * inv


# ---- adversarial stores ----------------------------------------------------------------------------------------------
N_DECOYS = 48     # >= kp + 8 for k <= 16 (kp = 32)
GAP = 1e-5        # decoys sit at least this far below the target row's exact score (and within a few 1e-5)


class Construction:
    """One target row r* whose scanned score falls as far below its exact score as the scan's roundings allow, and
    N_DECOYS decoy rows whose exact scores sit a few 1e-5 below r*'s and whose values the scan reads exactly.
    q: the raw query (exact sum of squares).  target / decoys: the values the store is given (fp32-exact, or binary64
    for a binary64 store).  scan_target: what the scan streams of r* (its shadow, for a binary64 store)."""

    def __init__(self, q, target, scan_target, decoys):
        self.q, self.target, self.scan_target, self.decoys = q, target, scan_target, decoys
        self.s_target = cosine(q, target)
        self.s_decoys = np.array([cosine(q, d) for d in decoys])

    def deviation(self, dtype, split=False, round_query=True):
        """s* - s~*: how far below its exact score the scan puts r*."""
        return self.s_target - model_score(self.q, self.scan_target, dtype, split, round_query)


def shadow_construction(dim):
    """bf16 shadow of a binary64 store: r* is 1 + 2^-8 + 2^-22 on the first half of the columns (rounds up to
    1 + 2^-7) and 1 + 2^-8 - 2^-22 on the second half (rounds down to 1); the query is 1 on the second half.
    Decoys: all-ones rows with m columns of the first half at 1 + 2^-7 (bf16-exact), m the fewest that put them GAP
    below r*.  The shadow's rounding alone takes cos(q, r*) down by 2.757e-3 at every dim."""
    h = dim // 2
    q = np.r_[np.zeros(h), np.ones(dim - h)]
    target = np.r_[np.full(h, 1 + 2.0 ** -8 + 2.0 ** -22), np.full(dim - h, 1 + 2.0 ** -8 - 2.0 ** -22)]
    s_t = cosine(q, target)
    for m in range(1, h + 1):
        d = np.ones(dim)
        d[:m] = 1 + 2.0 ** -7
        if s_t - cosine(q, d) >= GAP:
            break
    decoys = []
    for j in range(N_DECOYS):
        d = np.ones(dim)
        d[(j * m + np.arange(m)) % h] = 1 + 2.0 ** -7
        decoys.append(d)
    return Construction(q, target, bf16_shadow(target), decoys)


def _just_below_midpoint_query(dim, mid_bits):
    """A raw query (integers, exact sum of squares) whose normalised elements on all but one column lie just below a
    rounding midpoint of the scanned query type (mid_bits: 0x1000 tf32, 0x8000 bf16), at the bottom of their binade,
    so that rounding to nearest takes almost half an ulp -- 2^-11 (tf32) or 2^-8 (bf16) of each -- off them.
    Layout: a on columns [0, dim - 1 - p), a / 2 on [dim - 1 - p, dim - 1), c on column dim - 1; the normalised
    a-columns land at 2^e (1 + mid - 2^-22) when a^2 ((dim - 1 - p) + p / 4) + c^2 = (a / that)^2, and c tunes it.
    -> (q, p, c / a)."""
    a = 2.0 ** 20
    mid = mid_bits * 2.0 ** -23                             # relative position of the midpoint in the binade
    P = 4 ** int(math.floor(math.log(dim + 3, 4)))          # 1 / (2^e)^2: the binade of the a-columns
    if P * (1 - 2 * mid) < dim / 4 + 1:
        P //= 4
    p = max(0, math.floor((dim - 1 - P * (1 - 2 * mid)) * 4 / 3) + 1)
    assert p <= dim - 2, dim
    target = (1 + mid - 2.0 ** -22) / math.sqrt(P)
    c0 = math.sqrt(max(0.0, (a / target) ** 2 - (dim - 1 - p) * a * a - p * a * a / 4))
    mask = np.uint32(2 * mid_bits - 1)
    best = None
    for c in range(max(0, int(c0) - 64), int(c0) + 64):
        q = np.r_[np.full(dim - 1 - p, a), np.full(p, a / 2), [float(c)]]
        low = int(_bits(normalize(q)[:1])[0] & mask)
        if low < mid_bits and (best is None or low > best[0]):
            best = (low, q, c)
    assert best is not None and best[0] >= mid_bits - 8, (dim, best and best[0])
    return best[1], p, best[2] / a


def rounding_construction(dim, dtype, exact=False):
    """fp32 store (tf32 scan), binary64 store with an fp32 shadow (exact=True), or bf16 store (single-term query).
    Query: _just_below_midpoint_query.  Base row B, exact in the scanned type: 1 on the a-columns, 1/2 on the a/2
    columns, about c/a on the last.  r*: B with the low 13 mantissa bits set (fp32 and binary64 stores: truncated by
    almost 2^-10 of itself) or B itself (bf16 store: the query's rounding alone); for the binary64 store the original
    also sits just below half an fp32 ulp above that (its shadow rounds down by almost 2^-24 more).  Decoys: B with one
    a-column lowered by t grid steps, t the fewest that put them GAP below r*."""
    q, p, ca = _just_below_midpoint_query(dim, 0x1000 if dtype == VM_F32 else 0x8000)
    grid = to_bf16 if dtype == VM_BF16 else tf32_trunc
    na = dim - 1 - p
    B = np.r_[np.ones(na), np.full(p, 0.5), grid(np.float32([ca]))].astype(np.float32)
    if dtype == VM_BF16:
        target = scan = B.astype(np.float64)
    else:
        scan = (_bits(B) | np.where(B != 0, np.uint32(0x1FFF), np.uint32(0))).view(np.float32)
        target = scan.astype(np.float64)
        if exact:                                            # just under half an fp32 ulp above its shadow
            ulp = np.spacing(scan).astype(np.float64)
            target = target + ulp * (0.5 - 2.0 ** -16)
            assert np.array_equal(target.astype(np.float32), scan)
    s_t = cosine(q, target)
    step = 2.0 ** -8 if dtype == VM_BF16 else 2.0 ** -11     # grid step of values in [1/2, 1)
    for t in range(1, int(0.5 / step) + 1):
        d = B.copy()
        d[0] = 1 - t * step
        if s_t - cosine(q, d) >= GAP:
            break
    decoys = []
    for j in range(N_DECOYS):
        d = B.astype(np.float64)
        d[j % na] = 1 - t * step
        decoys.append(d)
    return Construction(q, target, scan, decoys)
