// scan_eps.h -- error bounds of the fast scans (DESIGN.md §2): for every row, |approximate cosine - exact cosine| <= eps,
// in cosine units (Cauchy-Schwarz).  Every exact answer rests on it: the top-k scan keeps keys >= L - 2 eps and the
// rescoring kernels certify a list once every key >= s_k - eps has been rescored, so a term that is too small drops a
// true top-k row without any counter noticing.  Kept in a header of plain host arithmetic so that the SAME code is
// compiled by tests/test_scan_eps_cpu.py, which checks it against bounds derived independently of it.
#pragma once
#include "../../include/vidmem.h"

namespace vm {

// Bound of a scan over the values the store holds.  kernel: 1 CUDA-core fp32 scan, 2 tcgen05 scan; split: bf16 store
// with the query fed as hi + lo bf16 terms.
inline double scan_eps_stored(int kernel, int store_dtype, int dim, int split)
{
    const double u = 1.1920928955078125e-07;                         // 2^-23
    const double fp32_acc = (double)(dim + 16) * u;                  // fp32 accumulation + normalisation of query and row
    if (kernel == 1) return fp32_acc;                                // CUDA-core fp32 scan
    if (store_dtype == VM_F32)                                       // tf32: rows truncated (2^-10), query pre-rounded to nearest (2^-11)
        return 9.765625e-4 + 4.8828125e-4 + 1e-6 + fp32_acc;
    if (!split) return 3.90625e-3 + fp32_acc;                        // bf16 store (exact operand), query rounded to bf16: 2^-8
    // bf16 store, query = hi + lo: residual 2^-16; the lo products are 2^-8 of the hi ones, their MMAs add one
    // accumulator rounding each (dim/16 of them) -- counted generously as dim/8 + 16 extra terms
    return 1.52587890625e-5 * 1.01 + (double)(dim + dim / 8 + 32) * u;
}

// shadow: the store keeps binary64 originals and the scan reads their rounded copy.  Rounding a row moves its
// direction by an angle of at most asin(u) (u = unit roundoff of the shadow type, relative per element, hence relative
// in norm), and a cosine moves by at most the angle.  fp32 shadow: u = 2^-24, taken as 2^-23.  bf16 shadow: u = 2^-8
// (8 significant bits); the shadow is rounded twice, binary64 -> fp32 -> bf16, so an element can move by 2^-8 + 2^-24
// of itself, taken as 1.01 * 2^-8.
inline double scan_eps(int kernel, int store_dtype, int dim, int split, bool shadow = false)
{
    const double base = scan_eps_stored(kernel, store_dtype, dim, split);
    if (!shadow) return base;
    return base + (store_dtype == VM_F32 ? 1.1920928955078125e-07 : 3.90625e-3 * 1.01);
}

// Bound of the all-pairs scorer (pairs.cu): pairs whose fp32 score lies within it of the threshold are re-decided in
// binary64.  tf32: both operands truncated twice over i and j.
inline float pairs_eps(int dtype, int dim)
{
    const float fp32_acc = (float)(dim + 32) * 1.1920928955078125e-07f;
    return dtype == VM_F32 ? 3.90625e-3f + fp32_acc : fp32_acc;
}

}  // namespace vm
