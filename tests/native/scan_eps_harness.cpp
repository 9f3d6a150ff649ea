// Host build of csrc/scan_eps.h for tests/test_scan_eps_cpu.py and tests/test_scan_bound_gpu.py: the error bounds the
// library scans with, evaluated by the same code.
#include "scan_eps.h"

extern "C" double eps_scan(int kernel, int store_dtype, int dim, int split, int shadow)
{
    return vm::scan_eps(kernel, store_dtype, dim, split, shadow != 0);
}

extern "C" double eps_scan_stored(int kernel, int store_dtype, int dim, int split)
{
    return vm::scan_eps_stored(kernel, store_dtype, dim, split);
}

extern "C" float eps_pairs(int dtype, int dim) { return vm::pairs_eps(dtype, dim); }
