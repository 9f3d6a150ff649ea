// common.cuh -- shared device/host helpers for libvidmem (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include <utility>
#include "../../include/vidmem.h"

namespace vm {

// ---- error plumbing --------------------------------------------------------------------
void set_error(const char *fmt, ...);
#define VM_CUDA_CHECK(expr)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            vm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return VM_ERR_CUDA;                                                                  \
        }                                                                                        \
    } while (0)
#define VM_REQUIRE(cond, code, ...)          \
    do {                                     \
        if (!(cond)) {                       \
            vm::set_error(__VA_ARGS__);      \
            return (code);                   \
        }                                    \
    } while (0)

// ---- programmatic dependent launch (PDL) -----------------------------------------------
// The kernels of one top-k call are launched back to back with cudaLaunchAttributeProgrammaticStreamSerialization
// (launch_pdl below): kernel N+1 may be scheduled -- and run its prologue: shared-memory carve-up, barrier init,
// TMEM allocation, work that only depends on its own arguments -- while kernel N drains; pdl_wait() blocks until
// kernel N has COMPLETED and its writes are visible.  Every kernel of the chain calls pdl_wait() before it touches
// global memory another kernel of the chain writes or reads, so the chain is transitively ordered.  Without the
// launch attribute both instructions are no-ops.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                                     Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// Raises Kernel's dynamic shared-memory limit to `bytes` on the current device.  The attribute is per device; it is
// set on a device's first launch only, so later launches pay no driver call.
template <auto Kernel>
static inline cudaError_t max_smem_once(int bytes)
{
    static bool set[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess || set[dev & 63]) return e;
    e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) set[dev & 63] = true;
    return e;
}

// ---- candidate keys --------------------------------------------------------------------
// A candidate is one u64: high word = order-preserving image of the fp32 score, low word =
// ~row.  Larger key == better candidate (higher score, then LOWER row), keys are unique per
// row, and 0 is reserved for "empty slot" (every real score maps to a high word >= 0x007FFFFF).
__host__ __device__ __forceinline__ uint32_t f32_ordered(float f)
{
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(f);
#else
    uint32_t b;
    memcpy(&b, &f, 4);
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float f32_from_ordered(uint32_t o)
{
    uint32_t b = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f;
    memcpy(&f, &b, 4);
    return f;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(float score, uint32_t row)
{
    return ((uint64_t)f32_ordered(score) << 32) | (uint64_t)(0xFFFFFFFFu - row);
}
__host__ __device__ __forceinline__ uint32_t key_row(uint64_t k) { return 0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFu); }
__host__ __device__ __forceinline__ float key_score(uint64_t k) { return f32_from_ordered((uint32_t)(k >> 32)); }

static constexpr int SEED_TAB_WORDS = 256 * 64;  // scan table: per-CTA maxima [<= 256 CTAs][<= 64 queries]; [64] published bounds,
                                                 // [64] publication counter, [64] spill counters follow
#ifdef __CUDACC__
// k-th largest of the per-CTA maxima of query q (one warp, G <= 256 CTAs): a lower bound on the shard's k-th best
// score, because k distinct rows (one per CTA) reach it.  16 radix bits; truncation rounds down.
__device__ __forceinline__ float seed_select(const uint32_t *seed_tab, int G, int nq_pad, int q, int k, int lane)
{
    uint32_t vals[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int i = lane + 32 * t;
        vals[t] = i < G ? __ldcg(seed_tab + (size_t)i * nq_pad + q) : 0u;
    }
    uint32_t prefix = 0;
    int need = k;
    for (int bit = 31; bit >= 16; --bit) {
        const uint32_t hi = bit == 31 ? 0u : (0xFFFFFFFFu << (bit + 1));
        int cnt = 0;
#pragma unroll
        for (int t = 0; t < 8; ++t) cnt += ((vals[t] & hi) == prefix && ((vals[t] >> bit) & 1u)) ? 1 : 0;
        const int tot = __reduce_add_sync(0xffffffffu, cnt);
        if (tot >= need) prefix |= 1u << bit;
        else need -= tot;
    }
    float sd = f32_from_ordered(prefix);
    if (!(sd > -INFINITY) || G < k) sd = -INFINITY;  // also catches NaN patterns
    return sd;
}

// band threshold for a lower bound L on the k-th best approximate score: L - band, rounded DOWN (a lower threshold
// only keeps more rows)
__device__ __forceinline__ float band_floor(float L, float band)
{
    if (!(L > -INFINITY)) return -INFINITY;
    const float t = __fsub_rd(L, band);
    return nextafterf(t, -INFINITY);
}

#endif

// ---- binary64 reference arithmetic -----------------------------------------------------
// Python's builtin sum() over float products (see oracle/vm_oracle.c): the first item enters
// through 0.0 + x, the rest through a naive or Neumaier recurrence.  Explicit _rn intrinsics
// keep nvcc from contracting mul+add into FMA, so every step rounds like CPython's doubles.
struct RefSum {
    double s, c;
    __device__ __forceinline__ void init() { s = 0.0; c = 0.0; }
    // Branch-free: with s = c = 0 the general step reproduces CPython's first step (0.0 + x)
    // exactly, so no "first item" case is needed; selects instead of an if keep the loop
    // unrollable and the loads pipelined.
    template <bool NEUMAIER>
    __device__ __forceinline__ void add(double x)
    {
        double t = __dadd_rn(s, x);
        if (NEUMAIER) {
            const bool big = fabs(s) >= fabs(x);
            const double hi = big ? s : x, lo = big ? x : s;
            c = __dadd_rn(c, __dadd_rn(__dadd_rn(hi, -t), lo));
        }
        s = t;
    }
    // Eight consecutive items at once.  Exactly the same operations in the same order as eight add()
    // calls, but laid out so the three dependency chains are visible to the scheduler: the running
    // sums t[u] (8 dependent DADDs, 8.2 cycles each on sm_100), the per-item error terms (independent
    // of each other) and the compensation chain, which overlaps the next block's running sums.
    // Measured: ~11 cycles/item instead of 34 for the item-at-a-time loop.
    template <bool NEUMAIER>
    __device__ __forceinline__ void add_block(const double (&x)[8])
    {
        double t[8];
        t[0] = __dadd_rn(s, x[0]);
#pragma unroll
        for (int u = 1; u < 8; ++u) t[u] = __dadd_rn(t[u - 1], x[u]);
        if (NEUMAIER) {
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const double prev = u ? t[u - 1] : s;
                const bool big = fabs(prev) >= fabs(x[u]);
                const double hi = big ? prev : x[u], lo = big ? x[u] : prev;
                c = __dadd_rn(c, __dadd_rn(__dadd_rn(hi, -t[u]), lo));
            }
        }
        s = t[7];
    }
    template <bool NEUMAIER>
    __device__ __forceinline__ double result() const
    {
        double r = s;
        if (NEUMAIER && c != 0.0 && isfinite(c)) r = __dadd_rn(r, c);
        return r;
    }
};

// acc += sum over i in [lo, hi) of prod(i), in index order (blocks of 8 + tail)
template <bool NEUMAIER, typename F>
__device__ __forceinline__ void ref_sum_range(RefSum &acc, int lo, int hi, F prod)
{
    int i = lo;
    for (; i + 8 <= hi; i += 8) {
        double x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) x[u] = prod(i + u);
        acc.add_block<NEUMAIER>(x);
    }
    for (; i < hi; ++i) acc.add<NEUMAIER>(prod(i));
}

__device__ __forceinline__ float load_as_float(const float *p, int64_t i) { return p[i]; }
__device__ __forceinline__ float load_as_float(const __nv_bfloat16 *p, int64_t i) { return __bfloat162float(p[i]); }
// one row element as a double (exact widening), by the row's storage type
__device__ __forceinline__ double load_elem(const float *p, int64_t i) { return (double)p[i]; }
__device__ __forceinline__ double load_elem(const __nv_bfloat16 *p, int64_t i) { return (double)__bfloat162float(p[i]); }
__device__ __forceinline__ double load_elem(const double *p, int64_t i) { return p[i]; }
__device__ __forceinline__ double load_as_double(const void *p, int dtype, int64_t i)
{
    if (dtype == VM_F32) return (double)((const float *)p)[i];
    if (dtype == VM_BF16) return (double)__bfloat162float(((const __nv_bfloat16 *)p)[i]);
    return ((const double *)p)[i];
}

static inline int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }
static inline int ld_for_dim(int dim) { return (dim + 7) & ~7; }
static inline size_t dtype_size(int dt) { return dt == VM_F32 ? 4 : dt == VM_BF16 ? 2 : 8; }

// ---- kernel launch interfaces (defined in the .cu files) -------------------------------
struct ScanArgs {
    const void *rows;        // [n][ld] store dtype
    const float *inv_norms;  // [n] 1/||row||; 0 = zero-norm row (scores 0.0), < 0 = skipped row (never returned)
    int dtype;               // store dtype
    int64_t n;
    int dim, ld;
    const float *queries;    // [nq_pad][ld] fp32, L2-normalised (zero query stays zero), device
    int nq;                  // queries in this launch
    int kp;                  // candidate list length per query (<= 64)
    uint64_t *cand;          // [ctas][nq][kp] keys out
    int ctas;                // number of CTAs to launch (lists produced)
    cudaStream_t stream;
    int dump = 0;            // tcgen05 scan only: small store -- emit EVERY row's key, cand = [tiles][nq][128] (see scan_tc.cu)
    // tcgen05 scan, band scheme (scan_tc.cu): every key with approximate score >= (bound on the k-th best) - band
    uint64_t *slab = nullptr;  // [ctas][nq][SCAN_SLAB] per-CTA append buffers
    int *scnt = nullptr;       // [ctas][nq] keys appended per slab (> SCAN_SLAB: the rest was spilled)
    uint64_t *ubuf = nullptr;  // [nq][ucap] shared spill buffer
    int *ucnt = nullptr;       // [nq] keys spilled, zeroed before the launch (> ucap: overflow)
    int ucap = 0;
    float band = 0.0f;         // 2 eps, rounded up
    int ksel = 0;              // k
    int split = 0;             // bf16 store: queries given as hi + lo bf16 terms, [2][nq_pad][ld]
    bool pdl = false;          // launch with programmatic stream serialization
};
static constexpr int SCAN_UNION_CAP = 16384; // shared spill-buffer entries per query (filtered with the final bound before staging)
static constexpr int SCAN_SLAB = 128;         // keys per (CTA, query) slab
static constexpr int SELECT_KEY_CAP = 4096;   // band keys the rescoring kernel stages per query after the final filter
static constexpr int SCAN_DUMP_TILE = 128;     // rows (= keys per query) per dumped tile
static constexpr int SCAN_DUMP_MAX_KEYS = 9472;  // per query: what the fused select kernel ranks in shared memory (148 x 64)
int launch_scan_simt(const ScanArgs &a);
int scan_simt_max_queries();
// second pass of the tcgen05 scan for uncertified queries (see scan_tc.cu "collect mode")
struct ScanCollect {
    const float *thr;    // [nq] thresholds written by the rescoring kernel (+inf = query is done)
    uint64_t *buf;       // [nq][cap]
    int *cnt;            // [nq], zeroed before the launch
    int cap;
    const int *pending;  // uncertified-query counter
};
// tcgen05 path; seed_tab [ctas][nq_pad] u32 + seed_ctr must be zeroed before the launch (NULL = no seeding);
// sc != NULL runs the collect pass instead of the top-kp pass
struct ScanInfo { int stages = 0, variant = 0; };  // what the launch chose (reported in vm_topk_stats): pipeline depth; 0 lists, 1 dump, 2 lists + threshold warp
int launch_scan_tc(const ScanArgs &a, const void *queries_store_dtype, uint32_t *seed_tab, int *seed_ctr,
                   const ScanCollect *sc = nullptr, ScanInfo *info = nullptr);
bool scan_tc_supported(int dtype, int dim, int nq, int kp, int split = 0);


// ---- argument blocks shared by api.cu and select.cu ------------------------------------
struct FinalizeArgs {
    int k;
    double min_score;
    int score_mode;
    int64_t row_offset;  // added to local rows in the output (sharded stores)
    int64_t *out_idx;    // [nq][k]
    double *out_score;   // [nq][k]
    int32_t *out_count;  // [nq]
};
struct RescoreArgs {
    const uint64_t *merged;
    int kp;
    const void *rows;
    const float *inv_norms;
    int dtype, ld, dim;
    int64_t n_rows;
    const void *queries;
    int q_dtype, nq;
    double eps;
    int sum_mode;
    FinalizeArgs fin;
    int32_t *flags, *uncertified_count;
    const int *extreme;  // store-level count of rows outside the scans' numeric range (forces the exact pass)
    float *collect_thr;  // [nq] out: threshold of the collect pass for uncertified queries (+inf otherwise); may be NULL
    unsigned long long *cum = nullptr;  // store-lifetime counters (vm_store_read_counters): [0] uncertified, [1] settled from the
                                        // band, [2] settled by the collect pass, [3] redone by the binary64 scan of every row, [4] error-bound violations
};
// where the fused select + rescore kernel takes a query's candidate keys from
struct SelectArgs {
    const uint64_t *cand = nullptr;  // list mode: [lists][nq][list_len] (CUDA-core scan lists, or dumped tiles)
    int lists = 0, list_len = 0;
    int complete = 0;                // list mode: the lists hold EVERY row of the shard (dump mode)
    // slab mode (tcgen05 scan): per-CTA slabs + shared spill buffer + the table of per-CTA maxima / published bounds
    const uint64_t *slab = nullptr;  // [ctas][nq][SCAN_SLAB]
    const int *scnt = nullptr;       // [ctas][nq]
    int ctas = 0;
    const uint64_t *ubuf = nullptr;  // [nq][ucap]
    const int *ucnt = nullptr;
    int ucap = 0;
    const uint32_t *seed_tab = nullptr;  // [ctas][nq_pad] final per-CTA maxima, then [64] published bounds (may be NULL)
    int nq_pad = 0, ksel = 0;
    float band = 0.0f;
};
struct ExactArgs {
    const void *rows;
    const float *inv_norms;
    int dtype, ld, dim;
    int64_t n;
    const void *queries;
    int q_dtype, nq, k, sum_mode;
    int32_t *flags;        // NULL = all queries
    double *xlist_score;   // [ctas][nq][k]
    uint32_t *xlist_row;
    int32_t *xlist_cnt;    // [ctas][nq]
    uint8_t *taken;        // [nq][ctas*k]
    int ctas;
    FinalizeArgs fin;
    unsigned long long *cum = nullptr;  // see RescoreArgs::cum
    int *done_ctr = nullptr;            // conditional form: ticket counter (zero between calls) -> in-kernel merge by the last CTA
};

}  // namespace vm
