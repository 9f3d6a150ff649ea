// select.cu -- everything after the streaming scan: candidate merge, binary64 rescoring in the
// reference's summation order + certification, the always-exact binary64 scan used for
// uncertified queries, the cross-shard merge and the cross-query max-by-id merge.
#include "common.cuh"

#include <type_traits>

namespace vm {

// =========================================================================================
// 1. merge per-CTA candidate sets -> the kp best keys per query
// =========================================================================================
// cand [lists][nq][kp] -> merged [nq][kp]: the kp largest keys in ARBITRARY order except that
// slot kp-1 holds the smallest of them (the "worst candidate" the certification needs); unused
// slots are 0.  One CTA per query.  Keys are unique, so an MSB-first radix select (8 passes of
// 8 bits, shared-memory histogram + one warp scanning the 256 bins) yields the exact kp-th
// largest key T; every key >= T is then emitted.  O(n) work instead of kp block-wide arg-max
// rounds.
static constexpr int MERGE_THREADS = 512;
static constexpr int MERGE_SURV = 1024;  // survivors ranked directly

// Exact kp-th largest key of skeys[0..total) by MSB-first radix select (8 passes x 8 bits).
// Block-wide; returns the same value in every thread.  Used when the cheap bound below does not
// thin the keys enough (heavily duplicated scores).
__device__ uint64_t radix_select_kth(const uint64_t *skeys, int total, int kp, int *hist, int *s_bin, int *s_need)
{
    const int tid = threadIdx.x, lane = tid & 31;
    uint64_t prefix = 0;
    int need = kp;
    for (int pass = 0; pass < 8; ++pass) {
        const int shift = 56 - 8 * pass;
        const uint64_t hmask = pass == 0 ? 0ull : (~0ull << (shift + 8));
        if (tid < 256) hist[tid] = 0;
        __syncthreads();
        for (int e = tid; e < total; e += MERGE_THREADS) {
            const uint64_t k = skeys[e];
            const bool act = k != 0 && (k & hmask) == prefix;
            const int bin = act ? (int)((k >> shift) & 0xFF) : -1;
            const unsigned peers = __match_any_sync(__activemask(), bin);
            if (act && (__ffs(peers) - 1) == lane) atomicAdd(&hist[bin], __popc(peers));
        }
        __syncthreads();
        if (tid < 32) {
            int mine[8], sum = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) { mine[i] = hist[255 - (8 * lane + i)]; sum += mine[i]; }
            int incl = sum;
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            int excl = incl - sum;
            if (excl < need && need <= incl) {
                int acc = excl;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    if (acc < need && need <= acc + mine[i]) { *s_bin = 255 - (8 * lane + i); *s_need = need - acc; }
                    acc += mine[i];
                }
            }
        }
        __syncthreads();
        prefix |= (uint64_t)(*s_bin) << shift;
        need = *s_need;
        __syncthreads();
    }
    return prefix;
}

// One CTA per query.
//  1. every list's maximum score is found by one warp (32-bit REDUX); the kp-th largest of those
//     maxima, L, is a lower bound on the kp-th largest key (kp different lists reach it);
//  2. keys with score >= L ("survivors", typically ~kp..2kp of the lists*kp keys) are compacted;
//  3. survivors are ranked against each other and written in descending order, so slot kp-1 is
//     the worst candidate the certification needs.
// Falls back to the exact radix select when fewer than kp lists are populated or more than
// MERGE_SURV keys survive.
__global__ void __launch_bounds__(MERGE_THREADS) merge_candidates_kernel(const uint64_t *__restrict__ cand, int lists, int nq,
                                                                       int kp, uint64_t *__restrict__ merged)
{
    extern __shared__ uint64_t skeys[];  // [lists*kp] then [lists] list maxima (u32)
    __shared__ uint64_t surv[MERGE_SURV];
    __shared__ int hist[256];
    __shared__ int s_bin, s_need, s_m, s_nz;
    __shared__ uint32_t s_L;
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int total = lists * kp;
    uint32_t *lmax = reinterpret_cast<uint32_t *>(skeys + total);
    if (tid == 0) { s_m = 0; s_nz = 0; }
    __syncthreads();
    int nz = 0;
#pragma unroll 4
    for (int e = tid; e < total; e += MERGE_THREADS) {
        int l = e / kp, j = e - l * kp;
        uint64_t k = cand[((int64_t)l * nq + q) * kp + j];
        skeys[e] = k;
        nz += k != 0;
    }
    if (nz) atomicAdd(&s_nz, nz);
    __syncthreads();
    const int nonzero = s_nz;
    uint64_t T = 1;  // smallest real key is > 0: T = 1 selects every non-empty slot
    bool ranked_path = false;
    if (nonzero >= kp) {
        if (lists >= kp) {
            // 1. per-list maximum score (high word of the key)
            for (int l = warp; l < lists; l += MERGE_THREADS / 32) {
                uint32_t m = 0;
                for (int j = lane; j < kp; j += 32) m = max(m, (uint32_t)(skeys[l * kp + j] >> 32));
                m = __reduce_max_sync(0xffffffffu, m);
                if (lane == 0) lmax[l] = m;
            }
            __syncthreads();
            if (warp == 0) {
                // kp-th largest of the list maxima: bitwise radix select with warp reductions
                uint32_t prefix = 0;
                int need = kp;
                for (int bit = 31; bit >= 0; --bit) {
                    const uint32_t hi = bit == 31 ? 0u : (0xFFFFFFFFu << (bit + 1));
                    int cnt = 0;
                    for (int l = lane; l < lists; l += 32) cnt += ((lmax[l] & hi) == prefix && ((lmax[l] >> bit) & 1u)) ? 1 : 0;
                    const int tot = __reduce_add_sync(0xffffffffu, cnt);
                    if (tot >= need) prefix |= 1u << bit;
                    else need -= tot;
                }
                if (lane == 0) s_L = prefix;
            }
            __syncthreads();
            const uint32_t Lb = s_L;
            if (Lb != 0) {
                // 2. compact the survivors
                for (int e = tid; e < total; e += MERGE_THREADS) {
                    const uint64_t k = skeys[e];
                    if ((uint32_t)(k >> 32) >= Lb && k != 0) {
                        const int p = atomicAdd(&s_m, 1);
                        if (p < MERGE_SURV) surv[p] = k;
                    }
                }
                __syncthreads();
                const int m = s_m;
                if (m >= kp && m <= MERGE_SURV) {
                    // 3. rank survivors (keys are unique) and emit the kp largest in descending order
                    for (int e = tid; e < m; e += MERGE_THREADS) {
                        const uint64_t k = surv[e];
                        int rank = 0;
                        for (int i = 0; i < m; ++i) rank += surv[i] > k ? 1 : 0;
                        if (rank < kp) merged[(int64_t)q * kp + rank] = k;
                    }
                    ranked_path = true;
                }
            }
        }
        if (!ranked_path) {
            __syncthreads();
            T = radix_select_kth(skeys, total, kp, hist, &s_bin, &s_need);
        }
    }
    if (ranked_path) return;  // uniform across the block
    if (tid == 0) s_m = 0;
    __syncthreads();
    for (int e = tid; e < total; e += MERGE_THREADS) {
        const uint64_t k = skeys[e];
        if (k >= T && k != 0) {
            if (nonzero >= kp && k == T) merged[(int64_t)q * kp + kp - 1] = k;  // the worst candidate
            else merged[(int64_t)q * kp + atomicAdd(&s_m, 1)] = k;
        }
    }
    __syncthreads();
    const int filled = s_m;
    const int last = nonzero >= kp ? kp - 1 : kp;
    for (int e = filled + tid; e < last; e += MERGE_THREADS) merged[(int64_t)q * kp + e] = 0;
}

// =========================================================================================
// 2. exact binary64 rescoring + sort + certification
// =========================================================================================

__device__ __forceinline__ double convert_score(double c, int score_mode)
{
    return score_mode == VM_SCORE_NEO4J ? __ddiv_rn(__dadd_rn(1.0, c), 2.0) : c;
}

// Reference cosine on (query, row): pre_llm_injector.py:374-388 in binary64, products and sums
// in index order.  Rows are read with their stored dtype; `dim` real columns only.
template <bool NEUMAIER, typename T>
__device__ double exact_cosine(const void *q, int q_dtype, int64_t qoff, const T *row, int dim)
{
    RefSum dot, qq, rr;
    dot.init(); qq.init(); rr.init();
    for (int i = 0; i < dim; ++i) {
        double x = load_as_double(q, q_dtype, qoff + i);
        double y = load_elem(row, i);
        dot.add<NEUMAIER>(__dmul_rn(x, y));
        qq.add<NEUMAIER>(__dmul_rn(x, x));
        rr.add<NEUMAIER>(__dmul_rn(y, y));
    }
    double n1 = __dsqrt_rn(qq.result<NEUMAIER>());
    double n2 = __dsqrt_rn(rr.result<NEUMAIER>());
    if (n1 == 0.0 || n2 == 0.0) return 0.0;
    return __ddiv_rn(dot.result<NEUMAIER>(), __dmul_rn(n1, n2));
}

// Same, with the query already staged as doubles in shared memory.
template <bool NEUMAIER, typename T>
__device__ double exact_cosine_sq(const double *sq, double n1, const T *row, int dim)
{
    RefSum dot, rr;
    dot.init(); rr.init();
    ref_sum_range<NEUMAIER>(dot, 0, dim, [&](int i) { return __dmul_rn(sq[i], load_elem(row, i)); });
    ref_sum_range<NEUMAIER>(rr, 0, dim, [&](int i) { const double y = load_elem(row, i); return __dmul_rn(y, y); });
    double n2 = __dsqrt_rn(rr.result<NEUMAIER>());
    if (n1 == 0.0 || n2 == 0.0) return 0.0;
    return __ddiv_rn(dot.result<NEUMAIER>(), __dmul_rn(n1, n2));
}

// (score desc, row asc) strict order
__device__ __forceinline__ bool better(double sa, uint32_t ra, double sb, uint32_t rb)
{
    return sa > sb || (sa == sb && ra < rb);
}

// One CTA per query.  The reference formula needs three sequential binary64 sums per
// (query, candidate): dot, ||q||^2 and ||row||^2.  Each is an independent chain, so they are
// spread over threads as TASKS -- task t < kp: dot of candidate t; kp <= t < 2kp: ||row||^2 of
// candidate t-kp; t == 2kp: ||q||^2 -- and every chain runs in index order (bit-identical to
// CPython).  Query and candidate rows are staged through shared memory as doubles in column
// chunks (coalesced loads; odd row pitch -> conflict-free per-thread walks).
// eps: bound on |approximate cosine - exact cosine| of the scan that produced the candidates.
static constexpr int RS_THREADS = 256;  // >= 2*64 + 1 tasks; the extra threads help staging
static constexpr int RS_SMEM_ROW_BYTES = 96 * 1024;

// 16-byte global load of 4 (fp32) / 8 (bf16) consecutive row elements -> floats
__device__ __forceinline__ void load_vec16(const float *p, float *o)
{
    const float4 t = *reinterpret_cast<const float4 *>(p);
    o[0] = t.x; o[1] = t.y; o[2] = t.z; o[3] = t.w;
}
__device__ __forceinline__ void load_vec16(const __nv_bfloat16 *p, float *o)
{
    const uint4 u = *reinterpret_cast<const uint4 *>(p);
    o[0] = __uint_as_float(u.x << 16); o[1] = __uint_as_float(u.x & 0xffff0000u);
    o[2] = __uint_as_float(u.y << 16); o[3] = __uint_as_float(u.y & 0xffff0000u);
    o[4] = __uint_as_float(u.z << 16); o[5] = __uint_as_float(u.z & 0xffff0000u);
    o[6] = __uint_as_float(u.w << 16); o[7] = __uint_as_float(u.w & 0xffff0000u);
}

__device__ __forceinline__ void load_vec16(const double *p, double *o)
{
    const double2 t = *reinterpret_cast<const double2 *>(p);
    o[0] = t.x; o[1] = t.y;
}
// what a staged row element is held as in shared memory: float is exact for fp32 / bf16 rows, binary64 rows stay binary64
template <typename T> struct StageOf { using type = float; };
template <> struct StageOf<double> { using type = double; };

template <bool NEUMAIER, typename T>
__global__ void __launch_bounds__(RS_THREADS, 1) rescore_kernel(const uint64_t *__restrict__ merged, int kp, const T *__restrict__ rows,
                                                            const float *__restrict__ inv_norms, int ld, int dim, int64_t n_rows,
                                                            const void *__restrict__ queries, int q_dtype, double eps,
                                                            FinalizeArgs f, int32_t *__restrict__ flags,
                                                            int32_t *__restrict__ uncertified_count, int chunk,
                                                            const int *__restrict__ extreme, float *__restrict__ collect_thr,
                                                            unsigned long long *__restrict__ cum, const int *__restrict__ incomplete)
{
    constexpr int VEC = 16 / (int)sizeof(T);      // elements per 16-byte load
    extern __shared__ double rs_smem[];
    double *sq = rs_smem;                          // [chunk] query as doubles
    using S = typename StageOf<T>::type;
    S *srow = reinterpret_cast<S *>(rs_smem + chunk);  // [kp][chunk + 1] candidate rows (odd pitch)
    const int pitch = chunk + 1;
    __shared__ double s_dot[64], s_rr[64], s_qq;
    __shared__ double s_score[64];
    __shared__ uint32_t s_row[64];
    __shared__ int s_valid[64];
    __shared__ int s_cnt;
    const int q = blockIdx.x, j = threadIdx.x;
    if (j == 0) s_cnt = 0;
    if (j < 64) {
        uint64_t key = j < kp ? merged[(int64_t)q * kp + j] : 0;
        s_valid[j] = key != 0;
        s_row[j] = key != 0 ? key_row(key) : 0;
    }
    __syncthreads();
    // task decode
    const int kind = j < kp ? 0 : (j < 2 * kp ? 1 : (j == 2 * kp ? 2 : 3));
    const int cand = kind == 0 ? j : (kind == 1 ? j - kp : 0);
    const bool active = kind == 2 || (kind < 2 && s_valid[cand]);
    RefSum acc;
    acc.init();
    for (int c0 = 0; c0 < dim; c0 += chunk) {
        const int len = min(chunk, dim - c0);          // real columns in this chunk
        const int vlen = (min(chunk, ld - c0) + VEC - 1) / VEC;  // 16-byte groups (rows are zero padded to ld)
        for (int i = j; i < len; i += RS_THREADS) sq[i] = load_as_double(queries, q_dtype, (int64_t)q * dim + c0 + i);
        // stage the candidate rows: batches of 4 independent 16-byte loads per thread
        const int groups = kp * vlen;
        for (int g0 = j; g0 < groups; g0 += 4 * RS_THREADS) {
            S buf[4][VEC];
            int rr_[4], cc_[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int g = g0 + u * RS_THREADS;
                rr_[u] = g < groups ? g / vlen : -1;
                cc_[u] = g < groups ? (g - rr_[u] * vlen) * VEC : 0;
                if (rr_[u] >= 0 && s_valid[rr_[u]]) load_vec16(rows + (int64_t)s_row[rr_[u]] * ld + c0 + cc_[u], buf[u]);
                else
#pragma unroll
                    for (int x = 0; x < VEC; ++x) buf[u][x] = (S)0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (rr_[u] >= 0)
#pragma unroll
                    for (int x = 0; x < VEC; ++x)
                        if (cc_[u] + x < chunk) srow[rr_[u] * pitch + cc_[u] + x] = buf[u][x];
        }
        __syncthreads();
        if (active) {
            const S *mine = srow + cand * pitch;
            if (kind == 0)
                ref_sum_range<NEUMAIER>(acc, 0, len, [&](int i) { return __dmul_rn(sq[i], (double)mine[i]); });
            else if (kind == 1)
                ref_sum_range<NEUMAIER>(acc, 0, len, [&](int i) { const double y = (double)mine[i]; return __dmul_rn(y, y); });
            else
                ref_sum_range<NEUMAIER>(acc, 0, len, [&](int i) { const double x = sq[i]; return __dmul_rn(x, x); });
        }
        __syncthreads();
    }
    if (active) {
        const double r = acc.result<NEUMAIER>();
        if (kind == 0) s_dot[cand] = r;
        else if (kind == 1) s_rr[cand] = r;
        else s_qq = r;
    }
    __syncthreads();
    const bool valid = j < 64 && s_valid[j];
    double sc = 0.0;
    const uint32_t row = j < 64 ? s_row[j] : 0;
    if (valid) {
        const double n1 = __dsqrt_rn(s_qq);
        const double n2 = __dsqrt_rn(s_rr[j]);
        sc = (n1 == 0.0 || n2 == 0.0) ? 0.0 : __ddiv_rn(s_dot[j], __dmul_rn(n1, n2));
    }
    if (j < 64) s_score[j] = sc;
    __syncthreads();
    int ncand = 0;
    for (int i = 0; i < 64; ++i) ncand += s_valid[i];
    // rank among valid candidates
    int rank = 0;
    if (valid)
        for (int i = 0; i < 64; ++i)
            if (s_valid[i] && i != j && better(s_score[i], s_row[i], sc, row)) ++rank;
    double outv = convert_score(sc, f.score_mode);
    bool emit = valid && rank < f.k && outv > f.min_score;
    if (emit) {
        f.out_idx[(int64_t)q * f.k + rank] = (int64_t)row + f.row_offset;
        f.out_score[(int64_t)q * f.k + rank] = outv;
        atomicAdd(&s_cnt, 1);
    }
    __syncthreads();
    // certification: every non-candidate row r has approx(r) <= approx(worst candidate), hence
    // exact(r) <= approx_worst + eps; certified iff that is strictly below the k-th exact score.
    // Fewer than kp candidates means every scorable row of the shard is already a candidate.
    // (merge_candidates_kernel puts the worst candidate in slot kp-1.)
    if (valid && rank == min(f.k, ncand) - 1) {
        bool cert = true;
        if (ncand >= kp && (int64_t)ncand < n_rows) {
            float worst = key_score(merged[(int64_t)q * kp + kp - 1]);
            cert = ((double)worst + eps) < sc;
        }
        if (incomplete && incomplete[q]) cert = false;  // the slabs / spill buffer this list was taken from overflowed: rows are missing
        // flag 1: a collect pass (all rows within 2 eps of this score) can settle the query;
        // flag 2: the error bound does not hold for this store -> binary64 scan of every row
        const bool bound_ok = !(extreme && *extreme != 0);
        if (!bound_ok && (int64_t)ncand < n_rows) cert = false;
        flags[q] = cert ? 0 : (bound_ok ? 1 : 2);
        if (collect_thr) {
            float t = (float)(sc - 2.0 * eps);
            t = nextafterf(nextafterf(t, -INFINITY), -INFINITY);  // the cast may have rounded up
            collect_thr[q] = (!cert && bound_ok) ? t : INFINITY;
        }
        if (!cert) { atomicAdd(uncertified_count, 1); if (cum) atomicAdd(cum, 1ull); }
    }
    if (ncand == 0 && j == 0) { flags[q] = 0; if (collect_thr) collect_thr[q] = INFINITY; }
    if (j == 0) f.out_count[q] = s_cnt;
    int cnt = s_cnt;
    for (int t = cnt + j; t < f.k; t += RS_THREADS) {
        f.out_idx[(int64_t)q * f.k + t] = -1;
        f.out_score[(int64_t)q * f.k + t] = 0.0;
    }
}

// =========================================================================================
// 2b. fused candidate selection + exact rescoring + band settlement (the normal path: ONE launch)
// =========================================================================================
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gsrc)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

static constexpr int SR_THREADS = 512;
// Rows of one query's near-tie band the rescoring kernel settles itself: as many as shared memory leaves room for
// (12 bytes each), between BAND_CAP_MIN and BAND_CAP_MAX.  Settling 2048 rows costs ~0.3 ms for the batch (64 staged
// sub-batches per query, the queries in parallel) and no extra pass over the store; bands of up to 4096 rows are left
// to the collect pass (a second streaming scan + its own rescoring), anything larger to the binary64 scan.
static constexpr int BAND_CAP_MIN = 1024, BAND_CAP_MAX = 2048;

// Exact scores of m gathered rows straight from global memory (block-wide; the collect pass, whose row sets do not fit
// shared memory).  The rows sit in DRAM (the scan streams them through L2 with evict-first), so all their 128-byte lines
// are first pulled into L2 by the whole block at once -- a thread walking its row would otherwise pay one serial DRAM
// miss per line.  Then 2m independent sequential chains (dot and ||row||^2 per row: the reference recurrences, in index
// order) run on 2m threads.  s_sc / s_rr / s_row: [m]; on return s_sc holds the reference scores.
template <bool NEUMAIER, typename T, int THREADS>
__device__ void band_score_global(const T *__restrict__ rows, int ld, int dim, const double *sq, double n1, int m, double *s_sc, double *s_rr,
                                  const uint32_t *s_row)
{
    const int tid = threadIdx.x;
    const int lines = (ld * (int)sizeof(T) + 127) / 128;
    for (int e = tid; e < m * lines; e += THREADS) {
        const int r = e / lines, l = e - r * lines;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char *>(rows + (int64_t)s_row[r] * ld) + (size_t)l * 128));
    }
    for (int t = tid; t < 2 * m; t += THREADS) {
        const int e = t >> 1;
        const T *row = rows + (int64_t)s_row[e] * ld;
        RefSum acc;
        acc.init();
        if (t & 1) {
            ref_sum_range<NEUMAIER>(acc, 0, dim, [&](int i) { const double y = load_elem(row, i); return __dmul_rn(y, y); });
            s_rr[e] = acc.result<NEUMAIER>();
        } else {
            ref_sum_range<NEUMAIER>(acc, 0, dim, [&](int i) { return __dmul_rn(sq[i], load_elem(row, i)); });
            s_sc[e] = acc.result<NEUMAIER>();
        }
    }
    __syncthreads();
    for (int e = tid; e < m; e += THREADS) {
        const double n2 = __dsqrt_rn(s_rr[e]);
        s_sc[e] = (n1 == 0.0 || n2 == 0.0) ? 0.0 : __ddiv_rn(s_sc[e], __dmul_rn(n1, n2));
    }
    __syncthreads();
}

// Exact top-k among m rows with reference scores s_sc (block-wide): every row is ranked by counting the rows that beat it
// (score desc, row asc: rows are distinct, so ranks are) and the first k are emitted.  Returns the number of entries
// emitted (uniform).
template <int THREADS>
__device__ int band_emit(int m, const double *s_sc, const uint32_t *s_row, int *s_out, const FinalizeArgs &f, int q)
{
    const int tid = threadIdx.x;
    if (tid == 0) *s_out = 0;
    __syncthreads();
    for (int e = tid; e < m; e += THREADS) {
        const double sc = s_sc[e];
        const uint32_t row = s_row[e];
        int rank = 0;
        for (int i = 0; i < m && rank < f.k; ++i) rank += better(s_sc[i], s_row[i], sc, row) ? 1 : 0;  // k better rows: out
        if (rank < f.k) {
            const double outv = convert_score(sc, f.score_mode);
            if (outv > f.min_score) {   // scores descend with the rank, so the emitted entries are a prefix
                f.out_idx[(int64_t)q * f.k + rank] = (int64_t)row + f.row_offset;
                f.out_score[(int64_t)q * f.k + rank] = outv;
                atomicMax(s_out, rank + 1);
            }
        }
    }
    __syncthreads();
    const int cntv = *s_out;
    if (tid == 0) f.out_count[q] = cntv;
    for (int t = cntv + tid; t < f.k; t += THREADS) {
        f.out_idx[(int64_t)q * f.k + t] = -1;
        f.out_score[(int64_t)q * f.k + t] = 0.0;
    }
    return cntv;
}

static constexpr uint32_t NO_ROW = 0xFFFFFFFFu;

// Stages up to kp rows (ids in s_rid[0, kp), NO_ROW = none) in shared memory with cp.async (16-byte, L2-cached, three
// column chunks; coalesced -- 32 threads each walking their own row in global memory would serialise in the load unit,
// one tag lookup per row per instruction) and runs the reference recurrences as independent sequential chains, chunk c
// overlapping the loads of chunk c+1: thread j < kp: dot(query, row j); kp <= j < 2 kp: ||row j-kp||^2; j == 2 kp and
// s_qq != NULL: ||query||^2.  Results -> s_dot / s_rr / *s_qq.  Block-wide; ends with a barrier.
template <bool NEUMAIER, typename T, int THREADS>
__device__ __forceinline__ void stage_and_chain(const T *__restrict__ rows, int ld, int dim, int kp, const uint32_t *s_rid,
                                                unsigned char *srow, int pitch, const double *sq, double *s_dot, double *s_rr, double *s_qq)
{
    const int tid = threadIdx.x, j = tid;
    const int gpr = ld * (int)sizeof(T) / 16;                 // 16-byte groups per row
    const int c1 = gpr / 3, c2 = 2 * gpr / 3;                 // chunk boundaries (in groups)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int g_lo = c == 0 ? 0 : (c == 1 ? c1 : c2), g_hi = c == 0 ? c1 : (c == 1 ? c2 : gpr);
        const int w = g_hi - g_lo;
        for (int e = tid; e < kp * w; e += THREADS) {
            const int r = e / w, g = g_lo + (e - r * w);
            const uint32_t rid = s_rid[r];
            if (rid != NO_ROW)
                cp_async16(srow + (size_t)r * pitch + (size_t)g * 16,
                           reinterpret_cast<const unsigned char *>(rows + (int64_t)rid * ld) + (size_t)g * 16);
        }
        cp_async_commit();
    }
    const int kind = j < kp ? 0 : (j < 2 * kp ? 1 : ((j == 2 * kp && s_qq != nullptr) ? 2 : 3));
    const int cidx = kind == 0 ? j : (kind == 1 ? j - kp : 0);
    const bool active = kind == 2 || (kind < 2 && s_rid[cidx] != NO_ROW);
    const T *mine = reinterpret_cast<const T *>(srow + (size_t)cidx * pitch);
    constexpr int EPG = 16 / (int)sizeof(T);                  // elements per 16-byte group
    RefSum acc;
    acc.init();
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        if (c == 0) cp_async_wait<2>();
        else if (c == 1) cp_async_wait<1>();
        else cp_async_wait<0>();
        __syncthreads();
        const int g_lo = c == 0 ? 0 : (c == 1 ? c1 : c2), g_hi = c == 0 ? c1 : (c == 1 ? c2 : gpr);
        const int i_lo = g_lo * EPG, i_hi = min(g_hi * EPG, dim);
        if (active) {
            if (kind == 0)
                ref_sum_range<NEUMAIER>(acc, i_lo, i_hi, [&](int i) { return __dmul_rn(sq[i], load_elem(mine, i)); });
            else if (kind == 1)
                ref_sum_range<NEUMAIER>(acc, i_lo, i_hi, [&](int i) { const double y = load_elem(mine, i); return __dmul_rn(y, y); });
            else
                ref_sum_range<NEUMAIER>(acc, i_lo, i_hi, [&](int i) { const double x = sq[i]; return __dmul_rn(x, x); });
        }
    }
    if (active) {
        const double r = acc.result<NEUMAIER>();
        if (kind == 0) s_dot[cidx] = r;
        else if (kind == 1) s_rr[cidx] = r;
        else *s_qq = r;
    }
    __syncthreads();
}

// Where one query's candidate keys come from.
struct SelectSrc {
    const uint64_t *cand;  // list mode: [lists][nq][list_len] (per-CTA lists of the CUDA-core scan, or dumped tiles)
    int lists, list_len;
    int complete;          // list mode: 1 = the lists hold EVERY row of the shard (dump mode)
    // slab mode (tcgen05 scan): per-CTA slabs + the shared spill buffer hold every key at or above the scan's final
    // band threshold; seed_tab = the final per-CTA maxima and the published bounds (NULL: no table)
    const uint64_t *slab;  // [ctas][nq][SCAN_SLAB]
    const int *scnt;       // [ctas][nq]
    int ctas;
    const uint64_t *ubuf;  // [nq][ucap]
    const int *ucnt;       // [nq] keys spilled (> ucap: overflow -> keys are missing)
    int ucap;
    const uint32_t *seed_tab;
    int nq_pad, ksel;
    float band;
    int key_cap;           // keys one CTA stages in shared memory
    int band_cap;          // band rows one CTA can settle (shared-memory room, see BAND_CAP_MIN / MAX)
};

// Slab mode: stages query q's keys in shared memory, filtered once more with the FINAL bound -- the k-th largest of the
// CTAs' final maxima or a published bound, whichever is larger, minus the band: both are lower bounds on the k-th best
// approximate score, so nothing below can matter, whereas the slabs were filled under the looser bounds in force while
// the scan ran (typically ~1000 keys per query come in, a few dozen stay).  Block-wide; returns the number of keys
// staged (uniform) and sets *incomplete when keys are missing (spill or staging overflow).
template <int THREADS>
__device__ int load_slab_keys(const SelectSrc &src, int q, int nq, uint64_t *skeys, int *s_cnts, int *s_total, float *s_bf, bool *incomplete)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (warp == 0) {
        float Lb = -INFINITY;
        if (src.seed_tab != nullptr) {
            if (src.ctas >= src.ksel) Lb = seed_select(src.seed_tab, src.ctas, src.nq_pad, q, src.ksel, lane);
            const uint32_t o = __ldcg(src.seed_tab + SEED_TAB_WORDS + q);
            if (o != 0u) Lb = fmaxf(Lb, f32_from_ordered(o));
        }
        if (lane == 0) { *s_bf = band_floor(Lb, src.band); *s_total = 0; }
    }
    for (int c = tid; c < src.ctas; c += THREADS) s_cnts[c] = min(src.scnt[(size_t)c * nq + q], SCAN_SLAB);
    __syncthreads();
    const float bf = *s_bf;
    // one warp per slab, lanes over its (contiguous) keys; the loads of four slabs are issued before any is consumed
    constexpr int WARPS = THREADS / 32, PER = SCAN_SLAB / 32, BATCH = 4;
    for (int c0 = warp; c0 < src.ctas; c0 += WARPS * BATCH) {
        uint64_t kk[BATCH][PER];
#pragma unroll
        for (int b = 0; b < BATCH; ++b) {
            const int c = c0 + b * WARPS;
            const int cnt = c < src.ctas ? s_cnts[c] : 0;
#pragma unroll
            for (int t = 0; t < PER; ++t)
                kk[b][t] = (lane + 32 * t < cnt) ? __ldcg(src.slab + ((size_t)c * nq + q) * SCAN_SLAB + lane + 32 * t) : 0ull;
        }
#pragma unroll
        for (int b = 0; b < BATCH; ++b)
#pragma unroll
            for (int t = 0; t < PER; ++t) {
                const uint64_t k = kk[b][t];
                if (k != 0 && key_score(k) >= bf) {
                    const int p = atomicAdd(s_total, 1);
                    if (p < src.key_cap) skeys[p] = k;
                }
            }
    }
    const int spilled = src.ucnt[q];
    const int ns = min(spilled, src.ucap);
    for (int e = tid; e < ns; e += THREADS) {
        const uint64_t k = __ldcg(src.ubuf + (size_t)q * src.ucap + e);
        if (k != 0 && key_score(k) >= bf) {
            const int p = atomicAdd(s_total, 1);
            if (p < src.key_cap) skeys[p] = k;
        }
    }
    __syncthreads();
    const int got = *s_total;
    *incomplete = spilled > src.ucap || got > src.key_cap;
    return min(got, src.key_cap);
}

// Slab-mode form of the merge for rows too large for the fused kernel's shared memory: the query's filtered keys ->
// its kp best in descending order, zero padded; incomplete[q] = keys were missing.  One CTA per query.
__global__ void __launch_bounds__(SR_THREADS) slab_top_kernel(SelectSrc src, int nq, int kp, uint64_t *__restrict__ merged,
                                                             int *__restrict__ incomplete)
{
    extern __shared__ __align__(16) unsigned char st_smem[];
    uint64_t *skeys = reinterpret_cast<uint64_t *>(st_smem);  // [key_cap]
    __shared__ int s_cnts[256];
    __shared__ int s_total, s_bin, s_need, s_m;
    __shared__ int hist[256];
    __shared__ float s_bf;
    const int q = blockIdx.x, tid = threadIdx.x;
    bool inc = false;
    const int total = load_slab_keys<SR_THREADS>(src, q, nq, skeys, s_cnts, &s_total, &s_bf, &inc);
    for (int e = tid; e < kp; e += SR_THREADS) merged[(int64_t)q * kp + e] = 0;
    if (tid == 0) { incomplete[q] = inc ? 1 : 0; s_m = 0; }
    __syncthreads();
    if (total <= MERGE_SURV) {
        for (int e = tid; e < total; e += SR_THREADS) {
            const uint64_t k = skeys[e];
            int rank = 0;
            for (int i = 0; i < total; ++i) rank += skeys[i] > k ? 1 : 0;
            if (rank < kp) merged[(int64_t)q * kp + rank] = k;
        }
        return;
    }
    const uint64_t Tk = radix_select_kth(skeys, total, kp, hist, &s_bin, &s_need);
    for (int e = tid; e < total; e += SR_THREADS) {
        const uint64_t k = skeys[e];
        if (k > Tk) merged[(int64_t)q * kp + atomicAdd(&s_m, 1)] = k;
        else if (k == Tk) merged[(int64_t)q * kp + kp - 1] = k;  // the worst candidate goes last
    }
}

// One CTA (512 threads) per query:
//   A. the query's candidate keys are loaded into shared memory (union buffer: typically a few dozen keys; dumped
//      tiles / per-CTA lists: thinned with the list-maxima bound, see merge_candidates_kernel) and the kp best by
//      approximate score are ranked;
//   B. their rows are pulled into shared memory with cp.async (16-byte, L2-cached) in three column chunks;
//   C. the reference recurrences (dot per candidate, ||row||^2 per candidate, ||q||^2) run as independent
//      sequential chains on 2kp+1 threads, chunk c overlapping the loads of chunk c+1;
//   D. rank, emit, certify: with s_k the k-th exact score, only rows whose approximate score reaches s_k - eps can
//      still matter.  When the source is complete they are all in shared memory already: if they are all among the
//      rescored kp the list is final, otherwise
//   E. the whole band (<= band_cap rows) is rescored with the reference recurrence right here and the exact top-k
//      of it is emitted -- no second scan.  Only an incomplete source (union-buffer overflow, CUDA-core lists) or a
//      band beyond band_cap flags the query for the collect pass / the binary64 scan of every row.
// Every rescored candidate also audits the scan's error bound: |approximate - exact| > eps flags the query for the
// binary64 scan (and is counted), so a wrong bound cannot silently produce a wrong list.
template <bool NEUMAIER, typename T>
__global__ void __launch_bounds__(SR_THREADS, 1) select_rescore_kernel(SelectSrc src, int nq, int kp,
                                                                   const T *__restrict__ rows, int ld, int dim, int64_t n_rows,
                                                                   const void *__restrict__ queries, int q_dtype, double eps,
                                                                   FinalizeArgs f, int32_t *__restrict__ flags,
                                                                   int32_t *__restrict__ uncertified_count,
                                                                   const int *__restrict__ extreme, float *__restrict__ collect_thr,
                                                                   unsigned long long *__restrict__ cum, const float *__restrict__ inv_norms)
{
    extern __shared__ __align__(16) unsigned char sr_smem[];
    uint64_t *skeys = reinterpret_cast<uint64_t *>(sr_smem);                       // [key_cap]
    uint32_t *lmax = reinterpret_cast<uint32_t *>(skeys + src.key_cap);            // [lists] (+pad)
    double *sq = reinterpret_cast<double *>(lmax + ((src.lists + 3) & ~3));        // [dim]
    const int pitch = ld * (int)sizeof(T) + 16;                                    // bytes, 16-B aligned rows
    unsigned char *srow = reinterpret_cast<unsigned char *>(sq + ((dim + 1) & ~1)); // [kp][pitch] staged rows
    double *b_sc = reinterpret_cast<double *>(srow + (((size_t)kp * pitch + 15) & ~(size_t)15));  // [band_cap] band scores
    uint32_t *b_row = reinterpret_cast<uint32_t *>(b_sc + src.band_cap);                       // [band_cap] band rows
    __shared__ uint64_t s_top[64];
    __shared__ uint32_t s_rid[64];
    __shared__ uint64_t surv[MERGE_SURV];
    __shared__ int hist[256];
    __shared__ int s_bin, s_need, s_m, s_nz, s_cnt, s_band, s_viol, s_out, s_total;
    __shared__ int s_cnts[256];
    __shared__ uint32_t s_L;
    __shared__ float s_thr, s_bf;
    __shared__ double s_dot[64], s_rr[64], s_qq, s_score[64];
    const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    pdl_launch_dependents();
    if (tid == 0) { s_m = 0; s_nz = 0; s_cnt = 0; s_band = 0; s_viol = 0; s_thr = -INFINITY; }
    if (tid < 64) s_top[tid] = 0;
    pdl_wait();  // the scan has completed: its keys are visible
    __syncthreads();

    // ---------------- A. candidate selection ----------------
    const bool union_mode = src.slab != nullptr;
    int total, lists = src.lists, list_len = src.list_len;
    bool overflow = false;
    int nz = 0;
    if (union_mode) {
        total = load_slab_keys<SR_THREADS>(src, q, nq, skeys, s_cnts, &s_total, &s_bf, &overflow);
        lists = 0;
        if (tid == 0) nz = total;  // staged keys are non-zero by construction
    } else {
        total = lists * list_len;
#pragma unroll 10
        for (int e = tid; e < total; e += SR_THREADS) {
            const int l = e / list_len, j = e - l * list_len;
            const uint64_t k = src.cand[((int64_t)l * nq + q) * list_len + j];
            skeys[e] = k;
            nz += k != 0;
        }
    }
    for (int i = tid; i < dim; i += SR_THREADS) sq[i] = load_as_double(queries, q_dtype, (int64_t)q * dim + i);
    if (nz) atomicAdd(&s_nz, nz);
    __syncthreads();
    const int nonzero = s_nz;
    bool done = false;
    if (total <= MERGE_SURV) {
        // few keys (the union buffer's normal case): rank them directly (keys are unique)
        for (int e = tid; e < total; e += SR_THREADS) {
            const uint64_t k = skeys[e];
            if (k == 0) continue;
            int rank = 0;
            for (int i = 0; i < total; ++i) rank += skeys[i] > k ? 1 : 0;
            if (rank < kp) s_top[rank] = k;
        }
        done = true;
    } else if (nonzero >= kp && lists >= kp && lists <= 256) {
        for (int l = warp; l < lists; l += SR_THREADS / 32) {
            uint32_t m = 0;
            for (int j = lane; j < list_len; j += 32) m = max(m, (uint32_t)(skeys[l * list_len + j] >> 32));
            m = __reduce_max_sync(0xffffffffu, m);
            if (lane == 0) lmax[l] = m;
        }
        __syncthreads();
        if (warp == 0) {
            uint32_t vals[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) vals[t] = (lane + 32 * t) < lists ? lmax[lane + 32 * t] : 0u;
            uint32_t prefix = 0;
            int need = kp;
            for (int bit = 31; bit >= 12; --bit) {  // 20 bits: truncation only loosens the bound
                const uint32_t hi = bit == 31 ? 0u : (0xFFFFFFFFu << (bit + 1));
                int cnt = 0;
#pragma unroll
                for (int t = 0; t < 8; ++t) cnt += ((vals[t] & hi) == prefix && ((vals[t] >> bit) & 1u)) ? 1 : 0;
                const int tot = __reduce_add_sync(0xffffffffu, cnt);
                if (tot >= need) prefix |= 1u << bit;
                else need -= tot;
            }
            if (lane == 0) s_L = prefix;
        }
        __syncthreads();
        const uint32_t Lb = s_L;
        if (Lb != 0) {
            for (int e = tid; e < total; e += SR_THREADS) {
                const uint64_t k = skeys[e];
                if ((uint32_t)(k >> 32) >= Lb && k != 0) {
                    const int p = atomicAdd(&s_m, 1);
                    if (p < MERGE_SURV) surv[p] = k;
                }
            }
            __syncthreads();
            const int m = s_m;
            if (m >= kp && m <= MERGE_SURV) {
                for (int e = tid; e < m; e += SR_THREADS) {
                    const uint64_t k = surv[e];
                    int rank = 0;
                    for (int i = 0; i < m; ++i) rank += surv[i] > k ? 1 : 0;
                    if (rank < kp) s_top[rank] = k;
                }
                done = true;
            }
        }
    }
    if (!done) {  // uniform across the block: exact radix select (few lists, heavy duplication, a large union)
        __syncthreads();
        uint64_t Tk = 1;
        if (nonzero >= kp) Tk = radix_select_kth(skeys, total, kp, hist, &s_bin, &s_need);
        if (tid == 0) s_m = 0;
        __syncthreads();
        for (int e = tid; e < total; e += SR_THREADS) {
            const uint64_t k = skeys[e];
            if (k >= Tk && k != 0) {
                if (nonzero >= kp && k == Tk) s_top[kp - 1] = k;  // the worst candidate goes last
                else s_top[atomicAdd(&s_m, 1)] = k;
            }
        }
    }
    __syncthreads();

    // ---------------- B + C. stage the candidate rows, sequential reference chains ----------------
    const int j = tid;
    const uint64_t mykey = j < 64 ? s_top[j] : 0;
    const bool cand_valid = j < kp && mykey != 0;
    if (j < 64) s_rid[j] = cand_valid ? key_row(mykey) : NO_ROW;
    __syncthreads();
    stage_and_chain<NEUMAIER, T, SR_THREADS>(rows, ld, dim, kp, s_rid, srow, pitch, sq, s_dot, s_rr, &s_qq);

    // ---------------- D. rank, emit, certify ----------------
    double sc = 0.0;
    const uint32_t row = cand_valid ? key_row(mykey) : 0;
    const double n1 = __dsqrt_rn(s_qq);
    if (n1 == 0.0) {
        // zero query (uniform: s_qq is shared): the reference scores 0.0 against every row (pre_llm_injector.py:385-386) and
        // its stable sort keeps store order -> the first k scorable rows, no scan result needed
        if (tid == 0) {
            int c = 0;
            const double outv = convert_score(0.0, f.score_mode);
            if (outv > f.min_score)
                for (int64_t r = 0; r < n_rows && c < f.k; ++r)
                    if (__ldg(inv_norms + r) >= 0.0f) {
                        f.out_idx[(int64_t)q * f.k + c] = r + f.row_offset;
                        f.out_score[(int64_t)q * f.k + c] = outv;
                        ++c;
                    }
            for (int t = c; t < f.k; ++t) { f.out_idx[(int64_t)q * f.k + t] = -1; f.out_score[(int64_t)q * f.k + t] = 0.0; }
            f.out_count[q] = c;
            flags[q] = 0;
            if (collect_thr) collect_thr[q] = INFINITY;
        }
        return;
    }
    if (cand_valid) {
        const double n2 = __dsqrt_rn(s_rr[j]);
        sc = (n1 == 0.0 || n2 == 0.0) ? 0.0 : __ddiv_rn(s_dot[j], __dmul_rn(n1, n2));
        // audit of the scan's error bound on every rescored candidate
        if (fabs((double)key_score(mykey) - sc) > eps) atomicAdd(&s_viol, 1);
    }
    if (j < 64) s_score[j] = sc;
    __syncthreads();
    int ncand = 0;
    for (int i = 0; i < kp; ++i) ncand += s_top[i] != 0;
    int rank = 0;
    if (cand_valid)
        for (int i = 0; i < kp; ++i)
            if (s_top[i] != 0 && i != j && better(s_score[i], key_row(s_top[i]), sc, row)) ++rank;
    const double outv = convert_score(sc, f.score_mode);
    const bool emit = cand_valid && rank < f.k && outv > f.min_score;
    if (emit) {
        f.out_idx[(int64_t)q * f.k + rank] = (int64_t)row + f.row_offset;
        f.out_score[(int64_t)q * f.k + rank] = outv;
        atomicAdd(&s_cnt, 1);
    }
    // the k-th exact score decides which other rows could still matter: approximate score >= s_k - eps
    if (cand_valid && ncand >= f.k && rank == f.k - 1) {
        float t = (float)(sc - eps);
        t = nextafterf(nextafterf(t, -INFINITY), -INFINITY);  // the cast may have rounded up
        s_thr = t;
    }
    __syncthreads();
    const float thr = s_thr;  // -inf when there are fewer than k candidates (then every key is in the band)
    {
        int inb = 0;
        for (int e = tid; e < total; e += SR_THREADS) {
            const uint64_t k = skeys[e];
            inb += (k != 0 && key_score(k) >= thr) ? 1 : 0;
        }
        if (inb) atomicAdd(&s_band, inb);
    }
    __syncthreads();
    const int band = s_band;
    const bool bound_ok = !(extreme && *extreme != 0) && s_viol == 0;
    const bool src_complete = union_mode ? !overflow : (src.complete != 0);
    bool cert;
    if (src_complete) cert = band <= ncand;            // every band row is among the rescored candidates
    else if (union_mode) cert = false;                 // overflowed union buffer: rows are missing
    else cert = ncand < kp || band < kp;               // per-CTA top-kp lists: outside rows are bounded by the kp-th key only
    if (!bound_ok && (int64_t)ncand < n_rows) cert = false;
    if (ncand == 0) cert = true;
    if (cert) {
        if (tid == 0) {
            flags[q] = 0;
            if (collect_thr) collect_thr[q] = INFINITY;
            f.out_count[q] = s_cnt;
        }
        const int cnt = s_cnt;
        for (int t = cnt + tid; t < f.k; t += SR_THREADS) {
            f.out_idx[(int64_t)q * f.k + t] = -1;
            f.out_score[(int64_t)q * f.k + t] = 0.0;
        }
        return;
    }
    if (tid == 0 && cum) { atomicAdd(cum, 1ull); if (s_viol) atomicAdd(cum + 4, 1ull); }
    if (bound_ok && src_complete && band <= src.band_cap) {
        // ---------------- E. settle from the band ----------------
        // the band's rows go through the same staging + chains as the candidates, kp rows at a time
        if (tid == 0) s_m = 0;
        __syncthreads();
        for (int e = tid; e < total; e += SR_THREADS) {
            const uint64_t k = skeys[e];
            if (k != 0 && key_score(k) >= thr) b_row[atomicAdd(&s_m, 1)] = key_row(k);
        }
        __syncthreads();
        for (int b0 = 0; b0 < band; b0 += kp) {
            const int cnt = min(kp, band - b0);
            if (tid < 64) s_rid[tid] = tid < cnt ? b_row[b0 + tid] : NO_ROW;
            __syncthreads();
            stage_and_chain<NEUMAIER, T, SR_THREADS>(rows, ld, dim, kp, s_rid, srow, pitch, sq, s_dot, s_rr, nullptr);
            if (tid < cnt) {
                const double n2 = __dsqrt_rn(s_rr[tid]);
                b_sc[b0 + tid] = (n1 == 0.0 || n2 == 0.0) ? 0.0 : __ddiv_rn(s_dot[tid], __dmul_rn(n1, n2));
            }
            __syncthreads();
        }
        band_emit<SR_THREADS>(band, b_sc, b_row, &s_out, f, q);
        if (tid == 0) {
            flags[q] = 0;
            if (collect_thr) collect_thr[q] = INFINITY;
            if (cum) atomicAdd(cum + 1, 1ull);
        }
        return;
    }
    // the collect pass (one more streaming scan gathering every row >= s_k - 2 eps) or, when the bound itself is
    // in doubt, the binary64 scan of every row settles the query; the provisional list stays in place until then
    if (tid == 0) {
        flags[q] = bound_ok ? 1 : 2;
        if (collect_thr) {
            float t = thr > -INFINITY ? (float)((double)thr - eps) : -INFINITY;
            t = nextafterf(t, -INFINITY);
            collect_thr[q] = bound_ok ? t : INFINITY;
        }
        atomicAdd(uncertified_count, 1);
        f.out_count[q] = s_cnt;
    }
    const int cnt = s_cnt;
    for (int t = cnt + tid; t < f.k; t += SR_THREADS) {
        f.out_idx[(int64_t)q * f.k + t] = -1;
        f.out_score[(int64_t)q * f.k + t] = 0.0;
    }
}

// =========================================================================================
// 2c. collect pass: exact top-k among the rows the second scan gathered for an uncertified query
// =========================================================================================
// One CTA (512 threads) per query with flag 1.  The collect scan stored every row whose approximate
// score reached (exact k-th candidate score - 2 eps): that set contains the reference's top-k (a row
// outside it is more than eps below the k-th candidate).  All gathered rows are scored with the
// reference recurrence (band_score_global + band_emit) and the best k by (score desc, row asc) are emitted; the query's flag is
// cleared.  If the buffer overflowed the flag becomes 2 and the binary64 scan of every row takes over.
static constexpr int CR_THREADS = 512;
template <bool NEUMAIER, typename T>
__global__ void __launch_bounds__(CR_THREADS, 1) collect_rescore_kernel(const uint64_t *__restrict__ buf, const int *__restrict__ cnt, int cap,
                                                                       const T *__restrict__ rows, int ld, int dim,
                                                                       const void *__restrict__ queries, int q_dtype, FinalizeArgs f,
                                                                       int32_t *__restrict__ flags, int32_t *__restrict__ uncertified_count,
                                                                       int nq, unsigned long long *__restrict__ cum, int stage_rows)
{
    // stage_rows > 0: the gathered rows take the rescoring kernel's staged route (stage_and_chain), stage_rows at a time;
    // 0 (rows too wide for shared memory): they are scored straight from global memory
    extern __shared__ __align__(16) unsigned char cr_smem[];
    double *sq = reinterpret_cast<double *>(cr_smem);               // [dim]
    double *s_sc = sq + ((dim + 1) & ~1);                           // [cap]
    double *s_rr = s_sc + cap;                                      // [cap] (global route only)
    uint32_t *s_row = reinterpret_cast<uint32_t *>(s_sc + (stage_rows > 0 ? cap : 2 * cap));     // [cap]
    const int pitch = ld * (int)sizeof(T) + 16;
    unsigned char *srow = reinterpret_cast<unsigned char *>(s_row + ((cap + 3) & ~3));  // [stage_rows][pitch] (staged route only)
    __shared__ double s_n1;
    __shared__ int s_out;
    __shared__ uint32_t s_rid[64];
    __shared__ double s_dot[64], s_r2[64];
    const int q = blockIdx.x, tid = threadIdx.x;
    if (flags[nq] == 0 || flags[q] != 1) return;
    const int m = cnt[q];
    if (m > cap) {  // too many rows inside the band: leave it to the full binary64 scan
        if (tid == 0) flags[q] = 2;
        return;
    }
    for (int i = tid; i < dim; i += CR_THREADS) sq[i] = load_as_double(queries, q_dtype, (int64_t)q * dim + i);
    for (int e = tid; e < m; e += CR_THREADS) s_row[e] = key_row(buf[(size_t)q * cap + e]);
    __syncthreads();
    if (tid == 0) {
        RefSum qq; qq.init();
        ref_sum_range<NEUMAIER>(qq, 0, dim, [&](int i) { return __dmul_rn(sq[i], sq[i]); });
        s_n1 = __dsqrt_rn(qq.result<NEUMAIER>());
    }
    __syncthreads();
    if (stage_rows > 0) {
        const double n1 = s_n1;
        for (int b0 = 0; b0 < m; b0 += stage_rows) {
            const int c = min(stage_rows, m - b0);
            if (tid < 64) s_rid[tid] = tid < c ? s_row[b0 + tid] : NO_ROW;
            __syncthreads();
            stage_and_chain<NEUMAIER, T, CR_THREADS>(rows, ld, dim, stage_rows, s_rid, srow, pitch, sq, s_dot, s_r2, nullptr);
            if (tid < c) {
                const double n2 = __dsqrt_rn(s_r2[tid]);
                s_sc[b0 + tid] = (n1 == 0.0 || n2 == 0.0) ? 0.0 : __ddiv_rn(s_dot[tid], __dmul_rn(n1, n2));
            }
            __syncthreads();
        }
    } else {
        band_score_global<NEUMAIER, T, CR_THREADS>(rows, ld, dim, sq, s_n1, m, s_sc, s_rr, s_row);
    }
    band_emit<CR_THREADS>(m, s_sc, s_row, &s_out, f, q);
    if (tid == 0) {
        flags[q] = 0;
        atomicSub(uncertified_count, 1);
        if (cum) atomicAdd(cum + 2, 1ull);
    }
}

// =========================================================================================
// 3. always-exact binary64 scan (uncertified queries / VM_FLAG_FORCE_EXACT)
// =========================================================================================
// Grid-stride over 128-row tiles; thread t scores row tile*128+t against one flagged query at a
// time.  Per-CTA exact top-k list in shared memory, updated by parallel rank-merge whenever a
// tile produced a row that beats the current k-th entry.  Lists go to xlist_*[cta][q][k]; they are reduced by
// exact_merge_kernel (VM_FLAG_FORCE_EXACT: every query) or -- in the conditional form that follows every fast
// pass, which exits at once when nothing is flagged -- by the last CTA to finish (ticket), so the rare fix-up is
// ONE launch.
#define XK 64

// k rounds of block arg-best over lists*k (score,row) pairs that stay in global/L2 -> best k of query q.
template <int THREADS>
__device__ void exact_merge_query(const double *__restrict__ xlist_score, const uint32_t *__restrict__ xlist_row,
                                  const int32_t *__restrict__ xlist_cnt, int lists, int nq, int k, int q, const FinalizeArgs &f,
                                  uint8_t *__restrict__ taken, double *w_s, uint32_t *w_r, int *w_p, int *s_out)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int total = lists * k;
    uint8_t *tk = taken + (int64_t)q * total;
    for (int e = tid; e < total; e += THREADS) tk[e] = 0;
    if (tid == 0) *s_out = 0;
    __syncthreads();
    auto scan_local = [&](double &bs, uint32_t &br, int &bp) {
        bp = -1; bs = 0.0; br = 0;
        for (int e = tid; e < total; e += THREADS) {
            int l = e / k, j = e - l * k;
            if (tk[e] || j >= xlist_cnt[(int64_t)l * nq + q]) continue;
            int64_t g = ((int64_t)l * nq + q) * k + j;
            double s = xlist_score[g];
            uint32_t r = xlist_row[g];
            if (bp < 0 || better(s, r, bs, br)) { bs = s; br = r; bp = e; }
        }
    };
    double bs; uint32_t br; int bp;
    scan_local(bs, br, bp);
    for (int r = 0; r < f.k; ++r) {
        double ms = bs; uint32_t mr = br; int mp = bp;
        for (int o = 16; o > 0; o >>= 1) {
            double ts = __shfl_xor_sync(0xffffffffu, ms, o);
            uint32_t tr = __shfl_xor_sync(0xffffffffu, mr, o);
            int tp = __shfl_xor_sync(0xffffffffu, mp, o);
            if (tp >= 0 && (mp < 0 || better(ts, tr, ms, mr))) { ms = ts; mr = tr; mp = tp; }
        }
        if (lane == 0) { w_s[warp] = ms; w_r[warp] = mr; w_p[warp] = mp; }
        __syncthreads();
        ms = w_s[0]; mr = w_r[0]; mp = w_p[0];
        for (int w = 1; w < THREADS / 32; ++w)
            if (w_p[w] >= 0 && (mp < 0 || better(w_s[w], w_r[w], ms, mr))) { ms = w_s[w]; mr = w_r[w]; mp = w_p[w]; }
        if (mp < 0) break;  // uniform
        double outv = convert_score(ms, f.score_mode);
        if (tid == 0 && outv > f.min_score) {
            f.out_idx[(int64_t)q * f.k + r] = (int64_t)mr + f.row_offset;
            f.out_score[(int64_t)q * f.k + r] = outv;
            *s_out = r + 1;
        }
        if (mp == bp) {
            tk[bp] = 1;
            scan_local(bs, br, bp);
        }
        __syncthreads();
    }
    __syncthreads();
    int cnt = *s_out;
    if (tid == 0) f.out_count[q] = cnt;
    for (int t = cnt + tid; t < f.k; t += THREADS) {
        f.out_idx[(int64_t)q * f.k + t] = -1;
        f.out_score[(int64_t)q * f.k + t] = 0.0;
    }
    __syncthreads();
}

// 256 threads per CTA: thread t < 128 runs the dot chain of row tile*128+t, thread 128+t its ||row||^2 chain.  The tile's
// rows are staged through shared memory in column chunks of 384 bytes per row (cp.async, coalesced, three buffers: the
// next two chunks load while the chains run over one) -- a thread walking its own row in global memory would make every warp
// instruction touch 32 different rows and serialise in the load unit (the first version of this kernel: 3.1 ms per
// query-pass over 1 M x 384 fp32).
static constexpr int XS_THREADS = 256;
static constexpr int XS_CG = 24;                    // 16-byte groups per staged chunk
static constexpr int XS_PITCH = XS_CG * 16 + 16;    // bytes; odd multiple of 16 -> conflict-free per-thread walks

template <bool NEUMAIER, typename T>
__global__ void __launch_bounds__(XS_THREADS) exact_scan_kernel(const T *__restrict__ rows, const float *__restrict__ inv_norms,
                                                               int64_t n, int ld, int dim, const void *__restrict__ queries,
                                                               int q_dtype, int nq, int32_t *__restrict__ flags, int k,
                                                               double *__restrict__ xlist_score, uint32_t *__restrict__ xlist_row,
                                                               int32_t *__restrict__ xlist_cnt, unsigned long long *__restrict__ cum,
                                                               int *__restrict__ done_ctr, FinalizeArgs f, uint8_t *__restrict__ taken)
{
    pdl_launch_dependents();
    pdl_wait();
    // flags[nq] is the uncertified-query counter written by the rescoring kernel: nothing to do when 0
    if (flags && flags[nq] == 0) return;
    if (flags && cum && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(cum + 3, (unsigned long long)flags[nq]);
    extern __shared__ __align__(16) unsigned char xs_smem[];
    double *sq = reinterpret_cast<double *>(xs_smem);                                          // [dim] query as doubles
    unsigned char *buf0 = reinterpret_cast<unsigned char *>(sq + ((dim + 1) & ~1));              // [3][128][XS_PITCH]
    __shared__ double l_score[XK], n_score[XK];
    __shared__ uint32_t l_row[XK], n_row[XK];
    __shared__ double c_score[128];
    __shared__ uint32_t c_row[128];
    __shared__ double s_dotv[128], s_rrv[128];
    __shared__ int l_cnt, c_cnt;
    __shared__ double s_n1;
    const int tid = threadIdx.x, rt = tid & 127;
    const bool is_rr = tid >= 128;
    const int gpr = ld * (int)sizeof(T) / 16;                   // 16-byte groups per row
    const int nchunks = (gpr + XS_CG - 1) / XS_CG;
    constexpr int EPG = 16 / (int)sizeof(T);                    // elements per group
    for (int q = 0; q < nq; ++q) {
        if (flags && flags[q] == 0) continue;  // uniform across the grid
        __syncthreads();
        for (int i = tid; i < dim; i += XS_THREADS) sq[i] = load_as_double(queries, q_dtype, (int64_t)q * dim + i);
        if (tid == 0) { l_cnt = 0; c_cnt = 0; }
        __syncthreads();
        if (tid == 0) {
            RefSum qq; qq.init();
            ref_sum_range<NEUMAIER>(qq, 0, dim, [&](int i) { return __dmul_rn(sq[i], sq[i]); });
            s_n1 = __dsqrt_rn(qq.result<NEUMAIER>());
        }
        __syncthreads();
        const double n1 = s_n1;
        // linear pipeline over (tile, chunk) steps with three buffers: the loads of steps s+1 and s+2 are in flight while
        // the chains run over step s, also across tile boundaries
        const int64_t ntiles = (n + 127) / 128;
        const int my_tiles = (int)((ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
        const int total_steps = my_tiles > 0 ? my_tiles * nchunks : 0;
        auto issue = [&](int st) {
            if (st < total_steps) {
                const int64_t tile = blockIdx.x + (int64_t)(st / nchunks) * gridDim.x;
                const int c = st % nchunks;
                unsigned char *buf = buf0 + (size_t)(st % 3) * 128 * XS_PITCH;
                const int g0 = c * XS_CG, gw = min(XS_CG, gpr - g0);
                for (int e = tid; e < 128 * gw; e += XS_THREADS) {
                    const int rr_ = e / gw, g = e - rr_ * gw;
                    const int64_t row = tile * 128 + rr_;
                    if (row < n)
                        cp_async16(buf + (size_t)rr_ * XS_PITCH + (size_t)g * 16,
                                   reinterpret_cast<const unsigned char *>(rows + row * (int64_t)ld) + (size_t)(g0 + g) * 16);
                }
            }
            cp_async_commit();  // always (an empty group keeps the wait arithmetic uniform)
        };
        issue(0);
        issue(1);
        RefSum acc;
        acc.init();
        for (int st = 0; st < total_steps; ++st) {
            const int64_t tile = blockIdx.x + (int64_t)(st / nchunks) * gridDim.x;
            const int c = st % nchunks;
            const int64_t r = tile * 128 + rt;
            const bool live = r < n && inv_norms[r] >= 0.0f;
            issue(st + 2);
            cp_async_wait<2>();   // everything but the two newest groups has landed: step st is complete
            __syncthreads();
            const unsigned char *cur = buf0 + (size_t)(st % 3) * 128 * XS_PITCH;
            const int i_lo = c * XS_CG * EPG, i_hi = min((c + 1) * XS_CG * EPG, dim);
            if (live && i_lo < i_hi) {
                const T *mine = reinterpret_cast<const T *>(cur + (size_t)rt * XS_PITCH);
                if (!is_rr)
                    ref_sum_range<NEUMAIER>(acc, i_lo, i_hi, [&](int i) { return __dmul_rn(sq[i], load_elem(mine, i - i_lo)); });
                else
                    ref_sum_range<NEUMAIER>(acc, i_lo, i_hi, [&](int i) { const double y = load_elem(mine, i - i_lo); return __dmul_rn(y, y); });
            }
            if (c + 1 < nchunks) {
                __syncthreads();  // all chains are done with this buffer before step st+3 is loaded into it
                continue;
            }
            // ---- the tile is complete ----
            if (live) { if (is_rr) s_rrv[rt] = acc.result<NEUMAIER>(); else s_dotv[rt] = acc.result<NEUMAIER>(); }
            acc.init();
            __syncthreads();      // also orders the buffer reuse
            double sc = 0.0;
            // candidate iff list not full or beats the current worst (k-th) entry
            bool hit = false;
            if (live && !is_rr) {
                const double n2 = __dsqrt_rn(s_rrv[rt]);
                sc = (n1 == 0.0 || n2 == 0.0) ? 0.0 : __ddiv_rn(s_dotv[rt], __dmul_rn(n1, n2));
                const int lc = l_cnt;
                hit = lc < k || better(sc, (uint32_t)r, l_score[lc - 1], l_row[lc - 1]);
            }
            if (hit) {
                const int p = atomicAdd(&c_cnt, 1);
                c_score[p] = sc;
                c_row[p] = (uint32_t)r;
            }
            // barrier + block-wide hit count in one step: every thread sees the same cc, so the
            // merge branch below is taken uniformly (a plain read of c_cnt could race with the
            // next tile's atomicAdd)
            const int cc = __syncthreads_count(hit ? 1 : 0);
            const int lc = l_cnt;
            if (cc > 0) {
                // rank-merge list (lc) and candidates (cc): entry e in [0, lc+cc)
                for (int e = tid; e < lc + cc; e += XS_THREADS) {
                    const double se = e < lc ? l_score[e] : c_score[e - lc];
                    const uint32_t re = e < lc ? l_row[e] : c_row[e - lc];
                    int rank = 0;
                    for (int i = 0; i < lc; ++i) rank += better(l_score[i], l_row[i], se, re) ? 1 : 0;
                    for (int i = 0; i < cc; ++i) rank += better(c_score[i], c_row[i], se, re) ? 1 : 0;
                    if (rank < k) { n_score[rank] = se; n_row[rank] = re; }
                }
                __syncthreads();
                const int nl = min(k, lc + cc);
                for (int e = tid; e < nl; e += XS_THREADS) { l_score[e] = n_score[e]; l_row[e] = n_row[e]; }
                if (tid == 0) { l_cnt = nl; c_cnt = 0; }
                __syncthreads();
            }
        }
        cp_async_wait<0>();
        __syncthreads();
        const int lc = l_cnt;
        const int64_t base = ((int64_t)blockIdx.x * nq + q) * k;
        for (int e = tid; e < lc; e += XS_THREADS) { xlist_score[base + e] = l_score[e]; xlist_row[base + e] = l_row[e]; }
        if (tid == 0) xlist_cnt[(int64_t)blockIdx.x * nq + q] = lc;
    }
    if (done_ctr == nullptr) return;
    // conditional form: the last CTA to finish reduces the per-CTA lists of every flagged query
    __shared__ int s_last, s_out;
    __shared__ double w_s[XS_THREADS / 32];
    __shared__ uint32_t w_r[XS_THREADS / 32];
    __shared__ int w_p[XS_THREADS / 32];
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(done_ctr, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int q = 0; q < nq; ++q) {
        if (flags[q] == 0) continue;
        exact_merge_query<XS_THREADS>(xlist_score, xlist_row, xlist_cnt, (int)gridDim.x, nq, k, q, f, taken, w_s, w_r, w_p, &s_out);
        if (tid == 0) flags[q] = 0;
    }
    if (tid == 0) { *done_ctr = 0; flags[nq] = 0; }
}

// One CTA (256 threads) per query; skips queries whose flag is 0.
__global__ void __launch_bounds__(256) exact_merge_kernel(const double *__restrict__ xlist_score, const uint32_t *__restrict__ xlist_row,
                                                         const int32_t *__restrict__ xlist_cnt, int lists, int nq, int k,
                                                         const int32_t *__restrict__ flags, FinalizeArgs f, uint8_t *__restrict__ taken)
{
    __shared__ double w_s[8];
    __shared__ uint32_t w_r[8];
    __shared__ int w_p[8];
    __shared__ int s_out;
    const int q = blockIdx.x;
    if (flags && (flags[nq] == 0 || flags[q] == 0)) return;
    exact_merge_query<256>(xlist_score, xlist_row, xlist_cnt, lists, nq, k, q, f, taken, w_s, w_r, w_p, &s_out);
}

// =========================================================================================
// 4. cross-shard merge: lists [L][nq][k] of (idx i64, score f64) + count [L][nq] -> best k
// =========================================================================================
// List l lives at base + l*stride (bytes) for each of the three arrays, so both the public
// [L][nq][k] layout and the packed all-gather receive buffer are accepted.
__global__ void __launch_bounds__(256) merge_topk_lists_kernel(const char *__restrict__ idx_b, const char *__restrict__ score_b,
                                                              const char *__restrict__ count_b, size_t stride, int lists, int nq, int k,
                                                              int64_t *__restrict__ out_idx, double *__restrict__ out_score,
                                                              int32_t *__restrict__ out_count)
{
    extern __shared__ unsigned char smem_raw[];
    const int q = blockIdx.x, tid = threadIdx.x;
    const int total = lists * k;
    double *s_s = (double *)smem_raw;
    int64_t *s_i = (int64_t *)(s_s + total);
    int *s_v = (int *)(s_i + total);
    for (int e = tid; e < total; e += 256) {
        int l = e / k, j = e - l * k;
        const int64_t *idx = (const int64_t *)(idx_b + (size_t)l * stride);
        const double *score = (const double *)(score_b + (size_t)l * stride);
        const int32_t *count = (const int32_t *)(count_b + (size_t)l * stride);
        int64_t g = (int64_t)q * k + j;
        bool v = j < count[q];
        s_s[e] = v ? score[g] : 0.0;
        s_i[e] = v ? idx[g] : -1;
        s_v[e] = v ? 1 : 0;
    }
    __syncthreads();
    int nvalid = 0;
    for (int e = 0; e < total; ++e) nvalid += s_v[e];
    for (int e = tid; e < total; e += 256) {
        if (!s_v[e]) continue;
        int rank = 0;
        for (int i = 0; i < total; ++i)
            if (s_v[i] && (s_s[i] > s_s[e] || (s_s[i] == s_s[e] && s_i[i] < s_i[e]))) ++rank;
        if (rank < k) { out_idx[(int64_t)q * k + rank] = s_i[e]; out_score[(int64_t)q * k + rank] = s_s[e]; }
    }
    int cnt = min(nvalid, k);
    if (tid == 0) out_count[q] = cnt;
    for (int t = cnt + tid; t < k; t += 256) { out_idx[(int64_t)q * k + t] = -1; out_score[(int64_t)q * k + t] = 0.0; }
}

// =========================================================================================
// 4b. cross-shard merge over peer memory: the all-gather and the merge in ONE kernel
// =========================================================================================
// Every rank has written its exact local lists [idx nq*k | score nq*k | count nq] into slot
// (gen & 1) of its own exchange buffer and then published `gen` in that buffer's flag word
// (p2p_publish_kernel, system-scope release).  This kernel -- one CTA per query -- waits until every
// peer's flag has reached `gen` (acquire loads over NVLink, bounded), pulls the peers' entries for its
// query with plain peer loads and ranks them.  Slot reuse two batches later is safe: a rank only
// reaches batch gen+2 after its merge of gen+1 saw every peer's flag gen+1, which each peer publishes
// after finishing its own merge of gen (stream order).
struct PeerPtrs { const unsigned char *p[16]; };

__global__ void p2p_publish_kernel(unsigned long long *flag, unsigned long long gen)
{
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(gen) : "memory");
}

__global__ void __launch_bounds__(256) merge_topk_p2p_kernel(PeerPtrs peers, int nranks, size_t slot_off, size_t flag_off,
                                                            unsigned long long gen, int nq, int k,
                                                            int64_t *__restrict__ out_idx, double *__restrict__ out_score,
                                                            int32_t *__restrict__ out_count)
{
    extern __shared__ unsigned char smem_raw[];
    const int q = blockIdx.x, tid = threadIdx.x;
    const int total = nranks * k;
    double *s_s = (double *)smem_raw;
    int64_t *s_i = (int64_t *)(s_s + total);
    int *s_v = (int *)(s_i + total);
    if (tid < nranks) {
        const unsigned long long *f = reinterpret_cast<const unsigned long long *>(peers.p[tid] + flag_off);
        unsigned long long v;
        const long long t0 = clock64();
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
            if (v >= gen) break;
            if (clock64() - t0 > 4000000000LL) { printf("vidmem: peer %d never published batch %llu\n", tid, gen); __trap(); }
        }
    }
    __syncthreads();
    for (int e = tid; e < total; e += 256) {
        const int l = e / k, j = e - l * k;
        const unsigned char *b = peers.p[l] + slot_off;
        const int64_t *idx = reinterpret_cast<const int64_t *>(b);
        const double *score = reinterpret_cast<const double *>(b + (size_t)nq * k * 8);
        const int32_t *count = reinterpret_cast<const int32_t *>(b + (size_t)nq * k * 16);
        const bool v = j < __ldcv(count + q);
        s_s[e] = v ? __ldcv(score + (size_t)q * k + j) : 0.0;
        s_i[e] = v ? __ldcv(idx + (size_t)q * k + j) : -1;
        s_v[e] = v ? 1 : 0;
    }
    __syncthreads();
    int nvalid = 0;
    for (int e = 0; e < total; ++e) nvalid += s_v[e];
    for (int e = tid; e < total; e += 256) {
        if (!s_v[e]) continue;
        int rank = 0;
        for (int i = 0; i < total; ++i)
            if (s_v[i] && (s_s[i] > s_s[e] || (s_s[i] == s_s[e] && s_i[i] < s_i[e]))) ++rank;
        if (rank < k) { out_idx[(int64_t)q * k + rank] = s_i[e]; out_score[(int64_t)q * k + rank] = s_s[e]; }
    }
    const int cnt = min(nvalid, k);
    if (tid == 0) out_count[q] = cnt;
    for (int t = cnt + tid; t < k; t += 256) { out_idx[(int64_t)q * k + t] = -1; out_score[(int64_t)q * k + t] = 0.0; }
}

// =========================================================================================
// 5. cross-query merge (pre_llm_injector.py:235-249): max score per id, stable sort desc, [:k2]
// =========================================================================================
__global__ void __launch_bounds__(256) merge_max_by_id_kernel(const int64_t *__restrict__ idx, const double *__restrict__ score,
                                                             const int32_t *__restrict__ count, int nq, int k, int k2,
                                                             int64_t *__restrict__ out_idx, double *__restrict__ out_score,
                                                             int32_t *__restrict__ out_count)
{
    extern __shared__ unsigned char smem_raw[];
    const int tid = threadIdx.x, total = nq * k;
    double *s_s = (double *)smem_raw;       // per entry: max score of its id (valid on representatives)
    int64_t *s_i = (int64_t *)(s_s + total);
    int *s_rep = (int *)(s_i + total);      // 1 = first occurrence of its id (dict insertion order)
    __shared__ int s_n;
    if (tid == 0) s_n = 0;
    for (int e = tid; e < total; e += 256) {
        int qi = e / k, j = e - qi * k;
        bool v = j < count[qi];
        s_i[e] = v ? idx[e] : -1;
        s_s[e] = v ? score[e] : 0.0;
        s_rep[e] = 0;
    }
    __syncthreads();
    for (int e = tid; e < total; e += 256) {
        if (s_i[e] < 0) continue;
        bool first = true;
        for (int i = 0; i < e; ++i)
            if (s_i[i] == s_i[e]) { first = false; break; }
        if (!first) continue;
        double m = s_s[e];
        for (int i = e + 1; i < total; ++i)
            if (s_i[i] == s_i[e] && score[i] > m) m = score[i];  // strict `>` replace == running max
        s_rep[e] = 1;
        // safe: only the representative writes its own slot, later entries read score[] (global)
        s_s[e] = m;
        atomicAdd(&s_n, 1);
    }
    __syncthreads();
    for (int e = tid; e < total; e += 256) {
        if (!s_rep[e]) continue;
        int rank = 0;
        for (int i = 0; i < total; ++i)
            if (s_rep[i] && (s_s[i] > s_s[e] || (s_s[i] == s_s[e] && i < e))) ++rank;  // stable: first seen wins ties
        if (rank < k2) { out_idx[rank] = s_i[e]; out_score[rank] = s_s[e]; }
    }
    if (tid == 0) *out_count = min(s_n, k2);
}

// =========================================================================================
// 6. scalar cosine seams (S2 / S4), one thread per pair
// =========================================================================================
template <bool NEUMAIER>
__global__ void cosine_pairs_kernel(const void *__restrict__ a, const void *__restrict__ b, int dtype, int64_t n, int dim,
                                    int zero_rule, double *__restrict__ out)
{
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    RefSum dot, aa, bb;
    dot.init(); aa.init(); bb.init();
    for (int c = 0; c < dim; ++c) {
        double x = load_as_double(a, dtype, i * dim + c), y = load_as_double(b, dtype, i * dim + c);
        dot.add<NEUMAIER>(__dmul_rn(x, y));
        aa.add<NEUMAIER>(__dmul_rn(x, x));
        bb.add<NEUMAIER>(__dmul_rn(y, y));
    }
    // zero_rule 2 = EmbeddingUtils.cosine_similarity (embedding_utils.py:29-39): magnitudes through `** 0.5`,
    // i.e. libm pow(x, 0.5) in CPython, here CUDA's pow (<= 2 ulp; not bit-pinned to a particular libm)
    double n1, n2;
    if (zero_rule == 2) { n1 = pow(aa.result<NEUMAIER>(), 0.5); n2 = pow(bb.result<NEUMAIER>(), 0.5); }
    else { n1 = __dsqrt_rn(aa.result<NEUMAIER>()); n2 = __dsqrt_rn(bb.result<NEUMAIER>()); }
    double den = __dmul_rn(n1, n2);
    bool zero = zero_rule == 1 ? (den == 0.0) : (n1 == 0.0 || n2 == 0.0);
    out[i] = zero ? 0.0 : __ddiv_rn(dot.result<NEUMAIER>(), den);
}

// ---- host wrappers ---------------------------------------------------------------------
int k_merge_candidates(const uint64_t *cand, int lists, int nq, int kp, uint64_t *merged, cudaStream_t st)
{
    size_t smem = (size_t)lists * kp * sizeof(uint64_t) + (size_t)lists * sizeof(uint32_t) + 16;
    VM_CUDA_CHECK((max_smem_once<merge_candidates_kernel>(200 * 1024)));
    VM_REQUIRE(smem <= 200 * 1024, VM_ERR_UNSUPPORTED, "candidate merge: %d lists x %d exceeds shared memory", lists, kp);
    merge_candidates_kernel<<<nq, MERGE_THREADS, smem, st>>>(cand, lists, nq, kp, merged);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}


// Calls f(neu) with neu a std::integral_constant<bool, Neumaier summation>, so f instantiates the matching
// <NEUMAIER> kernel.
template <typename F>
static int with_sum_mode(int sum_mode, F &&f)
{
    return sum_mode == VM_SUM_NEUMAIER ? f(std::true_type{}) : f(std::false_type{});
}

// Calls f(neu, (T *)nullptr) for the summation mode (as above) and the row type T of a row dtype.
template <typename F>
static int with_row_type(int dtype, int sum_mode, F &&f)
{
    auto by_sum = [&](auto *tag) { return with_sum_mode(sum_mode, [&](auto neu) { return f(neu, tag); }); };
    if (dtype == VM_F32) return by_sum((float *)nullptr);
    if (dtype == VM_F64) return by_sum((double *)nullptr);
    return by_sum((__nv_bfloat16 *)nullptr);
}

int k_rescore(const RescoreArgs &a, cudaStream_t st, const int *incomplete)
{
    // column chunk: whole rows when kp rows fit in RS_SMEM_ROW_BYTES, else a multiple of 8 columns
    const int ssz = a.dtype == VM_F64 ? 8 : 4;  // staged element size (StageOf)
    int chunk = RS_SMEM_ROW_BYTES / (ssz * a.kp) - 1;
    chunk &= ~7;
    if (chunk > a.ld) chunk = a.ld;
    const size_t smem = (size_t)chunk * sizeof(double) + (size_t)a.kp * (chunk + 1) * ssz + 16;
    return with_row_type(a.dtype, a.sum_mode, [&](auto neu, auto *tag) -> int {
        using T = std::remove_pointer_t<decltype(tag)>;
        constexpr bool NEU = decltype(neu)::value;
        VM_CUDA_CHECK((max_smem_once<rescore_kernel<NEU, T>>(160 * 1024)));
        rescore_kernel<NEU, T><<<a.nq, RS_THREADS, smem, st>>>(a.merged, a.kp, (const T *)a.rows, a.inv_norms, a.ld, a.dim,
                                                               a.n_rows, a.queries, a.q_dtype, a.eps, a.fin, a.flags,
                                                               a.uncertified_count, chunk, a.extreme, a.collect_thr, a.cum, incomplete);
        VM_CUDA_CHECK(cudaGetLastError());
        return VM_OK;
    });
}


// Fused path when the candidate keys + kp whole rows fit in shared memory; otherwise the caller falls
// back to k_merge_candidates + k_rescore.  Returns VM_ERR_UNSUPPORTED (without setting an error the
// caller must report) when it does not apply.
static constexpr size_t SR_SMEM_LIMIT = 180 * 1024;
// everything but the band scratch
static size_t select_rescore_base_smem(int key_cap, int lists, int kp, int dtype, int dim, int ld)
{
    const int es = (int)dtype_size(dtype);
    const size_t rows_area = (((size_t)kp * ((size_t)ld * es + 16) + 15) & ~(size_t)15) + 16;  // staged rows
    return (size_t)key_cap * 8 + (size_t)((lists + 3) & ~3) * 4 + (size_t)((dim + 1) & ~1) * 8 + rows_area + 32;
}
// band rows that fit next to it (0: not even BAND_CAP_MIN)
static int select_band_cap(int key_cap, int lists, int kp, int dtype, int dim, int ld)
{
    const size_t base = select_rescore_base_smem(key_cap, lists, kp, dtype, dim, ld);
    if (base + (size_t)BAND_CAP_MIN * 12 > SR_SMEM_LIMIT) return 0;
    size_t cap = (SR_SMEM_LIMIT - base) / 12;
    cap &= ~(size_t)63;
    if (cap > (size_t)BAND_CAP_MAX) cap = BAND_CAP_MAX;
    return (int)cap;
}
// lists == 0: slab mode (tcgen05 scan); else list mode with lists x list_len keys per query
bool select_rescore_fits(int lists, int list_len, int kp, int dtype, int dim, int ld)
{
    const int key_cap = lists > 0 ? lists * list_len : SELECT_KEY_CAP;
    return select_band_cap(key_cap, lists, kp, dtype, dim, ld) >= BAND_CAP_MIN && kp <= 64 && 2 * kp + 1 <= SR_THREADS;
}

static SelectSrc make_src(const SelectArgs &sa)
{
    const bool slab_mode = sa.slab != nullptr;
    const int lists = slab_mode ? 0 : sa.lists;
    return SelectSrc{sa.cand, lists, sa.list_len, sa.complete, sa.slab, sa.scnt, sa.ctas, sa.ubuf, sa.ucnt, sa.ucap, sa.seed_tab,
                     sa.nq_pad, sa.ksel, sa.band, slab_mode ? SELECT_KEY_CAP : lists * sa.list_len, 0};
}

int k_select_rescore(const SelectArgs &sa, const RescoreArgs &a, cudaStream_t st, bool pdl)
{
    SelectSrc src = make_src(sa);
    VM_REQUIRE(src.slab == nullptr || src.ctas <= 256, VM_ERR_UNSUPPORTED, "select: %d scan CTAs exceed 256", src.ctas);
    if (!select_rescore_fits(src.lists, src.list_len, a.kp, a.dtype, a.dim, a.ld)) return VM_ERR_UNSUPPORTED;
    src.band_cap = select_band_cap(src.key_cap, src.lists, a.kp, a.dtype, a.dim, a.ld);
    const size_t smem = select_rescore_base_smem(src.key_cap, src.lists, a.kp, a.dtype, a.dim, a.ld) + (size_t)src.band_cap * 12;
    return with_row_type(a.dtype, a.sum_mode, [&](auto neu, auto *tag) -> int {
        using T = std::remove_pointer_t<decltype(tag)>;
        constexpr bool NEU = decltype(neu)::value;
        VM_CUDA_CHECK((max_smem_once<select_rescore_kernel<NEU, T>>(180 * 1024)));
        VM_CUDA_CHECK(launch_pdl(select_rescore_kernel<NEU, T>, dim3(a.nq), dim3(SR_THREADS), smem, st, pdl, src, a.nq, a.kp,
                                 (const T *)a.rows, a.ld, a.dim, a.n_rows, a.queries, a.q_dtype, a.eps, a.fin, a.flags,
                                 a.uncertified_count, a.extreme, a.collect_thr, a.cum, a.inv_norms));
        VM_CUDA_CHECK(cudaGetLastError());
        return VM_OK;
    });
}

// slab-mode selection alone (rows too large for the fused kernel): merged [nq][kp], incomplete [nq]
int k_slab_top(const SelectArgs &sa, int nq, int kp, uint64_t *merged, int *incomplete, cudaStream_t st)
{
    const SelectSrc src = make_src(sa);
    VM_REQUIRE(src.slab != nullptr && src.ctas <= 256, VM_ERR_UNSUPPORTED, "slab selection: bad source");
    slab_top_kernel<<<nq, SR_THREADS, (size_t)src.key_cap * 8, st>>>(src, nq, kp, merged, incomplete);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_collect_rescore(const uint64_t *buf, const int *cnt, int cap, const RescoreArgs &a, cudaStream_t st)
{
    // staged route: scores + rows ids + 32 staged rows; global route (rows too wide): scores + norms + row ids
    const size_t head = (size_t)((a.dim + 1) & ~1) * 8;
    const size_t staged = head + (size_t)cap * 8 + (size_t)((cap + 3) & ~3) * 4 + (size_t)32 * ((size_t)a.ld * dtype_size(a.dtype) + 16) + 64;
    const int stage_rows = staged <= 200 * 1024 ? 32 : 0;
    const size_t smem = stage_rows ? staged : head + (size_t)cap * (8 + 8 + 4) + 32;
    VM_REQUIRE(smem <= 200 * 1024, VM_ERR_UNSUPPORTED, "collect pass: buffer of %d rows exceeds shared memory", cap);
    return with_row_type(a.dtype, a.sum_mode, [&](auto neu, auto *tag) -> int {
        using T = std::remove_pointer_t<decltype(tag)>;
        constexpr bool NEU = decltype(neu)::value;
        VM_CUDA_CHECK((max_smem_once<collect_rescore_kernel<NEU, T>>(200 * 1024)));
        collect_rescore_kernel<NEU, T><<<a.nq, CR_THREADS, smem, st>>>(buf, cnt, cap, (const T *)a.rows, a.ld, a.dim, a.queries,
                                                                       a.q_dtype, a.fin, a.flags, a.uncertified_count, a.nq, a.cum, stage_rows);
        VM_CUDA_CHECK(cudaGetLastError());
        return VM_OK;
    });
}

// a.flags == NULL: every query (VM_FLAG_FORCE_EXACT), scan + merge kernel.  a.flags != NULL: the conditional fix-up
// after a fast pass -- ONE launch (exits at once when nothing is flagged; otherwise the last CTA merges), optionally
// programmatically chained to the rescoring kernel.
int k_exact(const ExactArgs &a, cudaStream_t st, bool pdl)
{
    VM_REQUIRE((size_t)a.dim * sizeof(double) <= 40 * 1024, VM_ERR_UNSUPPORTED, "exact scan: dim %d too large", a.dim);
    const size_t smem = (size_t)((a.dim + 1) & ~1) * sizeof(double) + (size_t)3 * 128 * XS_PITCH + 16;  // query + three staged chunks
    const bool conditional = a.flags != nullptr && a.done_ctr != nullptr;
    const int rc = with_row_type(a.dtype, a.sum_mode, [&](auto neu, auto *tag) -> int {
        using T = std::remove_pointer_t<decltype(tag)>;
        constexpr bool NEU = decltype(neu)::value;
        VM_CUDA_CHECK((max_smem_once<exact_scan_kernel<NEU, T>>(200 * 1024)));
        VM_CUDA_CHECK(launch_pdl(exact_scan_kernel<NEU, T>, dim3(a.ctas), dim3(XS_THREADS), smem, st, pdl && conditional, (const T *)a.rows,
                                 a.inv_norms, a.n, a.ld, a.dim, a.queries, a.q_dtype, a.nq, a.flags, a.k, a.xlist_score, a.xlist_row,
                                 a.xlist_cnt, a.cum, conditional ? a.done_ctr : (int *)nullptr, a.fin, a.taken));
        VM_CUDA_CHECK(cudaGetLastError());
        return VM_OK;
    });
    if (rc != VM_OK || conditional) return rc;
    exact_merge_kernel<<<a.nq, 256, 0, st>>>(a.xlist_score, a.xlist_row, a.xlist_cnt, a.ctas, a.nq, a.k, a.flags, a.fin, a.taken);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_merge_topk_lists(const void *idx, const void *score, const void *count, size_t stride_bytes, int lists, int nq, int k,
                       int64_t *out_idx, double *out_score, int32_t *out_count, cudaStream_t st)
{
    int total = lists * k;
    VM_REQUIRE(total <= 4096, VM_ERR_UNSUPPORTED, "merge_topk_lists: lists*k = %d > 4096", total);
    size_t smem = (size_t)total * (8 + 8 + 4);
    VM_CUDA_CHECK((max_smem_once<merge_topk_lists_kernel>(100 * 1024)));
    merge_topk_lists_kernel<<<nq, 256, smem, st>>>((const char *)idx, (const char *)score, (const char *)count, stride_bytes, lists, nq, k,
                                                  out_idx, out_score, out_count);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_p2p_publish(void *flag, unsigned long long gen, cudaStream_t st)
{
    p2p_publish_kernel<<<1, 1, 0, st>>>((unsigned long long *)flag, gen);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_merge_topk_p2p(void *const *peers, int nranks, size_t slot_off, size_t flag_off, unsigned long long gen, int nq, int k,
                     int64_t *out_idx, double *out_score, int32_t *out_count, cudaStream_t st)
{
    VM_REQUIRE(nranks >= 1 && nranks <= 16, VM_ERR_UNSUPPORTED, "peer exchange supports up to 16 ranks");
    const int total = nranks * k;
    VM_REQUIRE(total <= 4096, VM_ERR_UNSUPPORTED, "merge: nranks*k = %d > 4096", total);
    PeerPtrs pp{};
    for (int r = 0; r < nranks; ++r) pp.p[r] = (const unsigned char *)peers[r];
    const size_t smem = (size_t)total * (8 + 8 + 4);
    VM_CUDA_CHECK((max_smem_once<merge_topk_p2p_kernel>(100 * 1024)));
    merge_topk_p2p_kernel<<<nq, 256, smem, st>>>(pp, nranks, slot_off, flag_off, gen, nq, k, out_idx, out_score, out_count);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_merge_max_by_id(const int64_t *idx, const double *score, const int32_t *count, int nq, int k, int k2,
                      int64_t *out_idx, double *out_score, int32_t *out_count, cudaStream_t st)
{
    int total = nq * k;
    VM_REQUIRE(total <= 4096, VM_ERR_UNSUPPORTED, "merge_max_by_id: nq*k = %d > 4096", total);
    size_t smem = (size_t)total * (8 + 8 + 4);
    VM_CUDA_CHECK((max_smem_once<merge_max_by_id_kernel>(100 * 1024)));
    merge_max_by_id_kernel<<<1, 256, smem, st>>>(idx, score, count, nq, k, k2, out_idx, out_score, out_count);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_cosine_pairs(const void *a, const void *b, int dtype, int64_t n, int dim, int zero_rule, int sum_mode, double *out,
                   cudaStream_t st)
{
    if (n <= 0) return VM_OK;
    int grid = (int)((n + 127) / 128);
    return with_sum_mode(sum_mode, [&](auto neu) -> int {
        cosine_pairs_kernel<decltype(neu)::value><<<grid, 128, 0, st>>>(a, b, dtype, n, dim, zero_rule, out);
        VM_CUDA_CHECK(cudaGetLastError());
        return VM_OK;
    });
}

}  // namespace vm
