// scan_simt.cu -- CUDA-core streaming scorer for small query batches (1..8 queries / pass).
//
// Bandwidth-bound: every store row is read exactly once per pass with 128-bit
// L1-bypassing loads; a warp takes 4 consecutive rows at a time, each lane owning 16-byte
// column chunks (coalesced 512 B per load instruction), the normalised queries sit in shared
// memory, and the 4 x QB partial dot products are reduced with a halving butterfly
// (V-1 shuffles for V values instead of 5V).  Fused epilogue: multiply by the cached 1/||row||,
// compare against the warp's running k-th key and insert into a warp-resident sorted list
// (one entry per lane, shfl_up insertion).  Per-warp lists are merged per CTA at the end and
// written as candidate keys; select.cu merges the CTAs and rescoring makes the result exact.
#include "common.cuh"

namespace vm {

static constexpr int SIMT_WARPS = 8;
static constexpr int SIMT_ROWS = 4;  // rows per warp step

__device__ __forceinline__ uint4 ldg_stream(const void *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// Butterfly reduction of V per-lane values across the warp.  While more than one value is
// left, lanes with (lane & S) keep the upper half and send the lower half (and vice versa), so
// each step halves the live values; afterwards plain xor all-reduce steps.  The value a lane
// ends with has index owner_index<V>(lane); lanes sharing that index all hold the full sum.
template <int CUR, int S>
__device__ __forceinline__ void bfly(float *v, int lane)
{
    if constexpr (S >= 1) {
        if constexpr (CUR > 1) {
            constexpr int H = CUR / 2;
            const bool up = (lane & S) != 0;
#pragma unroll
            for (int i = 0; i < H; ++i) {
                float send = up ? v[i] : v[i + H];
                float keep = up ? v[i + H] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, S);
            }
            bfly<H, S / 2>(v, lane);
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], S);
            bfly<1, S / 2>(v, lane);
        }
    }
}
template <int V>
__device__ __forceinline__ int owner_index(int lane)
{
    int idx = 0, half = V / 2, s = 16;
    while (half >= 1) {
        if (lane & s) idx += half;
        half >>= 1;
        s >>= 1;
    }
    return idx;
}

template <typename T> struct Chunk;
template <> struct Chunk<float> {
    static constexpr int N = 4;
    __device__ static __forceinline__ void unpack(const uint4 &u, float *f)
    {
        f[0] = __uint_as_float(u.x); f[1] = __uint_as_float(u.y); f[2] = __uint_as_float(u.z); f[3] = __uint_as_float(u.w);
    }
};
template <> struct Chunk<__nv_bfloat16> {
    static constexpr int N = 8;
    __device__ static __forceinline__ void unpack(const uint4 &u, float *f)
    {
        f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xffff0000u);
        f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xffff0000u);
        f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xffff0000u);
        f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xffff0000u);
    }
};

// warp-sorted insert of key k into `mine` (entry `lane` of a descending list)
__device__ __forceinline__ uint64_t warp_insert(uint64_t mine, uint64_t k, int lane)
{
    uint64_t up = __shfl_up_sync(0xffffffffu, mine, 1);
    bool gt = k > mine;
    bool gt_up = lane > 0 && k > up;
    return gt ? (gt_up ? up : k) : mine;
}

template <typename T, int QB>
__global__ void __launch_bounds__(SIMT_WARPS * 32, 2)
scan_simt_kernel(const T *__restrict__ rows, const float *__restrict__ inv_norms, int64_t n, int ld,
                 const float *__restrict__ queries, int q0, int nq_total, int kp, uint64_t *__restrict__ cand)
{
    constexpr int CN = Chunk<T>::N;
    constexpr int V = SIMT_ROWS * QB;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *sq = reinterpret_cast<float *>(smem_raw);                                  // [QB][ld]
    uint64_t *sl = reinterpret_cast<uint64_t *>(smem_raw + (size_t)QB * ld * 4);      // [WARPS][QB][32]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = tid; e < QB * ld; e += SIMT_WARPS * 32) {
        int q = e / ld;
        sq[e] = (q0 + q < nq_total) ? queries[(int64_t)(q0 + q) * ld + (e - q * ld)] : 0.0f;
    }
    __syncthreads();

    uint64_t list[QB], tau[QB];
#pragma unroll
    for (int q = 0; q < QB; ++q) { list[q] = 0; tau[q] = 0; }

    const int nchunks = ld / CN;
    const int my_idx = owner_index<V>(lane);
    const int my_r = my_idx / QB, my_q = my_idx % QB;
    const bool rep = (lane & ((32 / V) - 1)) == 0 || V >= 32;
    const int64_t gwarp = (int64_t)blockIdx.x * SIMT_WARPS + warp;
    const int64_t gstride = (int64_t)gridDim.x * SIMT_WARPS * SIMT_ROWS;

    for (int64_t row0 = gwarp * SIMT_ROWS; row0 < n; row0 += gstride) {
        float acc[V];
#pragma unroll
        for (int i = 0; i < V; ++i) acc[i] = 0.0f;
        const T *rp[SIMT_ROWS];
#pragma unroll
        for (int r = 0; r < SIMT_ROWS; ++r) {
            int64_t rr = row0 + r < n ? row0 + r : n - 1;  // clamp (masked below)
            rp[r] = rows + rr * (int64_t)ld;
        }
        // prefetch this lane's inverse norm early
        int64_t myrow = row0 + my_r;
        float inv = (myrow < n) ? __ldg(inv_norms + myrow) : -1.0f;
#pragma unroll 2
        for (int c = lane; c < nchunks; c += 32) {
            uint4 u[SIMT_ROWS];
#pragma unroll
            for (int r = 0; r < SIMT_ROWS; ++r) u[r] = ldg_stream(rp[r] + (int64_t)c * CN);
            float f[SIMT_ROWS][CN];
#pragma unroll
            for (int r = 0; r < SIMT_ROWS; ++r) Chunk<T>::unpack(u[r], f[r]);
#pragma unroll
            for (int q = 0; q < QB; ++q) {
                const float4 *qp = reinterpret_cast<const float4 *>(sq + (size_t)q * ld + (size_t)c * CN);
                float qa[CN];
                float4 t0 = qp[0];
                qa[0] = t0.x; qa[1] = t0.y; qa[2] = t0.z; qa[3] = t0.w;
                if constexpr (CN == 8) {
                    float4 t1 = qp[1];
                    qa[4] = t1.x; qa[5] = t1.y; qa[6] = t1.z; qa[7] = t1.w;
                }
#pragma unroll
                for (int r = 0; r < SIMT_ROWS; ++r)
#pragma unroll
                    for (int e = 0; e < CN; ++e) acc[r * QB + q] = fmaf(f[r][e], qa[e], acc[r * QB + q]);
            }
        }
        bfly<V, 16>(acc, lane);
        float score = acc[0] * inv;
        bool hit = rep && inv >= 0.0f;  // inv < 0: row beyond n or skipped row
        uint64_t key = make_key(score, (uint32_t)myrow);
        // per-lane query differs: select my tau without dynamic register indexing
        uint64_t mytau = 0;
#pragma unroll
        for (int q = 0; q < QB; ++q) mytau = (q == my_q) ? tau[q] : mytau;
        hit = hit && key > mytau;
        unsigned m = __ballot_sync(0xffffffffu, hit);
        while (m) {
            int src = __ffs(m) - 1;
            m &= m - 1;
            uint64_t k = __shfl_sync(0xffffffffu, key, src);
            int qq = owner_index<V>(src) % QB;
#pragma unroll
            for (int q = 0; q < QB; ++q) {
                if (q == qq && k > tau[q]) {  // warp-uniform
                    list[q] = warp_insert(list[q], k, lane);
                    tau[q] = __shfl_sync(0xffffffffu, list[q], kp - 1);
                }
            }
        }
    }

    // ---- CTA merge: warp q merges the SIMT_WARPS lists of query q -------------------------
#pragma unroll
    for (int q = 0; q < QB; ++q) sl[((size_t)warp * QB + q) * 32 + lane] = lane < kp ? list[q] : 0;
    __syncthreads();
    if (warp < QB && q0 + warp < nq_total) {
        const int q = warp;
        uint64_t mine = sl[(size_t)q * 32 + lane];  // warp 0's list as the base
        uint64_t t = __shfl_sync(0xffffffffu, mine, kp - 1);
        for (int w = 1; w < SIMT_WARPS; ++w) {
            for (int j = 0; j < kp; ++j) {
                uint64_t k = sl[((size_t)w * QB + q) * 32 + j];
                if (k <= t) break;  // lists are descending: nothing further can enter
                mine = warp_insert(mine, k, lane);
                t = __shfl_sync(0xffffffffu, mine, kp - 1);
            }
        }
        if (lane < kp) cand[((int64_t)blockIdx.x * nq_total + (q0 + q)) * kp + lane] = mine;
    }
}

int scan_simt_max_queries() { return 8; }

template <typename T, int QB>
static int launch_one(const ScanArgs &a, int q0)
{
    size_t smem = (size_t)QB * a.ld * 4 + (size_t)SIMT_WARPS * QB * 32 * 8;
    VM_REQUIRE(smem <= 160 * 1024, VM_ERR_UNSUPPORTED, "SIMT scan: dim %d too large for %d queries per pass", a.dim, QB);
    VM_CUDA_CHECK((max_smem_once<scan_simt_kernel<T, QB>>(160 * 1024)));
    scan_simt_kernel<T, QB><<<a.ctas, SIMT_WARPS * 32, smem, a.stream>>>((const T *)a.rows, a.inv_norms, a.n, a.ld, a.queries, q0,
                                                                         a.nq, a.kp, a.cand);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

// Scans all a.nq queries (8 per pass).  cand must hold [a.ctas][a.nq][a.kp] keys.
int launch_scan_simt(const ScanArgs &a)
{
    VM_REQUIRE(a.kp >= 1 && a.kp <= 32, VM_ERR_UNSUPPORTED, "SIMT scan: candidate list %d > 32", a.kp);
    VM_REQUIRE(a.n < 0xFFFFFFFFLL, VM_ERR_UNSUPPORTED, "shard has more than 2^32-2 rows");
    for (int q0 = 0; q0 < a.nq; q0 += 8) {
        int rem = a.nq - q0;
        int rc;
#define DISPATCH(QB)                                                            \
    rc = a.dtype == VM_F32 ? launch_one<float, QB>(a, q0) : launch_one<__nv_bfloat16, QB>(a, q0)
        if (rem >= 5) DISPATCH(8);
        else if (rem >= 3) DISPATCH(4);
        else if (rem == 2) DISPATCH(2);
        else DISPATCH(1);
#undef DISPATCH
        if (rc != VM_OK) return rc;
    }
    return VM_OK;
}

}  // namespace vm
