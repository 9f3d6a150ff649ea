// pairs.cu -- all-pairs cosine threshold scorer (entity / relation dedup): every (i, j), i < j,
// with cosine(x_i, x_j) > threshold.  Replaces Graph._are_same_context (src/pipeline/prune.py:67-79:
// S = cosine_similarity(E); fill_diagonal(S, 0); S > threshold) generalised to the pair set.
//
// A genuine dense contraction -> tcgen05 tensor cores (bf16 x bf16 -> fp32 in TMEM; kind::tf32 for
// fp32 rows).  The N x N score matrix (4 TB at N = 1M) never exists: each 128 x 256 accumulator tile
// is consumed straight out of TMEM by the epilogue, which applies the cached inverse norms, compares
// against the threshold and appends the (rare) hits with one atomic each.  Only tiles that touch the
// strict upper triangle are scheduled; tiles are rasterised in groups of 8 (64 from 2^18 rows) column blocks x all
// row blocks so that the group's column panel stays in L2 while the row panels stream; the CTA pairs keep pace with each
// other through a launch-wide step counter (pairs_keep_pace) so that a row block is fetched from DRAM once per group.
//
// Persistent, warp-specialised (192 threads): warp 0 TMA producer (A 128-row box + B 256-row box per
// 128-byte K block, 4 stages of 48 KB), warp 1 MMA issuer (M=128, N=256, 4 MMAs per stage, 2
// accumulator stages = all 512 TMEM columns), warps 2-5 epilogue.
// Pairs whose fp32 score lies within eps of the threshold are re-decided in binary64 by
// pairs_finalize_kernel, so the emitted pair SET is exact for the stored values.
#include "tc_common.cuh"
#include "raster.h"
#include "scan_eps.h"
#include <stdlib.h>
#include <mutex>

namespace vm {
using namespace tc;

static constexpr int P_BM = 128, P_BN = 256;
static constexpr int P_STAGES = 4, P_ACC = 2, P_THREADS = 192;
static constexpr int P_A_BYTES = P_BM * 128, P_B_BYTES = P_BN * 128, P_STAGE_BYTES = P_A_BYTES + P_B_BYTES;
// Column blocks (of 256 rows) per raster group, chosen per call (PairsParams::gj_log2).  All CTAs work inside one group at
// a time: its column panel stays in L2 while the row blocks stream, so a row block is re-read from DRAM once per GROUP.
// 8 blocks (2 048 rows, 3 MB at D=768) were the round-1 choice; at 1 M rows that is 488 groups = 375 GB of DRAM reads
// per pass, and the kernel runs under the power cap, where DRAM energy costs SM clock.  64 blocks (16 384 rows, 25 MB of
// the 126 MB L2) cut the re-reads 8x: 1 M x 768 bf16 717 -> 619 ms (SM clock under the cap 1.01 -> 1.34 GHz); 128 blocks
// 639 ms, 256 blocks (100 MB: no longer L2 resident) 735 ms.  Below 2^18 rows the narrow groups are kept (few groups
// either way; measured equal within run-to-run noise).
static constexpr int P_GJ_LOG2_SMALL = 3, P_GJ_LOG2_LARGE = 6;
// L2 eviction priority of the streamed row blocks (A) and of the group's column panel (B); A/B builds override them.
// Plain priority for both: with the pairs kept together (pairs_keep_pace) ordinary LRU already holds the panel and the
// one or two live row blocks -- measured at 1 M x 768: 49 GB of DRAM reads per pass (the raster's minimum: 62 groups x
// half the operand) against 100 GB with evict-first rows / evict-last panel, same run time.
#ifndef VM_PAIRS_HINT_A
#define VM_PAIRS_HINT_A L2_EVICT_NORMAL
#endif
#ifndef VM_PAIRS_HINT_B
#define VM_PAIRS_HINT_B L2_EVICT_NORMAL
#endif
static constexpr int64_t P_GJ_LARGE_FROM_ROWS = 1 << 18;

struct PairsParams {
    int64_t n;
    int nbi, nbj, KB;
    float thr, thr_lo;        // threshold, threshold - eps
    const float *inv;         // [n] 1/||row||, 0 for a zero row
    int32_t *st_i, *st_j;     // staging: every pair with approx score > thr_lo
    float *st_s;
    unsigned long long *st_cnt;
    long long st_cap;
    long long total_tiles;
    int part, nparts;
    int gj_log2;              // log2(column blocks per raster group)
    int groups;               // raster groups
    unsigned long long *prog; // tile-sequence steps issued by all CTA pairs of this launch (pace keeping, see pairs_keep_pace)
};

template <bool TF32>
__global__ void __launch_bounds__(P_THREADS, 1)
pairs_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, PairsParams p)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint8_t *base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *stages = base;                                                   // [P_STAGES][A 16K | B 32K]
    float *sinv = reinterpret_cast<float *>(base + P_STAGES * P_STAGE_BYTES);  // [P_ACC][256]
    uint64_t *bars = reinterpret_cast<uint64_t *>(sinv + P_ACC * P_BN);
    uint64_t *full = bars, *empty = bars + P_STAGES, *tfull = empty + P_STAGES, *tempty = tfull + P_ACC;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + P_ACC);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    constexpr int ELEMS = TF32 ? 32 : 64;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < P_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int a = 0; a < P_ACC; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // tile sequence of this CTA: u = blockIdx.x, blockIdx.x + gridDim.x, ... ; t = u * nparts + part
    auto valid_tile = [&](int bi, int bj) {
        return bi < p.nbi && bj < p.nbj && ((long long)bj * P_BN + P_BN - 1 > (long long)bi * P_BM);
    };

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            TileIter<2> ti;
            for (ti.init(blockIdx.x, gridDim.x, p.groups, p.gj_log2, p.part, p.nparts); ti.valid(); ti.next()) {
                const int bi = ti.bi(), bj = ti.bj();
                if (!valid_tile(bi, bj)) continue;
                for (int kb = 0; kb < p.KB; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full[stage], P_STAGE_BYTES);
                    uint8_t *sa = stages + (size_t)stage * P_STAGE_BYTES;
                    tma_load_2d(&tmA, &full[stage], sa, kb * ELEMS, bi * P_BM, L2_EVICT_FIRST);
                    tma_load_2d(&tmB, &full[stage], sa + P_A_BYTES, kb * ELEMS, bj * P_BN, L2_EVICT_LAST);
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc(TF32 ? 2u : 1u, P_BM, P_BN);
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            const uint32_t s0 = smem_u32(stages);
            TileIter<2> ti;
            for (ti.init(blockIdx.x, gridDim.x, p.groups, p.gj_log2, p.part, p.nparts); ti.valid(); ti.next()) {
                const int bi = ti.bi(), bj = ti.bj();
                if (!valid_tile(bi, bj)) continue;
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * P_BN);
                for (int kb = 0; kb < p.KB; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = s0 + (uint32_t)stage * P_STAGE_BYTES;
                    const uint32_t b_addr = a_addr + P_A_BYTES;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        umma<TF32>(d_tmem, make_smem_desc_sw128(a_addr + j * 32), make_smem_desc_sw128(b_addr + j * 32), idesc,
                                   (uint32_t)((kb | j) != 0));
                    umma_commit(&empty[stage]);
                    if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tfull[acc]);
                if (++acc == P_ACC) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int e = threadIdx.x - 64;  // 0..127
        const int quad = warp & 3;
        const int row_in_tile = quad * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        TileIter<2> ti;
        for (ti.init(blockIdx.x, gridDim.x, p.groups, p.gj_log2, p.part, p.nparts); ti.valid(); ti.next()) {
            const int bi = ti.bi(), bj = ti.bj();
            if (!valid_tile(bi, bj)) continue;
            const long long i = (long long)bi * P_BM + row_in_tile;
            const long long j0 = (long long)bj * P_BN;
            const float inv_i = i < p.n ? __ldg(p.inv + i) : -1.0f;
            // columns' inverse norms for this tile (2 per epilogue thread)
            float *sj = sinv + acc * P_BN;
            for (int c = e; c < P_BN; c += 128) sj[c] = (j0 + c < p.n) ? __ldg(p.inv + j0 + c) : 0.0f;
            // pre-filter threshold on acc * inv_j: (thr_lo / inv_i) nudged down so rounding cannot lose a pair
            float thr_i;
            if (inv_i > 0.0f) thr_i = p.thr_lo / inv_i, thr_i -= fabsf(thr_i) * 1e-6f;
            else thr_i = (inv_i == 0.0f && 0.0f > p.thr_lo) ? -INFINITY : INFINITY;
            named_bar_sync(1, 128);  // sj visible
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * P_BN);
#pragma unroll 1
            for (int c = 0; c < P_BN; c += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + c, v);
                float w[32];
#pragma unroll
                for (int q4 = 0; q4 < 8; ++q4) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(sj + c + 4 * q4);
                    w[4 * q4] = t4.x; w[4 * q4 + 1] = t4.y; w[4 * q4 + 2] = t4.z; w[4 * q4 + 3] = t4.w;
                }
                tmem_ld_wait();
                uint32_t hits = 0;
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) hits |= (__uint_as_float(v[jj]) * w[jj] > thr_i) ? (1u << jj) : 0u;
                while (hits) {  // rare
                    const int jj = __ffs(hits) - 1;
                    hits &= hits - 1;
                    float a = 0.0f, wj = 0.0f;
#pragma unroll
                    for (int x = 0; x < 32; ++x) { a = (x == jj) ? __uint_as_float(v[x]) : a; wj = (x == jj) ? w[x] : wj; }
                    const long long j = j0 + c + jj;
                    const float s = a * wj * inv_i;
                    if (j < p.n && j > i && s > p.thr_lo) {
                        const unsigned long long pos = atomicAdd(p.st_cnt, 1ull);
                        if ((long long)pos < p.st_cap) { p.st_i[pos] = (int32_t)i; p.st_j[pos] = (int32_t)j; p.st_s[pos] = s; }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            if (++acc == P_ACC) { acc = 0; acc_phase ^= 1; }
            // sj[acc] is refilled two tiles later, behind the next tile's barrier: no extra sync needed
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// =========================================================================================
// 2-CTA variant: a CTA pair (cluster of 2) computes one 256 x 256 tile with tcgen05.mma.cta_group::2.
// Each CTA stages only 128 rows of A and HALF of B per K block (32 KB instead of 48 KB) and the
// tensor core reads B from both shared memories, so shared-memory traffic per SM drops from
// ~192 B/cycle (the 1-CTA kernel's limiter) to ~128 B/cycle at full MMA rate.
// =========================================================================================
static constexpr int P2_STAGES = 6, P2_STAGE_BYTES = 2 * P_A_BYTES;

// Pace keeping.  The tile sequence is dealt to the CTA pairs statically (pair p takes steps p, p + npairs, ...), and the L2
// reuse of the raster rests on all pairs working on the SAME one or two row blocks of the current group: a row block is
// fetched from DRAM once and then read by the 64 pairs that score it against the group's 64 column blocks.  Nothing kept
// the pairs together, and over a 0.7 s launch (1 M rows: ~10^5 tiles per pair) they drift apart -- ncu at 1 M rows: L2 hit
// rate 60 %, 2.1 TB of DRAM reads (1 400 x the operand; 96 % and 26 x at 262 144 rows), i.e. most row-block loads missed.
// Every MMA thread now counts its sequence steps into one global counter, and a producer that is more than `window` steps
// ahead of the launch-wide count waits for the others -- softly: after ~16 us it goes on regardless, so pairs that are not
// resident yet (another kernel holding SMs) can never block the ones that are.
__device__ __forceinline__ void pairs_keep_pace(const unsigned long long *prog, long long my_step, long long window)
{
    if (my_step <= window) return;
    for (int spin = 0; spin < 64; ++spin) {
        unsigned long long done;
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(done) : "l"(prog) : "memory");
        if ((long long)done + window >= my_step) return;
        __nanosleep(256);
    }
}

template <bool TF32>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(P_THREADS, 1)
pairs_tc2_kernel(const __grid_constant__ CUtensorMap tmA, PairsParams p)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint8_t *base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *stages = base;                                                     // [P2_STAGES][A 16K | B-half 16K]
    float *sinv = reinterpret_cast<float *>(base + P2_STAGES * P2_STAGE_BYTES);  // [P_ACC][256]
    uint64_t *bars = reinterpret_cast<uint64_t *>(sinv + P_ACC * P_BN);
    uint64_t *full = bars, *empty = bars + P2_STAGES, *tfull = empty + P2_STAGES, *tempty = tfull + P_ACC;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty + P_ACC);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();  // 0 = leader
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    constexpr int ELEMS = TF32 ? 32 : 64;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        for (int s = 0; s < P2_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int a = 0; a < P_ACC; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 8); }  // 4 local + 4 peer warps
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc_2sm(tmem_slot, 512);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int nb = (int)((p.n + 255) / 256);  // 256-row blocks (rows and columns)

    auto valid_tile = [&](int bi, int bj) { return bi < nb && bj < nb && bj >= bi; };

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            TileIter<1> ti;
            long long step = 0;                                  // sequence steps of this pair so far (valid or not)
            const long long window = 4ll * npairs;
            for (ti.init(pair, npairs, p.groups, p.gj_log2, p.part, p.nparts); ti.valid(); ti.next(), ++step) {
                const int bi = ti.bi(), bj = ti.bj();
                if (!valid_tile(bi, bj)) continue;
                if (rank == 0) pairs_keep_pace(p.prog, step * npairs, window);   // the peer follows through the stage barriers
                for (int kb = 0; kb < p.KB; ++kb) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * P2_STAGE_BYTES);  // both CTAs' bytes
                    uint8_t *sa = stages + (size_t)stage * P2_STAGE_BYTES;
                    tma_load_2d_2sm(&tmA, &full[stage], sa, kb * ELEMS, bi * 256 + (int)rank * 128, VM_PAIRS_HINT_A);
                    tma_load_2d_2sm(&tmA, &full[stage], sa + P_A_BYTES, kb * ELEMS, bj * 256 + (int)rank * 128, VM_PAIRS_HINT_B);
                    if (++stage == P2_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            const uint32_t idesc = make_idesc(TF32 ? 2u : 1u, 256, 256);
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            const uint32_t s0 = smem_u32(stages);
            TileIter<1> ti;
            for (ti.init(pair, npairs, p.groups, p.gj_log2, p.part, p.nparts); ti.valid(); ti.next()) {
                const int bi = ti.bi(), bj = ti.bj();
                atomicAdd(p.prog, 1ull);                         // one per sequence step, valid or not (pairs_keep_pace)
                if (!valid_tile(bi, bj)) continue;
                mbar_wait(&tempty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * P_BN);
                for (int kb = 0; kb < p.KB; ++kb) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t a_addr = s0 + (uint32_t)stage * P2_STAGE_BYTES;
                    const uint32_t b_addr = a_addr + P_A_BYTES;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        umma_2sm<TF32>(d_tmem, make_smem_desc_sw128(a_addr + j * 32), make_smem_desc_sw128(b_addr + j * 32), idesc,
                                       (uint32_t)((kb | j) != 0));
                    umma_commit_2sm(&empty[stage]);  // frees the stage in both CTAs
                    if (++stage == P2_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit_2sm(&tfull[acc]);        // accumulator ready in both CTAs
                if (++acc == P_ACC) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int e = threadIdx.x - 64;  // 0..127
        const int quad = warp & 3;
        const int row_in_tile = quad * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        TileIter<1> ti;
        for (ti.init(pair, npairs, p.groups, p.gj_log2, p.part, p.nparts); ti.valid(); ti.next()) {
            const int bi = ti.bi(), bj = ti.bj();
            if (!valid_tile(bi, bj)) continue;
            const long long i = (long long)bi * 256 + rank * 128 + row_in_tile;
            const long long j0 = (long long)bj * 256;
            const float inv_i = i < p.n ? __ldg(p.inv + i) : -1.0f;
            float *sj = sinv + acc * P_BN;
            for (int c = e; c < P_BN; c += 128) sj[c] = (j0 + c < p.n) ? __ldg(p.inv + j0 + c) : 0.0f;
            float thr_i;
            if (inv_i > 0.0f) thr_i = p.thr_lo / inv_i, thr_i -= fabsf(thr_i) * 1e-6f;
            else thr_i = (inv_i == 0.0f && 0.0f > p.thr_lo) ? -INFINITY : INFINITY;
            named_bar_sync(1, 128);
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * P_BN);
#pragma unroll 1
            for (int c = 0; c < P_BN; c += 32) {
                uint32_t v[32];
                tmem_ld32(taddr + c, v);
                float w[32];
#pragma unroll
                for (int q4 = 0; q4 < 8; ++q4) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(sj + c + 4 * q4);
                    w[4 * q4] = t4.x; w[4 * q4 + 1] = t4.y; w[4 * q4 + 2] = t4.z; w[4 * q4 + 3] = t4.w;
                }
                tmem_ld_wait();
                uint32_t hits = 0;
#pragma unroll
                for (int jj = 0; jj < 32; ++jj) hits |= (__uint_as_float(v[jj]) * w[jj] > thr_i) ? (1u << jj) : 0u;
                while (hits) {  // rare
                    const int jj = __ffs(hits) - 1;
                    hits &= hits - 1;
                    float a = 0.0f, wj = 0.0f;
#pragma unroll
                    for (int x = 0; x < 32; ++x) { a = (x == jj) ? __uint_as_float(v[x]) : a; wj = (x == jj) ? w[x] : wj; }
                    const long long j = j0 + c + jj;
                    const float s = a * wj * inv_i;
                    if (j < p.n && j > i && s > p.thr_lo) {
                        const unsigned long long pos = atomicAdd(p.st_cnt, 1ull);
                        if ((long long)pos < p.st_cap) { p.st_i[pos] = (int32_t)i; p.st_j[pos] = (int32_t)j; p.st_s[pos] = s; }
                    }
                }
            }
            // hand the accumulator stage back to the leader's MMA thread (local or remote arrive)
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (rank == 0) mbar_arrive(&tempty[acc]);
                else mbar_arrive_remote(&tempty[acc], 0);
            }
            if (++acc == P_ACC) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, 512);
    }
}

// Staged pairs -> output.  Pairs within eps of the threshold are re-decided with a binary64
// cosine (index-order sums) on the stored values; the rest are kept as they are.
template <typename T>
__global__ void pairs_finalize_kernel(const T *__restrict__ x, int ld, int dim, float thr, float eps,
                                      const int32_t *__restrict__ st_i, const int32_t *__restrict__ st_j,
                                      const float *__restrict__ st_s, const unsigned long long *__restrict__ st_cnt,
                                      long long st_cap, int64_t *__restrict__ out_i, int64_t *__restrict__ out_j,
                                      float *__restrict__ out_s, unsigned long long *__restrict__ out_cnt, long long cap)
{
    const unsigned long long staged = *st_cnt;
    const long long m = (long long)(staged < (unsigned long long)st_cap ? staged : (unsigned long long)st_cap);
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < m; e += (long long)gridDim.x * blockDim.x) {
        const int i = st_i[e], j = st_j[e];
        float s = st_s[e];
        bool keep = s > thr;
        if (fabsf(s - thr) <= eps) {
            const T *a = x + (int64_t)i * ld, *b = x + (int64_t)j * ld;
            double dot = 0.0, aa = 0.0, bb = 0.0;
            for (int c = 0; c < dim; ++c) {
                const double u = (double)load_as_float(a, c), v = (double)load_as_float(b, c);
                dot += u * v; aa += u * u; bb += v * v;
            }
            const double den = sqrt(aa) * sqrt(bb);
            const double ex = den > 0.0 ? dot / den : 0.0;
            keep = ex > (double)thr;
            s = (float)ex;
        }
        if (keep) {
            const unsigned long long pos = atomicAdd(out_cnt, 1ull);
            if ((long long)pos < cap) { out_i[pos] = i; out_j[pos] = j; out_s[pos] = s; }
        }
    }
    // staging overflow: report at least the staged count so the caller sees count > cap
    if (blockIdx.x == 0 && threadIdx.x == 0 && staged > (unsigned long long)st_cap) atomicMax(out_cnt, staged);
}

// Multi-GPU concatenation: `gathered` holds, per rank r, [i slot*8 | j slot*8 | s slot*4] at r * per_rank_bytes with
// counts[r] valid entries; they are packed in rank order into out_* (capacity cap) and *out_count = sum of counts.
__global__ void pairs_concat_kernel(const char *__restrict__ gathered, size_t per_rank_bytes, long long slot,
                                    const long long *__restrict__ counts, int nranks, long long cap, int64_t *__restrict__ out_i,
                                    int64_t *__restrict__ out_j, float *__restrict__ out_s, long long *__restrict__ out_count)
{
    const int r = blockIdx.y;
    long long off = 0, total = 0;
    for (int q = 0; q < nranks; ++q) { if (q < r) off += counts[q]; total += counts[q]; }
    const long long m = counts[r] < slot ? counts[r] : slot;
    const char *b = gathered + (size_t)r * per_rank_bytes;
    const int64_t *gi = reinterpret_cast<const int64_t *>(b), *gj = reinterpret_cast<const int64_t *>(b + (size_t)slot * 8);
    const float *gs = reinterpret_cast<const float *>(b + (size_t)slot * 16);
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < m; e += (long long)gridDim.x * blockDim.x)
        if (off + e < cap) { out_i[off + e] = gi[e]; out_j[off + e] = gj[e]; out_s[off + e] = gs[e]; }
    if (r == 0 && blockIdx.x == 0 && threadIdx.x == 0) *out_count = total;
}

int k_pairs_concat(const void *gathered, size_t per_rank_bytes, int64_t slot, const int64_t *counts, int nranks, int64_t cap,
                   int64_t *out_i, int64_t *out_j, float *out_score, int64_t *out_count, cudaStream_t st)
{
    dim3 grid((unsigned)imin64((slot + 255) / 256, 256), (unsigned)nranks);
    pairs_concat_kernel<<<grid, 256, 0, st>>>((const char *)gathered, per_rank_bytes, (long long)slot, (const long long *)counts, nranks,
                                             (long long)cap, out_i, out_j, out_score, (long long *)out_count);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

int k_row_inv_norms(const void *rows, int dtype, float *inv_norms, int64_t row0, int64_t n, int ld, int *extreme, cudaStream_t st,
                    const double *exact = nullptr);

namespace {
// Scratch of one (device, stream): calls on different streams of a device -- from different host threads too -- never
// share buffers; calls on the same stream reuse them in stream order.
struct PairsWs {
    void *inv = nullptr, *st_i = nullptr, *st_j = nullptr, *st_s = nullptr, *cnt = nullptr;
    size_t inv_bytes = 0, st_entries = 0;
    cudaStream_t stream = nullptr;
    bool used = false;
};
constexpr int PWS_STREAMS = 8;
PairsWs g_pws[16][PWS_STREAMS];
std::mutex g_pws_mu;
PairsWs *pairs_ws(int device, cudaStream_t st)
{
    std::lock_guard<std::mutex> lock(g_pws_mu);
    PairsWs *free_slot = nullptr;
    for (PairsWs &w : g_pws[device]) {
        if (w.used && w.stream == st) return &w;
        if (!w.used && !free_slot) free_slot = &w;
    }
    if (free_slot) { free_slot->used = true; free_slot->stream = st; }
    return free_slot;
}
int ensure(void **p, size_t *have, size_t need)
{
    if (need <= *have) return VM_OK;
    if (*p) cudaFree(*p);
    *p = nullptr; *have = 0;
    cudaError_t e = cudaMalloc(p, need);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e)); return VM_ERR_OOM; }
    *have = need;
    return VM_OK;
}
}  // namespace

int k_pairs_above(int device, const void *x, int dtype, int64_t n, int dim, int ld, float threshold, int64_t cap,
                  int64_t *out_i, int64_t *out_j, float *out_score, int64_t *out_count, int part, int nparts, int flags,
                  cudaStream_t st)
{
    (void)flags;
    VM_REQUIRE(device >= 0 && device < 16, VM_ERR_BADARG, "device index %d outside [0, 16)", device);
    VM_CUDA_CHECK(cudaMemsetAsync(out_count, 0, 8, st));
    if (n <= 1) return VM_OK;  // prune.py:73-74
    VM_REQUIRE(((uintptr_t)x & 127) == 0, VM_ERR_BADARG, "rows buffer must be 128-byte aligned");
    PairsWs *wp = pairs_ws(device, st);
    VM_REQUIRE(wp, VM_ERR_UNSUPPORTED, "all-pairs scorer: more than %d distinct streams in use on device %d", PWS_STREAMS, device);
    PairsWs &w = *wp;
    int rc = ensure(&w.inv, &w.inv_bytes, (size_t)n * 4);
    if (rc != VM_OK) return rc;
    const size_t st_cap = (size_t)cap + ((size_t)cap / 8 > 65536 ? (size_t)cap / 8 : 65536);
    if (st_cap > w.st_entries) {
        size_t have;
        have = w.st_entries * 4; rc = ensure(&w.st_i, &have, st_cap * 4); if (rc != VM_OK) return rc;
        have = w.st_entries * 4; rc = ensure(&w.st_j, &have, st_cap * 4); if (rc != VM_OK) return rc;
        have = w.st_entries * 4; rc = ensure(&w.st_s, &have, st_cap * 4); if (rc != VM_OK) return rc;
        w.st_entries = st_cap;
    }
    if (!w.cnt) VM_CUDA_CHECK(cudaMalloc(&w.cnt, 16));
    VM_CUDA_CHECK(cudaMemsetAsync(w.cnt, 0, 16, st));
    rc = k_row_inv_norms(x, dtype, (float *)w.inv, 0, n, ld, nullptr, st);
    if (rc != VM_OK) return rc;

    const int es = dtype == VM_F32 ? 4 : 2;
    const float eps = pairs_eps(dtype, dim);
    PairsParams p{};
    p.n = n;
    p.nbi = (int)((n + P_BM - 1) / P_BM);
    p.nbj = (int)((n + P_BN - 1) / P_BN);
    p.KB = (ld * es + 127) / 128;
    p.thr = threshold;
    p.thr_lo = threshold - eps;
    p.inv = (const float *)w.inv;
    p.st_i = (int32_t *)w.st_i; p.st_j = (int32_t *)w.st_j; p.st_s = (float *)w.st_s;
    p.st_cnt = (unsigned long long *)w.cnt;
    p.prog = (unsigned long long *)w.cnt + 1;   // zeroed with the staging counter above
    p.st_cap = (long long)st_cap;
    p.gj_log2 = n >= P_GJ_LARGE_FROM_ROWS ? P_GJ_LOG2_LARGE : P_GJ_LOG2_SMALL;
    const long long P_GJ = 1ll << p.gj_log2;
    const long long groups = (p.nbj + P_GJ - 1) / P_GJ;
    p.groups = (int)groups;
    p.total_tiles = P_GJ * P_GJ * groups * (groups + 1);  // full groups (2 P_GJ row blocks per group step); tiles outside the matrix are skipped in-kernel
    p.part = part; p.nparts = nparts;

    CUtensorMap tmA, tmB;
    rc = make_tmap_2d(&tmA, x, dtype, (uint64_t)n, (uint64_t)ld, (uint64_t)ld, P_BM);
    if (rc != VM_OK) return rc;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
#ifdef VIDMEM_TRIAGE_KERNELS
    static const bool one_cta = getenv("VIDMEM_PAIRS_1CTA") != nullptr;  // perf triage builds only: force the 1-CTA kernel
#else
    constexpr bool one_cta = false;  // the shipped library has no environment switch that changes what a kernel computes
#endif
    if (!one_cta) {
        // ---- CTA-pair kernel: 256 x 256 tiles ----
        const long long nb = (n + 255) / 256, groups = (nb + P_GJ - 1) / P_GJ;
        p.total_tiles = P_GJ * P_GJ * groups * (groups + 1) / 2;
        const size_t smem = (size_t)P2_STAGES * P2_STAGE_BYTES + P_ACC * P_BN * 4 + 8 * (2 * P2_STAGES + 2 * P_ACC) + 16 + 1024;
        const long long my_tiles = (p.total_tiles + nparts - 1) / nparts;
        long long pairs = sms / 2;
        if (my_tiles < pairs) pairs = my_tiles;
        const int grid = (int)(2 * pairs);
        if (dtype == VM_F32) {
            VM_CUDA_CHECK((max_smem_once<pairs_tc2_kernel<true>>(227 * 1024)));
            pairs_tc2_kernel<true><<<grid, P_THREADS, smem, st>>>(tmA, p);
        } else {
            VM_CUDA_CHECK((max_smem_once<pairs_tc2_kernel<false>>(227 * 1024)));
            pairs_tc2_kernel<false><<<grid, P_THREADS, smem, st>>>(tmA, p);
        }
    } else {
        rc = make_tmap_2d(&tmB, x, dtype, (uint64_t)n, (uint64_t)ld, (uint64_t)ld, P_BN);
        if (rc != VM_OK) return rc;
        const size_t smem = (size_t)P_STAGES * P_STAGE_BYTES + P_ACC * P_BN * 4 + 8 * (2 * P_STAGES + 2 * P_ACC) + 16 + 1024;
        const long long my_tiles = (p.total_tiles + nparts - 1) / nparts;
        const int grid = (int)(my_tiles < sms ? my_tiles : sms);
        if (dtype == VM_F32) {
            VM_CUDA_CHECK((max_smem_once<pairs_tc_kernel<true>>(227 * 1024)));
            pairs_tc_kernel<true><<<grid, P_THREADS, smem, st>>>(tmA, tmB, p);
        } else {
            VM_CUDA_CHECK((max_smem_once<pairs_tc_kernel<false>>(227 * 1024)));
            pairs_tc_kernel<false><<<grid, P_THREADS, smem, st>>>(tmA, tmB, p);
        }
    }
    VM_CUDA_CHECK(cudaGetLastError());
    if (dtype == VM_F32)
        pairs_finalize_kernel<float><<<64, 256, 0, st>>>((const float *)x, ld, dim, threshold, eps, p.st_i, p.st_j, p.st_s, p.st_cnt,
                                                         p.st_cap, out_i, out_j, out_score, (unsigned long long *)out_count, cap);
    else
        pairs_finalize_kernel<__nv_bfloat16><<<64, 256, 0, st>>>((const __nv_bfloat16 *)x, ld, dim, threshold, eps, p.st_i, p.st_j,
                                                                 p.st_s, p.st_cnt, p.st_cap, out_i, out_j, out_score,
                                                                 (unsigned long long *)out_count, cap);
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

}  // namespace vm
