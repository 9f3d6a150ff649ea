// scan_tc.cu -- tcgen05 / TMA streaming scorer: the bandwidth-bound scan for query batches.
//
// One persistent CTA per SM, warp-specialised (288 threads; 192 in dump mode):
//   warp 0   TMA producer   streams the store as 128-row x 128-byte boxes (SWIZZLE_128B) through a
//                           ring of 16 KB shared-memory stages, L2 evict-first; loads the
//                           normalised queries once (evict-last) -- no thread ever touches a row
//   warp 1   MMA issuer     one thread issues tcgen05.mma (kind::tf32 for an fp32 store, kind::f16
//                           for bf16): D[128 rows x nq] += A[128 x 32B] * Q[nq x 32B]^T, accumulators
//                           in TMEM (8 stages x nq columns), tcgen05.commit frees stages / publishes D
//   warps 2-5 epilogue      tcgen05.ld their 32-lane TMEM quadrant (lane = store row, column = query),
//                           multiply by the cached 1/||row|| (fused normalisation), compare with the
//                           per-query band threshold; a survivor is APPENDED, lock-free, to this CTA's
//                           private slab of the query (a shared-memory counter hands out the slot, the key
//                           goes to global memory with a fire-and-forget store).  No queues, no CTA-wide
//                           barriers, no serial drain: the four warps run independently, tile after tile.
//   warp 8   bound service  keeps the thresholds current (see below); sleeps between rounds
//
// What the scan keeps -- the COMPLETE NEAR-TIE BAND, not a top-kp list.  Let a_(k) be the k-th best approximate
// score of the shard and eps the scan's error bound.  A row can only be in the exact top-k if its approximate score
// reaches a_(k) - 2 eps (its exact score must reach the k-th exact score, which is >= a_(k) - eps).  Every CTA filters
// with the band threshold B = L - 2 eps, where L <= a_(k) is a lower bound that only grows:
//   * seed: each CTA publishes, per query, the maximum of its first tile; the k-th largest of those <= 148 maxima is
//     reached by k distinct rows, so it is <= a_(k).  Derived once by the CTA that owns the query (q mod G),
//     published with an atomic max, adopted by all CTAs (bounded waits; a late CTA only loosens the bound);
//   * bound service (one warp per CTA, off the critical path): publishes this CTA's RUNNING maximum per query, the
//     owner CTA of a query keeps re-deriving the k-th largest of all CTAs' maxima -- the bound follows the
//     shard-wide top-k --, a CTA whose own slab fills up publishes its own k-th best (k of its own rows reach it:
//     what finds a tight cluster that lives in ONE CTA, e.g. the 64 consecutive near-duplicate chunks of a static
//     scene), and every CTA adopts whatever has been published.
// A slab holds 64 keys per (CTA, query); beyond that keys go to the query's shared spill buffer (global atomic; rare
// once the own-k-th bound is in place).  Slabs + spill therefore hold EVERY row with approximate score >= the final
// threshold: select.cu filters them once more with the final bound, rescores the best kp in binary64, and if more
// than those lie within eps of the k-th exact score it rescores that whole band from the same keys -- no second
// scan.  Only a spill overflow (thousands of near-ties: duplicates, a zero query) falls back to the collect pass.
// bf16 stores, split query (ScanArgs::split): the normalised fp32 query is fed as q_hi + q_lo (two bf16 terms, 16
// mantissa bits), two MMAs per K slice into the same accumulator, so eps drops from 2^-8 to ~2^-16 + (D+16) 2^-23.
// HBM traffic = the store bytes exactly once per batch of <= 64 queries.
// Collect mode (second pass for queries the first pass could not settle): thresholds are fixed per
// query (exact k-th candidate score - 2 eps; +inf for queries that need nothing) and every row at or
// above its query's threshold is appended to that query's global buffer.
// Dump mode (template DUMP, stores of <= 9472 rows): with one tile per CTA there is nothing to filter with.
// The epilogue writes the key of EVERY row, [tile][query][128], and select.cu ranks all of them per query.
#include "tc_common.cuh"

namespace vm {
using namespace tc;

static constexpr int TC_BLOCK_M = 128;
static constexpr int TC_STAGE_BYTES = TC_BLOCK_M * 128;
static constexpr int TC_ACC = 8;      // accumulator stages in TMEM (8 x 64 columns = all 512)
static constexpr int TC_THREADS_SVC = 288;  // TMA warp, MMA warp, 4 epilogue warps, (2 idle), bound-service warp 8
static constexpr int TC_THREADS = 192;      // dump mode: no service warp
static constexpr int TC_TMEM_COLS = 512;
static constexpr int TC_MAX_STAGES = 8;

// second-pass ("collect") arguments; thr == nullptr selects the normal mode
struct CollectArgs {
    const float *thr;      // [nq] per-query score threshold (+inf: ignore the query)
    uint64_t *buf;         // [nq][cap] collected keys
    int *cnt;              // [nq] number of rows at or above the threshold (may exceed cap)
    int cap;
    const int *pending;    // device counter of uncertified queries: 0 -> the kernel exits at once
};

// where the survivors go (normal mode)
struct BandArgs {
    uint64_t *slab;   // [ctas][nq][SCAN_SLAB] private append buffers
    int *scnt;        // [ctas][nq] keys appended to each slab (may exceed SCAN_SLAB: the rest went to the spill buffer)
    uint64_t *ubuf;   // [nq][ucap] shared spill buffer
    int *ucnt;        // [nq] keys spilled (may exceed ucap: overflow, the query goes to the collect pass)
    int ucap;
    float band;       // 2 eps, rounded up
    int ksel;         // k: the bound is the k-th largest per-CTA maximum
    int use_seed;     // first-tile seeding + owner selects (needs ksel <= ctas <= 256)
};

struct TcLayout {
    int nq_pad, KB, stages, split;
    uint32_t off_b, off_a, off_tauf, off_lcnt, off_cmax, off_wmax, off_flags, off_bars, off_tmem, total;
};

static TcLayout make_layout(int dtype, int ld, int nq, int split = 0)
{
    TcLayout L{};
    const int es = dtype == VM_F32 ? 4 : 2;
    L.nq_pad = (nq + 15) & ~15;
    L.KB = (ld * es + 127) / 128;
    L.split = (split && dtype == VM_BF16) ? 1 : 0;
    uint32_t o = 0;
    L.off_b = o; o += (uint32_t)L.KB * L.nq_pad * 128 * (L.split ? 2 : 1);
    const uint32_t epi = (uint32_t)L.nq_pad * (4 + 4 + 4 + 16) + 64 + 8 * (2 * TC_MAX_STAGES + 1 + 2 * TC_ACC) + 16;
    int64_t room = 227 * 1024 - 2048 - (int64_t)o - epi;
    L.stages = (int)(room / TC_STAGE_BYTES);
    if (L.stages > TC_MAX_STAGES) L.stages = TC_MAX_STAGES;
    if (L.stages < 0) L.stages = 0;
    L.off_a = o; o += (uint32_t)L.stages * TC_STAGE_BYTES;
    L.off_tauf = o; o += (uint32_t)L.nq_pad * 4;   // 16-byte aligned: everything above is a multiple of 128
    L.off_lcnt = o; o += (uint32_t)L.nq_pad * 4;
    L.off_cmax = o; o += (uint32_t)L.nq_pad * 4;
    L.off_wmax = o; o += (uint32_t)L.nq_pad * 16;  // [4][nq_pad] seeding scratch
    L.off_flags = o; o += 64;
    L.off_bars = o; o += 8 * (2 * TC_MAX_STAGES + 1 + 2 * TC_ACC);
    L.off_tmem = o; o += 16;
    L.total = o + 1024;  // slack for the 1024-byte alignment of the swizzled tiles
#ifdef VIDMEM_AB_SMEMPAD
    if (L.total < 220 * 1024) L.total = 220 * 1024;
#endif
    return L;
}

// k-th largest score (ordered bits, low 12 bits truncated: rounds down) among the first n <= SCAN_SLAB keys of one slab
// (global memory; a slot whose store has not landed yet reads as 0 and is ignored): a lower bound on the shard's k-th
// best, because k rows of this CTA reach it.  Warp-collective: one coalesced load, then a 20-step radix select over
// warp reductions (~1 us; the single-thread insertion sort it replaces took ~10 us of dependent L2 loads, during which
// the service warp adopted no published bounds).  Returns 0 when fewer than k keys are there.
__device__ __forceinline__ uint32_t own_kth_score(const uint64_t *slab, int n, int k, int lane)
{
    constexpr int PER = SCAN_SLAB / 32;
    uint32_t vals[PER];
#pragma unroll
    for (int t = 0; t < PER; ++t) {
        const int i = lane + 32 * t;
        vals[t] = i < n ? (uint32_t)(__ldcg(slab + i) >> 32) : 0u;
    }
    uint32_t prefix = 0;
    int need = k;
    for (int bit = 31; bit >= 12; --bit) {
        const uint32_t hi = bit == 31 ? 0u : (0xFFFFFFFFu << (bit + 1));
        int cnt = 0;
#pragma unroll
        for (int t = 0; t < PER; ++t) cnt += ((vals[t] & hi) == prefix && ((vals[t] >> bit) & 1u)) ? 1 : 0;
        const int tot = __reduce_add_sync(0xffffffffu, cnt);
        if (tot >= need) prefix |= 1u << bit;
        else need -= tot;
    }
    // fewer than k non-empty keys: the select runs out of candidates and ends on a prefix no key carries -> no bound
    int ge = 0;
#pragma unroll
    for (int t = 0; t < PER; ++t) ge += (vals[t] != 0u && vals[t] >= prefix) ? 1 : 0;
    ge = __reduce_add_sync(0xffffffffu, ge);
    return (ge >= k && prefix != 0u) ? prefix : 0u;
}

template <bool TF32, bool DUMP, bool SPLIT>
__global__ void __launch_bounds__(DUMP ? TC_THREADS : TC_THREADS_SVC, 1)
scan_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const float *__restrict__ inv_norms, int64_t n, int num_tiles, int nq, TcLayout L, uint64_t *__restrict__ dump_keys,
               uint32_t *__restrict__ seed_tab, int *__restrict__ seed_ctr, CollectArgs col, BandArgs ub, int svc_sleep)
{
    const bool collect = !DUMP && col.thr != nullptr;
#ifndef VIDMEM_AB_NOPDL
    pdl_launch_dependents();  // the next kernel of the stream may be scheduled as SMs free up (it waits for our completion)
#endif
    if (collect) {
        pdl_wait();
        if (*col.pending == 0) return;  // nothing left to refine (uniform across the grid)
    }

    extern __shared__ __align__(16) uint8_t smem_raw[];
    // align to 1024 B with pointer arithmetic on the __shared__ array (an integer round trip would
    // demote every later access to generic LD/ST)
    uint8_t *base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *sB = base + L.off_b;
    uint8_t *sA = base + L.off_a;
    float *tauf = (float *)(base + L.off_tauf);            // [nq_pad] band threshold per query (only grows)
    int *lcnt = (int *)(base + L.off_lcnt);                // [nq_pad] keys appended to this CTA's slab of the query
    uint32_t *cmax = (uint32_t *)(base + L.off_cmax);      // [nq_pad] best score (ordered bits) this CTA has seen
    uint32_t *wmax = (uint32_t *)(base + L.off_wmax);      // [4][nq_pad] seeding scratch
    volatile int *s_done = (volatile int *)(base + L.off_flags);  // [0] epilogue warps finished, [1] seed phase over
    uint64_t *bars = (uint64_t *)(base + L.off_bars);
    uint64_t *full = bars, *empty = bars + TC_MAX_STAGES, *qfull = bars + 2 * TC_MAX_STAGES;
    uint64_t *tfull = qfull + 1, *tempty = tfull + TC_ACC;
    uint32_t *tmem_slot = (uint32_t *)(base + L.off_tmem);

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
    const int lane = threadIdx.x & 31;
    const int nq_pad = L.nq_pad, KB = L.KB, stages = L.stages;
    constexpr int ELEMS = TF32 ? 32 : 64;  // elements per 128-byte K block

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(qfull, 1);
        for (int a = 0; a < TC_ACC; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, TC_TMEM_COLS);
#ifndef VIDMEM_AB_NOPDL
    if (!collect) pdl_wait();  // everything above overlapped the previous kernel; from here on we read what it wrote
#endif
    if (warp >= 2 && warp < 6) {
        const int e = threadIdx.x - 64;
        if (e < nq_pad) {
            lcnt[e] = 0;
            cmax[e] = 0u;
            tauf[e] = collect ? (e < nq ? col.thr[e] : INFINITY) : (e < nq ? -INFINITY : INFINITY);
        }
        if (e < 2) s_done[e] = 0;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    uint32_t *gbound = seed_tab ? seed_tab + SEED_TAB_WORDS : nullptr;  // [64] published lower bounds on a_(k), ordered bits

    if (warp == 0) {
        // ================================ TMA producer ================================
        // The whole warp runs the loop converged and ONE elected lane issues (elect.sync): the compiler then keeps the
        // loop state in uniform registers instead of wrapping every issue in a per-lane loop.  The issue thread's
        // instruction count per 16 KB block is what bounds a bf16 scan (2.2 us per tile), so it is kept minimal.
        if (elect_one()) {
            constexpr int QPARTS = SPLIT ? 2 : 1;  // query blocks: hi part, then (split) lo part = rows [nq_pad, 2 nq_pad) of tmB
            mbar_arrive_expect_tx(qfull, (uint32_t)(KB * QPARTS) * nq_pad * 128);
            for (int part = 0; part < QPARTS; ++part)
                for (int kb = 0; kb < KB; ++kb)
                    tma_load_2d(&tmB, qfull, sB + (size_t)(part * KB + kb) * nq_pad * 128, kb * ELEMS, part * nq_pad, L2_EVICT_LAST);
        }
        __syncwarp();
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(&empty[stage], phase ^ 1);
                if (elect_one()) {
                    mbar_arrive_expect_tx(&full[stage], TC_STAGE_BYTES);
                    tma_load_2d(&tmA, &full[stage], sA + (size_t)stage * TC_STAGE_BYTES, kb * ELEMS, tile * TC_BLOCK_M, L2_EVICT_FIRST);
                }
                __syncwarp();
                if (++stage == stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ==================================
        // Same scheme: converged warp, one elected lane issues the MMAs of a block and its commit.  Descriptors are
        // the stage-0 descriptor plus an offset in the 14-bit start-address field (units of 16 bytes).
        const uint32_t idesc = make_idesc(TF32 ? 2u : 1u, TC_BLOCK_M, (uint32_t)nq_pad);
        mbar_wait(qfull, 0);
        tc_fence_after();
        int stage = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        const uint64_t da0 = make_smem_desc_sw128(smem_u32(sA)), db0 = make_smem_desc_sw128(smem_u32(sB));
        const uint32_t kb_step = (uint32_t)(nq_pad * 128) >> 4, lo_step = (uint32_t)(KB * nq_pad * 128) >> 4;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            mbar_wait(&tempty[acc], acc_phase ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(acc * nq_pad);
            for (int kb = 0; kb < KB; ++kb) {
                mbar_wait(&full[stage], phase);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t da = da0 + (uint64_t)((uint32_t)stage * (TC_STAGE_BYTES >> 4));
                    const uint64_t db = db0 + (uint64_t)((uint32_t)kb * kb_step);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {  // 4 x 32-byte K slices per 128-byte swizzle row
                        umma<TF32>(d_tmem, da + 2 * j, db + 2 * j, idesc, (uint32_t)((kb | j) != 0));
                        if constexpr (SPLIT) umma<TF32>(d_tmem, da + 2 * j, db + lo_step + 2 * j, idesc, 1u);
                    }
                    umma_commit(&empty[stage]);               // stage reusable once these MMAs have read it
                    if (kb == KB - 1) umma_commit(&tfull[acc]);  // ... and the accumulator is complete
                }
                __syncwarp();
                if (++stage == stages) { stage = 0; phase ^= 1; }
            }
            if (++acc == TC_ACC) { acc = 0; acc_phase ^= 1; }
        }
    } else if (warp < 6) {
        // ================================ epilogue =====================================
        const int e = threadIdx.x - 64;   // 0..127
        const int quad = warp & 3;        // TMEM lane quadrant this warp may read
        const int row_in_tile = quad * 32 + lane;
        int acc = 0;
        uint32_t acc_phase = 0;
        if constexpr (DUMP) {
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int64_t r = (int64_t)tile * TC_BLOCK_M + row_in_tile;
                const float iv = r < n ? __ldg(inv_norms + r) : -1.0f;
                mbar_wait(&tfull[acc], acc_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * nq_pad);
                uint64_t *out = dump_keys + (int64_t)tile * nq * TC_BLOCK_M + row_in_tile;
                for (int c = 0; c < nq_pad; c += 16) {
                    uint32_t v[16];
                    tmem_ld16(taddr + c, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j)
                        if (c + j < nq)  // coalesced: 32 consecutive rows of one query per warp store
                            out[(int64_t)(c + j) * TC_BLOCK_M] = iv >= 0.0f ? make_key(__uint_as_float(v[j]) * iv, (uint32_t)r) : 0ull;
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[acc]);
                if (++acc == TC_ACC) { acc = 0; acc_phase ^= 1; }
            }
        } else {
        if (ub.use_seed && !collect) {
            // ---- cooperative bound seeding from the first tile (see file header) ----
            const int64_t row0 = (int64_t)blockIdx.x * TC_BLOCK_M + row_in_tile;
            const float inv0 = row0 < n ? __ldg(inv_norms + row0) : -1.0f;
            mbar_wait(&tfull[0], 0);
            tc_fence_after();
            const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16);
            for (int c = 0; c < nq_pad; c += 16) {
                uint32_t v[16];
                tmem_ld16(taddr0 + c, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float sc = inv0 >= 0.0f ? __uint_as_float(v[j]) * inv0 : -INFINITY;
                    const uint32_t mx = __reduce_max_sync(0xffffffffu, f32_ordered(sc));
                    if (lane == 0) wmax[(warp - 2) * nq_pad + c + j] = mx;
                }
            }
            named_bar_sync(1, 128);
            if (e < nq_pad) {
                uint32_t m = wmax[e];
#pragma unroll
                for (int w = 1; w < 4; ++w) m = max(m, wmax[w * nq_pad + e]);
                seed_tab[(size_t)blockIdx.x * nq_pad + e] = m;
                cmax[e] = m;  // the running maximum starts from the first tile's (a real row's score, survivor or not)
            }
            __threadfence();
            named_bar_sync(1, 128);
            if (e == 0) {
                atomicAdd(seed_ctr, 1);
                const long long t0 = clock64();
                while (*(volatile int *)seed_ctr < (int)gridDim.x)
                    if (clock64() - t0 > 400000) break;  // ~0.2 ms: late CTAs only loosen the bound
                __threadfence();
            }
            named_bar_sync(1, 128);
            // The bound of query q is derived once, by the CTA that owns it (q mod G), and published; a second,
            // short bounded wait lets every CTA adopt all nq bounds (64 exact selects in every CTA cost ~15 us).
            const int G = (int)gridDim.x;
            int *pub_ctr = reinterpret_cast<int *>(gbound + 64);
            if (warp == 2) {
                for (int q = blockIdx.x; q < nq; q += G) {
                    const float sd = seed_select(seed_tab, G, nq_pad, q, ub.ksel, lane);
                    if (lane == 0) {
                        if (sd > -INFINITY) atomicMax(gbound + q, f32_ordered(sd));
                        __threadfence();
                        atomicAdd(pub_ctr, 1);
                    }
                }
                if (lane == 0) {
                    const long long t0 = clock64();
                    while (*(volatile int *)pub_ctr < nq)
                        if (clock64() - t0 > 200000) break;  // ~0.1 ms: a missing bound only means "no threshold yet"
                    __threadfence();
                }
            }
            named_bar_sync(1, 128);
            if (e < nq) {
                const uint32_t o = __ldcg(gbound + e);
                if (o != 0u) tauf[e] = band_floor(f32_from_ordered(o), ub.band);  // the service warp takes over after the go-ahead below
            }
            named_bar_sync(1, 128);
        }
        if (!collect && e == 0) s_done[1] = 1;  // go-ahead for the bound service: the seed is in place
        uint64_t *my_slab = collect ? nullptr : ub.slab + (size_t)blockIdx.x * nq * SCAN_SLAB;
        int64_t row = (int64_t)blockIdx.x * TC_BLOCK_M + row_in_tile;
        float inv = row < n ? __ldg(inv_norms + row) : -1.0f;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            // prefetch the next tile's inverse norm so its DRAM latency hides behind this tile
            const int64_t row_next = row + (int64_t)gridDim.x * TC_BLOCK_M;
            const float inv_next = (tile + (int)gridDim.x < num_tiles && row_next < n) ? __ldg(inv_norms + row_next) : -1.0f;
            const bool valid = inv >= 0.0f;  // < 0: beyond the shard or a skipped row
            mbar_wait(&tfull[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * nq_pad);
            // 16 queries (TMEM columns) at a time; the load of chunk c+1 is issued before chunk c is
            // processed so its TMEM latency hides behind the compares
            auto process = [&](const uint32_t (&v)[16], int c) {
                // thresholds of these 16 queries (a stale, lower value only lets an extra key through)
                float tf[16];
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(tauf + c + 4 * j4);
                    tf[4 * j4] = t4.x; tf[4 * j4 + 1] = t4.y; tf[4 * j4 + 2] = t4.z; tf[4 * j4 + 3] = t4.w;
                }
                if (valid) {
                    uint32_t hits = 0;
#pragma unroll
                    for (int j = 0; j < 16; ++j) hits |= (__uint_as_float(v[j]) * inv >= tf[j]) ? (1u << j) : 0u;
                    hits &= nq - c >= 16 ? 0xFFFFu : ((1u << (nq - c > 0 ? nq - c : 0)) - 1u);
                    while (hits) {  // rare path
                        const int j = __ffs(hits) - 1;
                        hits &= hits - 1;
                        const int q = c + j;
                        float s = 0.0f;
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) s = (jj == j) ? __uint_as_float(v[jj]) * inv : s;
                        const uint64_t key = make_key(s, (uint32_t)row);
                        if (collect) {
                            const int pos = atomicAdd(col.cnt + q, 1);
                            if (pos < col.cap) col.buf[(size_t)q * col.cap + pos] = key;
                        } else {
#ifdef VIDMEM_AB_NORARE
                            if (key == 1) tauf[q] = 0.0f;
                            continue;
#endif
                            const int pos = atomicAdd(&lcnt[q], 1);           // shared-memory counter hands out the slot
                            atomicMax(&cmax[q], (uint32_t)(key >> 32));
                            if (pos < SCAN_SLAB) __stcg(my_slab + (size_t)q * SCAN_SLAB + pos, key);   // fire and forget
                            else {
                                const int p = atomicAdd(ub.ucnt + q, 1);     // slab full: the query's shared spill buffer
                                if (p < ub.ucap) __stcg(ub.ubuf + (size_t)q * ub.ucap + p, key);
                                else tauf[q] = INFINITY;  // spill overflow: the query is re-done anyway, stop collecting
                            }
                        }
                    }
                }
            };
            uint32_t va[16], vb[16];
#ifdef VIDMEM_AB_NOEPI
            if (tile < 0)
#endif
            tmem_ld16(taddr, va);
#ifdef VIDMEM_AB_NOEPI
            if (tile < 0)
#endif
            for (int c = 0; c < nq_pad; c += 32) {
                tmem_ld_wait();
                if (c + 16 < nq_pad) tmem_ld16(taddr + c + 16, vb);
                process(va, c);
                if (c + 16 < nq_pad) {
                    tmem_ld_wait();
                    if (c + 32 < nq_pad) tmem_ld16(taddr + c + 32, va);
                    process(vb, c + 16);
                }
            }
#ifdef VIDMEM_AB_TILEBAR
            named_bar_sync(1, 128);
#endif
            // release the accumulator stage to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
            if (++acc == TC_ACC) { acc = 0; acc_phase ^= 1; }
            row = row_next;
            inv = inv_next;
        }
        if (!collect) {
            named_bar_sync(1, 128);  // all four warps have appended their last keys
            if (e < nq) {
                ub.scnt[(size_t)blockIdx.x * nq + e] = lcnt[e];
                // final running maximum of this CTA: select.cu derives the final bound from the table
                if (seed_tab != nullptr) __stcg(seed_tab + (size_t)blockIdx.x * nq_pad + e, cmax[e]);
            }
        }
        }  // !DUMP
        __syncwarp();
        if (lane == 0) atomicAdd((int *)s_done, 1);
    } else {
        // ================================ bound service ================================
        // Off the critical path (one warp, sleeps between rounds); a stale bound only keeps a few more rows.
#ifdef VIDMEM_AB_NOSVC
        if (false) {
#else
        if (!DUMP && warp == 8 && seed_tab != nullptr && !collect) {
#endif
            const int G = (int)gridDim.x;
            while (s_done[1] == 0 && s_done[0] < 4) __nanosleep(100);   // wait for the seed phase (it writes tauf)
            uint32_t pub0 = 0xFFFFFFFFu, pub1 = 0xFFFFFFFFu;            // running maxima last written to the table (lanes q, q+32)
            uint32_t kth_done = 0;                                       // 4 bits per query (q, q+32): highest slab level whose own k-th is published
            const uint64_t *my_slab = ub.slab + (size_t)blockIdx.x * nq * SCAN_SLAB;
            // the exit test is a warp vote: a lane that lags behind must not leave the loop while the others
            // are already inside the next round's warp reductions
            while (!__any_sync(0xffffffffu, s_done[0] >= 4)) {
                // 1. this CTA's running maxima -> the table
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int q = lane + 32 * h;
                    if (q < nq) {
                        const uint32_t c = *(volatile uint32_t *)(cmax + q);
                        uint32_t &pub = h ? pub1 : pub0;
                        if (c != pub && c != 0u) { __stcg(seed_tab + (size_t)blockIdx.x * nq_pad + q, c); pub = c; }
                    }
                }
                __syncwarp();
                // 2. queries this CTA owns: k-th largest of all CTAs' maxima (warp-collective)
                if (G >= ub.ksel)
                    for (int q = blockIdx.x; q < nq; q += G) {
                        const float sd = seed_select(seed_tab, G, nq_pad, q, ub.ksel, lane);
                        if (lane == 0 && sd > -INFINITY) atomicMax(gbound + q, f32_ordered(sd));
                    }
                __syncwarp();
                // 3. a slab that is half full / full: this CTA's own k-th best is a valid bound too (k of its rows reach it).
                //    Served by the whole warp, at most KTH_PER_ROUND per round so that steps 1, 2 and 4 never starve
                //    (on a store of tight clusters every cluster hit fills half a slab at once).
#ifndef VIDMEM_AB_KTH_LEVELS
#define VIDMEM_AB_KTH_LEVELS 2
#endif
#ifndef VIDMEM_AB_KTH_PER_ROUND
#define VIDMEM_AB_KTH_PER_ROUND 1
#endif
                {
                    constexpr int LV = VIDMEM_AB_KTH_LEVELS;   // levels: slab >> (LV - level) keys, level = 1 .. LV
                    int served = 0;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int q = lane + 32 * h;
                        int level = 0;
                        if (q < nq) {
                            const int have = *(volatile int *)(lcnt + q);
#pragma unroll
                            for (int l = 1; l <= LV; ++l) level = have >= (SCAN_SLAB >> (LV - l)) ? l : level;
                        }
                        const int done = (int)((kth_done >> (4 * h)) & 15u);
                        unsigned todo = __ballot_sync(0xffffffffu, level > done && (SCAN_SLAB >> (LV - level)) >= ub.ksel);
                        while (todo && (VIDMEM_AB_KTH_PER_ROUND == 0 || served < VIDMEM_AB_KTH_PER_ROUND)) {
                            const int src = __ffs(todo) - 1;
                            todo &= todo - 1;
                            ++served;
                            const int lv = __shfl_sync(0xffffffffu, level, src);
                            const int qq = src + 32 * h;
                            const uint32_t ok = own_kth_score(my_slab + (size_t)qq * SCAN_SLAB, SCAN_SLAB >> (LV - lv), ub.ksel, lane);
                            if (lane == src && ok != 0u) {
                                atomicMax(gbound + qq, ok);
                                kth_done = (kth_done & ~(15u << (4 * h))) | ((uint32_t)lv << (4 * h));
                            }
                        }
                    }
                }
                __syncwarp();
                // 4. adopt whatever has been published
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int q = lane + 32 * h;
                    if (q < nq) {
                        const uint32_t o = __ldcg(gbound + q);
                        if (o != 0u) {
                            const float f = band_floor(f32_from_ordered(o), ub.band);
                            if (f > tauf[q]) *(volatile float *)(tauf + q) = f;   // only this warp writes tauf from here on
                        }
                    }
                }
                __nanosleep(svc_sleep);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TC_TMEM_COLS);
    }
}

bool scan_tc_supported(int dtype, int dim, int nq, int kp, int split)
{
    (void)kp;
    if (dtype != VM_F32 && dtype != VM_BF16) return false;
    if (nq < 1 || nq > 64) return false;
    TcLayout L = make_layout(dtype, ld_for_dim(dim), nq, split);
    return L.stages >= 3;
}

// queries_store_dtype: the normalised queries in the STORE dtype: fp32 [nq_pad][ld] (tf32 path), bf16 [nq_pad][ld],
// or bf16 [2][nq_pad][ld] (hi terms, then lo terms) with a.split.
int launch_scan_tc(const ScanArgs &a, const void *queries_store_dtype, uint32_t *seed_tab, int *seed_ctr, const ScanCollect *sc,
                   ScanInfo *info)
{
    VM_REQUIRE(a.n >= 1 && a.n < 0x7FFFFF00LL, VM_ERR_UNSUPPORTED, "tcgen05 scan: shard rows %lld outside [1, 2^31)", (long long)a.n);
    TcLayout L = make_layout(a.dtype, a.ld, a.nq, a.split);
    VM_REQUIRE(L.stages >= 3, VM_ERR_UNSUPPORTED, "tcgen05 scan: dim %d x %d queries does not fit shared memory", a.dim, a.nq);
    CUtensorMap tmA, tmB;
    int rc = make_tmap_2d_cached(&tmA, a.rows, a.dtype, (uint64_t)a.n, (uint64_t)a.ld, (uint64_t)a.ld, TC_BLOCK_M);
    if (rc != VM_OK) return rc;
    rc = make_tmap_2d_cached(&tmB, queries_store_dtype, a.dtype, (uint64_t)L.nq_pad * (L.split ? 2 : 1), (uint64_t)a.ld, (uint64_t)a.ld,
                             (uint32_t)L.nq_pad);
    if (rc != VM_OK) return rc;
    const int num_tiles = (int)((a.n + TC_BLOCK_M - 1) / TC_BLOCK_M);
    const bool dump = a.dump && !sc;
    if (sc || dump || a.ctas > 256) { seed_tab = nullptr; seed_ctr = nullptr; }
    CollectArgs col{};
    if (sc) { col.thr = sc->thr; col.buf = sc->buf; col.cnt = sc->cnt; col.cap = sc->cap; col.pending = sc->pending; }
    BandArgs ub{a.slab, a.scnt, a.ubuf, a.ucnt, a.ucap, a.band, a.ksel, 0};
    // first-tile seeding needs at least k CTAs (k first-tile maxima); without it the scan still works -- every row
    // is a survivor until a slab fills up and the CTA's own k-th best takes over
    ub.use_seed = (seed_tab && seed_ctr && a.ksel >= 1 && a.ctas >= a.ksel) ? 1 : 0;
    if (!sc && !dump)
        VM_REQUIRE(ub.slab && ub.scnt && ub.ubuf && ub.ucnt && ub.ucap > 0 && ub.ksel >= 1, VM_ERR_BADARG, "tcgen05 scan: slab / spill buffers missing");
    if (dump) VM_REQUIRE(TC_BLOCK_M == SCAN_DUMP_TILE && (int64_t)num_tiles * TC_BLOCK_M <= SCAN_DUMP_MAX_KEYS && a.ctas == num_tiles,
                         VM_ERR_UNSUPPORTED, "tcgen05 scan: dump mode needs one CTA per tile and at most %d rows", SCAN_DUMP_MAX_KEYS);
    // The bound service polls faster where the epilogue, not HBM, paces the scan (bf16 tiles stream in 2.2 us) and
    // lazily where an fp32 tile (4.4 us) hides everything anyway.
#ifdef VIDMEM_AB_SVCSLEEP
    const int svc_sleep = VIDMEM_AB_SVCSLEEP;
#else
    const int svc_sleep = a.dtype == VM_F32 ? 500 : 200;
#endif
    if (info && !sc) { info->stages = L.stages; info->variant = dump ? 1 : 2; }
    const bool pdl = a.pdl && !sc;
#ifdef VIDMEM_AB_CLASSIC_LAUNCH
#define LAUNCH_IMPL(TF, DU, SP) scan_tc_kernel<TF, DU, SP><<<a.ctas, DU ? TC_THREADS : TC_THREADS_SVC, L.total, a.stream>>>(tmA, tmB, a.inv_norms, a.n, num_tiles, a.nq, L, a.cand, seed_tab, seed_ctr, col, ub, svc_sleep)
#else
#define LAUNCH_IMPL(TF, DU, SP) VM_CUDA_CHECK(launch_pdl(scan_tc_kernel<TF, DU, SP>, dim3(a.ctas), dim3(DU ? TC_THREADS : TC_THREADS_SVC), L.total, a.stream, pdl, \
                                 tmA, tmB, a.inv_norms, a.n, num_tiles, a.nq, L, a.cand, seed_tab, seed_ctr, col, ub, svc_sleep))
#endif
#define LAUNCH_TC(TF, DU, SP)                                                                                                \
    do {                                                                                                                   \
        VM_CUDA_CHECK((max_smem_once<scan_tc_kernel<TF, DU, SP>>(227 * 1024)));                                              \
        LAUNCH_IMPL(TF, DU, SP);                                                                                           \
    } while (0)
    if (a.dtype == VM_F32) { if (dump) LAUNCH_TC(true, true, false); else LAUNCH_TC(true, false, false); }
    else if (L.split) { if (dump) LAUNCH_TC(false, true, true); else LAUNCH_TC(false, false, true); }
    else { if (dump) LAUNCH_TC(false, true, false); else LAUNCH_TC(false, false, false); }
#undef LAUNCH_TC
#undef LAUNCH_IMPL
    VM_CUDA_CHECK(cudaGetLastError());
    return VM_OK;
}

}  // namespace vm
