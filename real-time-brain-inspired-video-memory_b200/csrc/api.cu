// api.cu -- the C ABI of libvidmem.so (include/vidmem.h): handles, workspaces, orchestration of
// scan -> merge -> exact rescoring -> (rare) exact re-scan, NCCL gather + merge for shards.
#include "common.cuh"

#include <dlfcn.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <new>
#include <vector>

namespace vm {

// ---- thread-local error message -----------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ---- kernels implemented in the other translation units -----------------------------------
int k_convert_rows(const void *src, int src_dtype, void *dst, int dst_dtype, int64_t n, int dim, int ld, cudaStream_t st);
int k_row_inv_norms(const void *rows, int dtype, float *inv_norms, int64_t row0, int64_t n, int ld, int *extreme, cudaStream_t st,
                    const double *exact = nullptr);
int k_invalidate_rows(float *inv_norms, const int64_t *rows_dev, int64_t n, int64_t size, cudaStream_t st);
int k_normalize_queries(const void *q, int q_dtype, int nq, int nq_pad, int dim, int ld, float *out_f32, void *out_bf16,
                        int32_t *zero_me, uint32_t *zero_tab, int zero_tab_n, int tf32_round, int split, bool pdl, cudaStream_t st);
int k_synth_fill(void *rows, int dtype, uint64_t seed, int64_t row0, int64_t n, int dim, int ld, uint64_t dup_period,
                 cudaStream_t st);
int k_merge_candidates(const uint64_t *cand, int lists, int nq, int kp, uint64_t *merged, cudaStream_t st);

int k_slab_top(const SelectArgs &sa, int nq, int kp, uint64_t *merged, int *incomplete, cudaStream_t st);
int k_rescore(const RescoreArgs &a, cudaStream_t st, const int *incomplete);
int k_select_rescore(const SelectArgs &sa, const RescoreArgs &a, cudaStream_t st, bool pdl);
bool select_rescore_fits(int lists, int list_len, int kp, int dtype, int dim, int ld);
int k_collect_rescore(const uint64_t *buf, const int *cnt, int cap, const RescoreArgs &a, cudaStream_t st);
int k_exact(const ExactArgs &a, cudaStream_t st, bool pdl);
int k_merge_topk_lists(const void *idx, const void *score, const void *count, size_t stride_bytes, int lists, int nq, int k,
                       int64_t *out_idx, double *out_score, int32_t *out_count, cudaStream_t st);
int k_p2p_publish(void *flag, unsigned long long gen, cudaStream_t st);
int k_merge_topk_p2p(void *const *peers, int nranks, size_t slot_off, size_t flag_off, unsigned long long gen, int nq, int k,
                     int64_t *out_idx, double *out_score, int32_t *out_count, cudaStream_t st);
int k_merge_max_by_id(const int64_t *idx, const double *score, const int32_t *count, int nq, int k, int k2,
                      int64_t *out_idx, double *out_score, int32_t *out_count, cudaStream_t st);
int k_cosine_pairs(const void *a, const void *b, int dtype, int64_t n, int dim, int zero_rule, int sum_mode, double *out,
                   cudaStream_t st);
int k_pairs_above(int device, const void *x, int dtype, int64_t n, int dim, int ld, float threshold, int64_t cap,
                  int64_t *out_i, int64_t *out_j, float *out_score, int64_t *out_count, int part, int nparts, int flags,
                  cudaStream_t st);
int k_pairs_concat(const void *gathered, size_t per_rank_bytes, int64_t slot, const int64_t *counts, int nranks, int64_t cap,
                   int64_t *out_i, int64_t *out_j, float *out_score, int64_t *out_count, cudaStream_t st);

// growable device ranges (arena.cu): a reserved virtual range, physically backed from its start as the store grows
struct Arena;
int arena_create(Arena **out, int device, size_t max_bytes);
int arena_grow(Arena *a, size_t bytes);
void arena_destroy(Arena *a);
void *arena_base(const Arena *a);
size_t arena_mapped(const Arena *a);

static constexpr int MAXQ = 64;   // queries per scan pass
static constexpr int MAXK = 64;   // k and candidate-list bound
static constexpr int XCTAS = 148; // exact-scan grid
static constexpr int MAX_DEVICES = 64;
static constexpr int COLLECT_CAP = 4096;         // rows per query the collect pass may gather
static constexpr int FLAG_INTERNAL_CAPTURE = 1 << 30;  // set by the CUDA-graph path while capturing

// The top-k results of a batch as one contiguous block [idx nq*k i64 | score nq*k f64 | count nq i32], so that one
// copy moves all three arrays: the host readback, the all-gather and the peer-exchange slot all use this layout.
struct ResultBlock {
    int64_t *idx;
    double *score;
    int32_t *count;
    static ResultBlock at(void *base, int nq, int k)
    {
        char *b = (char *)base;
        return {(int64_t *)b, (double *)(b + (size_t)nq * k * 8), (int32_t *)(b + (size_t)nq * k * 16)};
    }
    // the rows of query q0 onwards in three separate [nq][k], [nq][k], [nq] arrays
    ResultBlock from(int q0, int k) const { return {idx + (size_t)q0 * k, score + (size_t)q0 * k, count + q0}; }
};
static constexpr size_t result_bytes(int nq, int k) { return (size_t)nq * k * 16 + (size_t)nq * 4; }
// one rank's block of the cross-shard exchange: the result block padded to 8 bytes
static constexpr size_t packed_bytes(int nq, int k) { return (result_bytes(nq, k) + 7) & ~(size_t)7; }

// copies a result block from (pinned) host memory into the caller's three arrays
static void unpack_to_host(const void *pack, int nq, int k, const ResultBlock &out)
{
    const ResultBlock p = ResultBlock::at(const_cast<void *>(pack), nq, k);
    memcpy(out.idx, p.idx, (size_t)nq * k * 8);
    memcpy(out.score, p.score, (size_t)nq * k * 8);
    memcpy(out.count, p.count, (size_t)nq * 4);
}

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

struct Buf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need)
    {
        if (need <= bytes) return VM_OK;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e)); return VM_ERR_OOM; }
        bytes = need;
        return VM_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

struct Workspace {
    bool ready = false;
    int lists_max = 0;
    Buf q_raw, q_f32, q_bf16, seed, cand, merged, o_idx, flags, col_thr, col_cnt, col_buf, xs, xr, xc, taken, gather_send, gather_recv, misc, ubuf, done, scnt, sel_inc;
    int32_t *h_uncert = nullptr;  // pinned
    unsigned char *h_pack = nullptr;  // pinned: the ResultBlock of one batch
    unsigned char *h_q = nullptr;     // pinned: host queries of one batch
    void release()
    {
        Buf *all[] = {&q_raw, &q_f32, &q_bf16, &seed, &cand, &merged, &o_idx, &flags, &col_thr, &col_cnt, &col_buf, &xs, &xr, &xc, &taken,
                      &gather_send, &gather_recv, &misc, &ubuf, &done, &scnt, &sel_inc};
        for (Buf *b : all) b->release();
        if (h_uncert) cudaFreeHost(h_uncert);
        if (h_pack) cudaFreeHost(h_pack);
        if (h_q) cudaFreeHost(h_q);
        h_uncert = nullptr; h_pack = nullptr; h_q = nullptr;
        ready = false;
    }
};

}  // namespace vm

using namespace vm;

struct vm_store {
    int device = 0, dim = 0, ld = 0, dtype = VM_F32, sm_count = 148;
    int64_t capacity = 0, size = 0;
    void *rows = nullptr;
    float *inv_norms = nullptr;
    // binary64 store (vm_store_create_exact / vm_store_attach_exact): the rows as the caller gave them, [capacity][ld]
    // doubles.  `rows` is then their rounded SHADOW in `dtype`, which only the scan reads; every exact pass
    // (rescoring, band, collect, binary64 scan) reads rows_exact, so scores and order are those of the originals.
    double *rows_exact = nullptr;
    bool owns = false;
    // growable store (vm_store_create_growable): the three buffers live in reserved virtual ranges that are backed
    // with physical memory as `capacity` grows towards max_capacity; base addresses never move (arena.cu)
    Arena *ar_rows = nullptr, *ar_inv = nullptr, *ar_exact = nullptr;
    int64_t max_capacity = 0;
    const void *exact_rows() const { return rows_exact ? (const void *)rows_exact : (const void *)rows; }
    int exact_dtype() const { return rows_exact ? (int)VM_F64 : dtype; }
    int *extreme = nullptr;  // device counter: rows outside the fast scans' numeric range
    unsigned long long *cum = nullptr;  // device, [4]: lifetime certification counters (RescoreArgs::cum)
    int64_t n_batches = 0, n_queries = 0;  // host side of vm_store_read_counters
    int last_band_ctas = 0, last_band_nq = 0;  // shape of the slab counters the last tcgen05 band scan left (vm_store_band_keys)
    Buf stage, stage_idx;
    Workspace ws;
    // VM_FLAG_TIMING: a ring of event pairs, one per timed call, so a whole timed loop can be read back afterwards
    static constexpr int EV_RING = 64;
    cudaEvent_t evr[EV_RING][2] = {};
    int ev_next = 0;     // slot the next timed call records into
    int ev_pending = 0;  // timed calls since the last vm_store_avg_scan_ms (capped at EV_RING)
    int ev_cur = -1;     // slot of the call in flight / most recent call
    bool timed = false;
    // CUDA-graph cache of the host-buffer top-k pipeline (launch-bound small stores / small batches)
    struct GraphEntry {
        cudaGraphExec_t exec = nullptr;
        uint64_t version = 0;
        int nq = 0, k = 0, flags = 0, score_mode = 0, sum_mode = 0, q_dtype = 0;
        double min_score = 0.0;
        int64_t row_offset = 0;  // baked into the captured FinalizeArgs
        vm_topk_stats stats{};
    };
    GraphEntry graphs[4];
    int graph_next = 0;
    uint64_t version = 1;         // bumped by every mutation: cached graphs bake in row counts and TMA descriptors
    uint64_t seen_version = 0;    // version at the previous top-k call
    int stable_calls = 0;         // consecutive top-k calls without a mutation in between
    cudaStream_t gstream = nullptr;  // blocking stream the graphs run on (ordered with the legacy default stream)
};

// exchange buffer of one rank: two result slots + a generation flag
static constexpr size_t XCHG_SLOT_BYTES = (result_bytes(MAXQ, MAXK) + 255) & ~(size_t)255;
static constexpr size_t XCHG_FLAG_OFF = 2 * XCHG_SLOT_BYTES;
static constexpr size_t XCHG_BYTES = XCHG_FLAG_OFF + 256;

struct vm_comm {
    void *nccl = nullptr;  // ncclComm_t
    int nranks = 1, rank = 0, device = 0;
    void *peer[16] = {};   // peer-mapped exchange buffers (optional, see vm_comm_attach_peer_buffers)
    bool p2p = false;
    unsigned long long gen = 0;
    // vm_pairs_above_sharded: local hit lists, gathered counts and gathered lists
    Buf pl_i, pl_j, pl_s, pl_cnt, pg_cnt, pg_send, pg_recv;
    int64_t *h_counts = nullptr;  // pinned [nranks]
};

// ---- NCCL, resolved at run time so the library loads on hosts without it --------------------
struct Id128 { char b[128]; };
namespace {
struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, /*ncclUniqueId by value*/ Id128, int) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
}  // namespace
static NcclApi g_nccl;

static int nccl_load()
{
    if (g_nccl.h) return VM_OK;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    VM_REQUIRE(h, VM_ERR_NCCL, "cannot load libnccl.so.2: %s", dlerror());
    g_nccl.GetUniqueId = (int (*)(void *))dlsym(h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void **, int, Id128, int))dlsym(h, "ncclCommInitRank");
    g_nccl.AllGather = (int (*)(const void *, void *, size_t, int, void *, cudaStream_t))dlsym(h, "ncclAllGather");
    g_nccl.Broadcast = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))dlsym(h, "ncclBroadcast");
    g_nccl.CommDestroy = (int (*)(void *))dlsym(h, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char *(*)(int))dlsym(h, "ncclGetErrorString");
    VM_REQUIRE(g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.AllGather && g_nccl.Broadcast && g_nccl.CommDestroy, VM_ERR_NCCL,
               "libnccl lacks a required symbol");
    g_nccl.h = h;
    return VM_OK;
}
#define VM_NCCL_CHECK(expr)                                                                            \
    do {                                                                                               \
        int _r = (expr);                                                                               \
        if (_r != 0) {                                                                                 \
            set_error("%s failed: %s", #expr, g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "?"); \
            return VM_ERR_NCCL;                                                                        \
        }                                                                                              \
    } while (0)

// ---- small helpers ----------------------------------------------------------------------------
static int check_arch(int device, int *sm_count)
{
    cudaDeviceProp p;
    VM_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    VM_REQUIRE(p.major == 10, VM_ERR_UNSUPPORTED, "device %d is sm_%d%d; libvidmem is built for sm_100a only", device,
               p.major, p.minor);
    if (sm_count) *sm_count = p.multiProcessorCount;
    return VM_OK;
}

static int ws_prepare(vm_store *s)
{
    Workspace &w = s->ws;
    if (w.ready) return VM_OK;
    int lists = 2 * s->sm_count;
    w.lists_max = lists;
    int rc;
#define ENS(b, bytes) if ((rc = (b).ensure(bytes)) != VM_OK) return rc
    ENS(w.q_raw, (size_t)MAXQ * s->dim * 8);
    ENS(w.q_f32, (size_t)MAXQ * s->ld * 4);
    ENS(w.q_bf16, (size_t)2 * MAXQ * s->ld * 2);  // hi terms, then lo terms (split query)
    ENS(w.cand, (size_t)lists * MAXQ * (MAXK > SCAN_SLAB ? MAXK : SCAN_SLAB) * 8);  // per-CTA lists / dumped tiles / slabs
    ENS(w.merged, (size_t)MAXQ * MAXK * 8);
    ENS(w.o_idx, result_bytes(MAXQ, MAXK) + 64);
    ENS(w.flags, (size_t)(MAXQ + 2) * 4);
    // per-CTA maxima [256][64] + published per-query bounds [64] + their counter [64] + union-buffer counters [64] (scan_tc.cu);
    // zeroed as one block by the normalise kernel
    ENS(w.seed, (size_t)(SEED_TAB_WORDS + 3 * MAXQ) * 4);
    ENS(w.ubuf, (size_t)MAXQ * SCAN_UNION_CAP * 8);
    ENS(w.done, 64);
    ENS(w.scnt, (size_t)256 * MAXQ * 4);
    ENS(w.sel_inc, (size_t)MAXQ * 4);
    VM_CUDA_CHECK(cudaMemset(w.done.p, 0, 64));
    ENS(w.col_thr, (size_t)MAXQ * 4);
    ENS(w.col_cnt, (size_t)MAXQ * 4);
    ENS(w.col_buf, (size_t)MAXQ * COLLECT_CAP * 8);
    ENS(w.xs, (size_t)XCTAS * MAXQ * MAXK * 8);
    ENS(w.xr, (size_t)XCTAS * MAXQ * MAXK * 4);
    ENS(w.xc, (size_t)XCTAS * MAXQ * 4);
    ENS(w.taken, (size_t)MAXQ * XCTAS * MAXK);
#undef ENS
    VM_CUDA_CHECK(cudaMallocHost((void **)&w.h_uncert, 64));
    VM_CUDA_CHECK(cudaMallocHost((void **)&w.h_pack, result_bytes(MAXQ, MAXK) + 64));
    VM_CUDA_CHECK(cudaMallocHost((void **)&w.h_q, (size_t)MAXQ * s->dim * 8));
    w.ready = true;
    return VM_OK;
}

static double scan_eps_stored(int kernel, int store_dtype, int dim, int split);
// shadow: the store keeps binary64 originals and the scan reads their rounded copy.  Rounding a row moves its
// direction by an angle of at most asin(u) (u = unit roundoff of the shadow type, relative per element, hence relative
// in norm), and a cosine moves by at most the angle: + 2^-24 (fp32 shadow) or + 2^-9 (bf16 shadow), taken with margin.
static double scan_eps(int kernel, int store_dtype, int dim, int split, bool shadow = false)
{
    const double base = scan_eps_stored(kernel, store_dtype, dim, split);
    if (!shadow) return base;
    return base + (store_dtype == VM_F32 ? 1.1920928955078125e-07 : 1.953125e-3 * 1.01);
}
static double scan_eps_stored(int kernel, int store_dtype, int dim, int split)
{
    // Bound on |approximate cosine - exact cosine| (DESIGN.md "certification"), in cosine units (Cauchy-Schwarz).
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

// ---- library --------------------------------------------------------------------------------
extern "C" int vm_version(void) { return VM_ABI_VERSION; }
extern "C" const char *vm_last_error(void) { return g_err; }

extern "C" int vm_device_info(int device, int *sm_count, int *cc_major, int *cc_minor, size_t *total_mem)
{
    cudaDeviceProp p;
    VM_CUDA_CHECK(cudaGetDeviceProperties(&p, device));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem) *total_mem = p.totalGlobalMem;
    return VM_OK;
}

extern "C" int vm_ld(int dim) { return ld_for_dim(dim); }

// ---- store -----------------------------------------------------------------------------------
static int store_new(vm_store **out, int device, int dim, int dtype, int64_t capacity)
{
    VM_REQUIRE(out, VM_ERR_BADARG, "out is NULL");
    VM_REQUIRE(dim >= 1 && dim <= 4096, VM_ERR_BADARG, "dim %d outside [1, 4096]", dim);
    VM_REQUIRE(dtype == VM_F32 || dtype == VM_BF16, VM_ERR_BADARG, "store dtype must be VM_F32 or VM_BF16");
    VM_REQUIRE(capacity >= 1 && capacity < 0xFFFFFFFFLL, VM_ERR_BADARG, "capacity %lld outside [1, 2^32-2]", (long long)capacity);
    int sms = 0;
    int rc = check_arch(device, &sms);
    if (rc != VM_OK) return rc;
    vm_store *s = new (std::nothrow) vm_store();
    VM_REQUIRE(s, VM_ERR_OOM, "host allocation failed");
    s->device = device; s->dim = dim; s->ld = ld_for_dim(dim); s->dtype = dtype; s->capacity = capacity; s->sm_count = sms;
    {
        DeviceGuard g(device);
        if (cudaMalloc((void **)&s->extreme, 4) != cudaSuccess || cudaMemset(s->extreme, 0, 4) != cudaSuccess ||
            cudaMalloc((void **)&s->cum, 64) != cudaSuccess || cudaMemset(s->cum, 0, 64) != cudaSuccess) {
            set_error("store allocation failed");
            vm_store_destroy(s);
            return VM_ERR_OOM;
        }
    }
    *out = s;
    return VM_OK;
}

extern "C" int vm_store_create(vm_store **out, int device, int dim, int dtype, int64_t capacity)
{
    int rc = store_new(out, device, dim, dtype, capacity);
    if (rc != VM_OK) return rc;
    vm_store *s = *out;
    DeviceGuard g(device);
    s->owns = true;
    size_t bytes = (size_t)capacity * s->ld * dtype_size(dtype);
    cudaError_t e = cudaMalloc(&s->rows, bytes);
    if (e == cudaSuccess) e = cudaMalloc((void **)&s->inv_norms, (size_t)capacity * 4);
    if (e != cudaSuccess) {
        set_error("store allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
        vm_store_destroy(s);
        *out = nullptr;
        return VM_ERR_OOM;
    }
    return VM_OK;
}

extern "C" int vm_store_create_exact(vm_store **out, int device, int dim, int shadow_dtype, int64_t capacity)
{
    int rc = vm_store_create(out, device, dim, shadow_dtype, capacity);
    if (rc != VM_OK) return rc;
    vm_store *s = *out;
    DeviceGuard g(device);
    const size_t bytes = (size_t)capacity * s->ld * 8;
    cudaError_t e = cudaMalloc((void **)&s->rows_exact, bytes);
    if (e != cudaSuccess) {
        set_error("store allocation of %zu bytes (binary64 rows) failed: %s", bytes, cudaGetErrorString(e));
        vm_store_destroy(s);
        *out = nullptr;
        return VM_ERR_OOM;
    }
    return VM_OK;
}

// back the first `capacity` rows of a growable store
static int store_back(vm_store *s, int64_t capacity)
{
    int rc = arena_grow(s->ar_rows, (size_t)capacity * s->ld * dtype_size(s->dtype));
    if (rc == VM_OK) rc = arena_grow(s->ar_inv, (size_t)capacity * 4);
    if (rc == VM_OK && s->ar_exact) rc = arena_grow(s->ar_exact, (size_t)capacity * s->ld * 8);
    return rc;
}

extern "C" int vm_store_create_growable(vm_store **out, int device, int dim, int dtype, int exact, int64_t initial_capacity,
                                        int64_t max_capacity)
{
    VM_REQUIRE(initial_capacity >= 1 && max_capacity >= initial_capacity, VM_ERR_BADARG, "need 1 <= initial_capacity <= max_capacity");
    int rc = store_new(out, device, dim, dtype, max_capacity);   // validates dim / dtype / the row-count limit
    if (rc != VM_OK) return rc;
    vm_store *s = *out;
    DeviceGuard g(device);
    s->max_capacity = max_capacity;
    s->capacity = initial_capacity;
    rc = arena_create(&s->ar_rows, device, (size_t)max_capacity * s->ld * dtype_size(dtype));
    if (rc == VM_OK) rc = arena_create(&s->ar_inv, device, (size_t)max_capacity * 4);
    if (rc == VM_OK && exact) rc = arena_create(&s->ar_exact, device, (size_t)max_capacity * s->ld * 8);
    if (rc == VM_OK) rc = store_back(s, initial_capacity);
    if (rc != VM_OK) { vm_store_destroy(s); *out = nullptr; return rc; }
    s->rows = arena_base(s->ar_rows);
    s->inv_norms = (float *)arena_base(s->ar_inv);
    if (exact) s->rows_exact = (double *)arena_base(s->ar_exact);
    return VM_OK;
}

extern "C" int vm_store_reserve(vm_store *s, int64_t capacity)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    if (capacity <= s->capacity) return VM_OK;
    VM_REQUIRE(s->ar_rows, VM_ERR_STATE, "store is not growable (created over fixed buffers of %lld rows)", (long long)s->capacity);
    VM_REQUIRE(capacity <= s->max_capacity, VM_ERR_OVERFLOW, "capacity %lld exceeds the reserved maximum %lld", (long long)capacity,
               (long long)s->max_capacity);
    DeviceGuard g(s->device);
    int rc = store_back(s, capacity);   // maps new physical chunks behind the resident rows; nothing is copied or moved
    if (rc != VM_OK) return rc;
    s->capacity = capacity;
    return VM_OK;
}

extern "C" int64_t vm_store_max_capacity(const vm_store *s) { return s ? (s->ar_rows ? s->max_capacity : s->capacity) : -1; }
extern "C" void *vm_store_rows_ptr(const vm_store *s) { return s ? s->rows : nullptr; }
extern "C" float *vm_store_inv_norms_ptr(const vm_store *s) { return s ? s->inv_norms : nullptr; }
extern "C" double *vm_store_rows_exact_ptr(const vm_store *s) { return s ? s->rows_exact : nullptr; }
extern "C" size_t vm_store_resident_bytes(const vm_store *s)
{
    if (!s) return 0;
    if (s->ar_rows) return arena_mapped(s->ar_rows) + arena_mapped(s->ar_inv) + (s->ar_exact ? arena_mapped(s->ar_exact) : 0);
    return (size_t)s->capacity * ((size_t)s->ld * (dtype_size(s->dtype) + (s->rows_exact ? 8 : 0)) + 4);
}

extern "C" int vm_store_attach_exact(vm_store **out, int device, int dim, int shadow_dtype, int64_t capacity, void *rows_dev,
                                     float *inv_norms_dev, double *rows_exact_dev)
{
    VM_REQUIRE(rows_exact_dev && ((uintptr_t)rows_exact_dev & 15) == 0, VM_ERR_BADARG, "binary64 rows buffer must be 16-byte aligned");
    int rc = vm_store_attach(out, device, dim, shadow_dtype, capacity, rows_dev, inv_norms_dev);
    if (rc != VM_OK) return rc;
    (*out)->rows_exact = rows_exact_dev;
    return VM_OK;
}

extern "C" int vm_store_attach(vm_store **out, int device, int dim, int dtype, int64_t capacity, void *rows_dev,
                               float *inv_norms_dev)
{
    VM_REQUIRE(rows_dev && inv_norms_dev, VM_ERR_BADARG, "attach needs device buffers");
    VM_REQUIRE(((uintptr_t)rows_dev & 127) == 0, VM_ERR_BADARG, "rows buffer must be 128-byte aligned");
    int rc = store_new(out, device, dim, dtype, capacity);
    if (rc != VM_OK) return rc;
    (*out)->rows = rows_dev;
    (*out)->inv_norms = inv_norms_dev;
    (*out)->owns = false;
    return VM_OK;
}

extern "C" int vm_store_destroy(vm_store *s)
{
    if (!s) return VM_OK;
    DeviceGuard g(s->device);
    cudaDeviceSynchronize();
    if (s->owns) { cudaFree(s->rows); cudaFree(s->inv_norms); if (s->rows_exact) cudaFree(s->rows_exact); }
    arena_destroy(s->ar_rows); arena_destroy(s->ar_inv); arena_destroy(s->ar_exact);
    if (s->extreme) cudaFree(s->extreme);
    if (s->cum) cudaFree(s->cum);
    s->stage.release(); s->stage_idx.release();
    s->ws.release();
    for (auto &pr : s->evr) { if (pr[0]) cudaEventDestroy(pr[0]); if (pr[1]) cudaEventDestroy(pr[1]); }
    for (auto &ge : s->graphs) if (ge.exec) cudaGraphExecDestroy(ge.exec);
    if (s->gstream) cudaStreamDestroy(s->gstream);
    delete s;
    return VM_OK;
}

extern "C" int64_t vm_store_size(const vm_store *s) { return s ? s->size : -1; }
extern "C" int64_t vm_store_capacity(const vm_store *s) { return s ? s->capacity : -1; }
extern "C" int vm_store_dim(const vm_store *s) { return s ? s->dim : -1; }
extern "C" int vm_store_ld(const vm_store *s) { return s ? s->ld : -1; }

static int store_write(vm_store *s, int64_t row0, const void *rows, int src_dtype, int src_mem, int64_t n, cudaStream_t st)
{
    VM_REQUIRE(src_dtype == VM_F32 || src_dtype == VM_BF16 || src_dtype == VM_F64, VM_ERR_BADARG, "bad source dtype");
    if (n == 0) return VM_OK;
    VM_REQUIRE(rows, VM_ERR_BADARG, "rows is NULL");
    DeviceGuard g(s->device);
    const void *src = rows;
    if (src_mem == VM_MEM_HOST) {
        size_t bytes = (size_t)n * s->dim * dtype_size(src_dtype);
        int rc = s->stage.ensure(bytes);
        if (rc != VM_OK) return rc;
        VM_CUDA_CHECK(cudaMemcpyAsync(s->stage.p, rows, bytes, cudaMemcpyHostToDevice, st));
        src = s->stage.p;
    }
    char *dst = (char *)s->rows + (size_t)row0 * s->ld * dtype_size(s->dtype);
    int rc = k_convert_rows(src, src_dtype, dst, s->dtype, n, s->dim, s->ld, st);
    if (rc != VM_OK) return rc;
    if (s->rows_exact) {  // the originals, widened exactly (or copied) into the binary64 rows
        rc = k_convert_rows(src, src_dtype, s->rows_exact + (size_t)row0 * s->ld, VM_F64, n, s->dim, s->ld, st);
        if (rc != VM_OK) return rc;
    }
    return k_row_inv_norms(s->rows, s->dtype, s->inv_norms, row0, row0 + n, s->ld, s->extreme, st, s->rows_exact);
}

extern "C" int vm_store_append(vm_store *s, const void *rows, int src_dtype, int src_mem, int64_t n, int64_t *first_row,
                               void *stream)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    VM_REQUIRE(n >= 0, VM_ERR_BADARG, "n < 0");
    if (s->ar_rows && s->size + n > s->capacity) {
        // growable store: back more of the reserved range -- what this append needs, plus 256 MB worth of rows of slack
        // (capped at the maximum).  Mapping costs time in proportion to the NEW memory only (0.26 ms per 256 MB measured;
        // it can stall behind other users of the driver's resource-manager lock, e.g. a process polling NVML every few
        // milliseconds), so a bounded step keeps the worst insert latency of a streaming store well under a millisecond;
        // resident rows stay put either way.
        const int64_t row_bytes = (int64_t)s->ld * (int64_t)(dtype_size(s->dtype) + (s->rows_exact ? 8 : 0)) + 4;
        const int64_t slack_rows = ((int64_t)256 << 20) / row_bytes + 1;
        int64_t want = s->size + n + slack_rows;
        if (want > s->max_capacity) want = s->max_capacity;
        if (want >= s->size + n) {
            int rc = vm_store_reserve(s, want);
            if (rc != VM_OK && want > s->size + n) rc = vm_store_reserve(s, s->size + n);   // out of memory for the slack: take what is needed
            if (rc != VM_OK) return rc;
        }
    }
    VM_REQUIRE(s->size + n <= s->capacity, VM_ERR_OVERFLOW, "append of %lld rows exceeds capacity %lld (size %lld)",
               (long long)n, (long long)s->capacity, (long long)s->size);
    int rc = store_write(s, s->size, rows, src_dtype, src_mem, n, (cudaStream_t)stream);
    if (rc != VM_OK) return rc;
    if (first_row) *first_row = s->size;
    s->size += n;
    ++s->version;
    return VM_OK;
}

extern "C" int vm_store_update(vm_store *s, int64_t row0, const void *rows, int src_dtype, int src_mem, int64_t n, void *stream)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    VM_REQUIRE(row0 >= 0 && n >= 0 && row0 + n <= s->size, VM_ERR_BADARG, "update range [%lld, %lld) outside [0, %lld)",
               (long long)row0, (long long)(row0 + n), (long long)s->size);
    ++s->version;
    return store_write(s, row0, rows, src_dtype, src_mem, n, (cudaStream_t)stream);
}

extern "C" int vm_store_invalidate(vm_store *s, const int64_t *rows_host, int64_t n, void *stream)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    if (n <= 0) return VM_OK;
    VM_REQUIRE(rows_host, VM_ERR_BADARG, "rows is NULL");
    DeviceGuard g(s->device);
    int rc = s->stage_idx.ensure((size_t)n * 8);
    if (rc != VM_OK) return rc;
    VM_CUDA_CHECK(cudaMemcpyAsync(s->stage_idx.p, rows_host, (size_t)n * 8, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    ++s->version;
    return k_invalidate_rows(s->inv_norms, (const int64_t *)s->stage_idx.p, n, s->size, (cudaStream_t)stream);
}

extern "C" int vm_store_set_size(vm_store *s, int64_t n, int64_t recompute_from_row, void *stream)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    VM_REQUIRE(n >= 0 && n <= s->capacity, VM_ERR_BADARG, "size %lld outside [0, capacity]", (long long)n);
    DeviceGuard g(s->device);
    s->size = n;
    ++s->version;
    if (recompute_from_row >= 0 && recompute_from_row < n) {
        if (s->rows_exact) {
            // rows filled in place are shadow values (vm_synth_fill): their binary64 originals are those values, widened.
            // The shadow is [n][ld] with leading dimension ld, so it converts as a dense [n][ld] source.
            const int64_t r0 = recompute_from_row;
            int rc = k_convert_rows((const char *)s->rows + (size_t)r0 * s->ld * dtype_size(s->dtype), s->dtype,
                                    s->rows_exact + (size_t)r0 * s->ld, VM_F64, n - r0, s->ld, s->ld, (cudaStream_t)stream);
            if (rc != VM_OK) return rc;
        }
        return k_row_inv_norms(s->rows, s->dtype, s->inv_norms, recompute_from_row, n, s->ld, s->extreme, (cudaStream_t)stream, s->rows_exact);
    }
    return VM_OK;
}

extern "C" int vm_store_last_scan_ms(vm_store *s, float *ms)
{
    VM_REQUIRE(s && ms, VM_ERR_BADARG, "NULL argument");
    VM_REQUIRE(s->timed, VM_ERR_STATE, "no vm_topk call with VM_FLAG_TIMING has run the scan kernel yet");
    DeviceGuard g(s->device);
    VM_CUDA_CHECK(cudaEventSynchronize(s->evr[s->ev_cur][1]));
    VM_CUDA_CHECK(cudaEventElapsedTime(ms, s->evr[s->ev_cur][0], s->evr[s->ev_cur][1]));
    return VM_OK;
}

extern "C" int vm_store_avg_scan_ms(vm_store *s, float *ms, int *calls)
{
    VM_REQUIRE(s && ms, VM_ERR_BADARG, "NULL argument");
    VM_REQUIRE(s->timed && s->ev_pending > 0, VM_ERR_STATE, "no vm_topk call with VM_FLAG_TIMING since the last read");
    DeviceGuard g(s->device);
    VM_CUDA_CHECK(cudaEventSynchronize(s->evr[s->ev_cur][1]));
    double sum = 0.0;
    const int n = s->ev_pending;
    for (int i = 0; i < n; ++i) {
        const int slot = (s->ev_cur - i + 2 * vm_store::EV_RING) % vm_store::EV_RING;
        float t = 0.0f;
        VM_CUDA_CHECK(cudaEventElapsedTime(&t, s->evr[slot][0], s->evr[slot][1]));
        sum += t;
    }
    *ms = (float)(sum / n);
    if (calls) *calls = n;
    s->ev_pending = 0;
    return VM_OK;
}

// How many keys the last tcgen05 scan kept (a measure of how tight its bounds were): per query, keys appended to the
// per-CTA slabs (incl. those that went on to the spill buffer) and keys spilled.  Synchronises with the device.
extern "C" int vm_store_band_keys(vm_store *s, int nq_cap, int64_t *kept_per_query, int64_t *spilled_per_query, int *nq_out)
{
    VM_REQUIRE(s && kept_per_query && spilled_per_query, VM_ERR_BADARG, "NULL argument");
    VM_REQUIRE(s->ws.ready && s->last_band_ctas > 0, VM_ERR_STATE, "the last top-k call of this store was not a band-keeping tcgen05 scan");
    const int ctas = s->last_band_ctas, nq = s->last_band_nq;
    VM_REQUIRE(nq_cap >= nq, VM_ERR_BADARG, "room for %d queries needed", nq);
    DeviceGuard g(s->device);
    VM_CUDA_CHECK(cudaDeviceSynchronize());
    std::vector<int> sc((size_t)ctas * nq), uc(nq);
    VM_CUDA_CHECK(cudaMemcpy(sc.data(), s->ws.scnt.p, sc.size() * 4, cudaMemcpyDeviceToHost));
    VM_CUDA_CHECK(cudaMemcpy(uc.data(), (int *)s->ws.seed.p + SEED_TAB_WORDS + 2 * MAXQ, (size_t)nq * 4, cudaMemcpyDeviceToHost));
    for (int q = 0; q < nq; ++q) {
        int64_t k = 0;
        for (int c = 0; c < ctas; ++c) k += sc[(size_t)c * nq + q];
        kept_per_query[q] = k;
        spilled_per_query[q] = uc[q];
    }
    if (nq_out) *nq_out = nq;
    return VM_OK;
}

extern "C" int vm_store_read_counters(vm_store *s, vm_store_counters *out, int reset)
{
    VM_REQUIRE(s && out, VM_ERR_BADARG, "NULL argument");
    DeviceGuard g(s->device);
    unsigned long long h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    VM_CUDA_CHECK(cudaMemcpy(h, s->cum, sizeof(h), cudaMemcpyDeviceToHost));  // synchronises with the work enqueued so far
    out->batches = s->n_batches; out->queries = s->n_queries;
    out->uncertified = (int64_t)h[0]; out->band_settled = (int64_t)h[1]; out->collect_settled = (int64_t)h[2];
    out->full_rescans = (int64_t)h[3];
    out->bound_violations = (int64_t)h[4];
    if (reset) {
        VM_CUDA_CHECK(cudaMemset(s->cum, 0, sizeof(h)));
        s->n_batches = 0; s->n_queries = 0;
    }
    return VM_OK;
}

extern "C" int vm_store_clear(vm_store *s)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    DeviceGuard g(s->device);
    VM_CUDA_CHECK(cudaMemset(s->extreme, 0, 4));
    s->size = 0;
    ++s->version;
    return VM_OK;
}

// ---- top-k ------------------------------------------------------------------------------------
extern "C" size_t vm_topk_packed_bytes(int nq, int k) { return nq > 0 && k > 0 ? packed_bytes(nq, k) : 0; }

namespace {
struct TopkCall {
    vm_store *s;
    const void *queries;  // host or device, [nq][dim]
    int q_dtype, q_mem, nq, k;
    double min_score;
    int score_mode, sum_mode, flags;
    int64_t row_offset;
    ResultBlock d;  // device destinations for this batch
    cudaStream_t st;
    vm_topk_stats *stats;
    // optional host destinations: results are copied there inside the same synchronisation that reads
    // the uncertified-query counter (one stream sync per batch on the host-buffer path)
    ResultBlock h = {};
};
}  // namespace

// Result wait of the synchronous (host-buffer) calls.  cudaStreamSynchronize may park the thread for work longer
// than ~1 ms and then pays a 0.1-0.2 ms wake-up; a top-k call is latency-critical and short, so poll instead
// (VIDMEM_SYNC=block restores the blocking wait, e.g. on oversubscribed hosts).
static cudaError_t wait_stream(cudaStream_t st, const vm_store *s = nullptr)
{
    static const bool block = [] { const char *e = getenv("VIDMEM_SYNC"); return e && !strcmp(e, "block"); }();
    if (block) return cudaStreamSynchronize(st);
    if (s) {
        // a long scan (big shard) is slept through for ~3/4 of its roofline time, so the host core is not
        // spun for milliseconds; only the last stretch is polled
        const double est_us = (double)s->size * s->ld * (double)dtype_size(s->dtype) / 6.5e6;  // bytes / (6.5 TB/s)
        if (est_us > 400.0) {
            struct timespec ts;
            const long ns = (long)(est_us * 750.0);
            ts.tv_sec = ns / 1000000000L; ts.tv_nsec = ns % 1000000000L;
            nanosleep(&ts, nullptr);
        }
    }
    for (;;) {
        const cudaError_t e = cudaStreamQuery(st);
        if (e != cudaErrorNotReady) return e;
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
}

// Host-output path: the batch's device results are one ResultBlock (see ws_prepare); one D2H copy into pinned
// memory, then plain host copies into the caller's arrays.
static int pack_out_enqueue(const TopkCall &c)
{
    VM_CUDA_CHECK(cudaMemcpyAsync(c.s->ws.h_pack, c.d.idx, result_bytes(c.nq, c.k), cudaMemcpyDeviceToHost, c.st));
    return VM_OK;
}

// candidate-list length of the tcgen05 scan for top-k (0: k is too large for it)
static int tc_list_len(int k) { return k <= 16 ? 32 : (k <= 48 ? 64 : 0); }

// queries per scan pass: 64, or fewer when 64 normalised queries of this dimension do not fit the
// tcgen05 kernel's shared memory (e.g. 16 for a 1536-d fp32 store)
static int queries_per_pass(const vm_store *s, int k, int flags)
{
    const int kp = tc_list_len(k);
    if (!(flags & (VM_FLAG_FORCE_EXACT | VM_FLAG_FORCE_SIMT)) && kp)
        for (int nq = 64; nq >= 16; nq -= 16)
            if (scan_tc_supported(s->dtype, s->dim, nq, kp)) return nq;
    return MAXQ;
}

// One batch of <= MAXQ queries; results land in c.d (device).  May synchronise the stream
// (unless VM_FLAG_ASYNC) to learn whether any query needs the exact re-scan.
static int topk_batch(const TopkCall &c)
{
    vm_store *s = c.s;
    Workspace &w = s->ws;
    cudaStream_t st = c.st;
    const void *q_dev = c.queries;
    if (c.q_mem == VM_MEM_HOST) {
        // pageable host memory would make the copy synchronous: stage through the pinned buffer
        const size_t qbytes = (size_t)c.nq * s->dim * dtype_size(c.q_dtype);
        memcpy(w.h_q, c.queries, qbytes);
        VM_CUDA_CHECK(cudaMemcpyAsync(w.q_raw.p, w.h_q, qbytes, cudaMemcpyHostToDevice, st));
        q_dev = w.q_raw.p;
    }
    FinalizeArgs fin{c.k, c.min_score, c.score_mode, c.row_offset, c.d.idx, c.d.score, c.d.count};
    ExactArgs ex{s->exact_rows(), s->inv_norms, s->exact_dtype(), s->ld, s->dim, s->size, q_dev, c.q_dtype, c.nq, c.k, c.sum_mode,
                 nullptr, (double *)w.xs.p, (uint32_t *)w.xr.p, (int32_t *)w.xc.p, (uint8_t *)w.taken.p, XCTAS, fin, s->cum,
                 (int *)w.done.p};
    if (!(c.flags & FLAG_INTERNAL_CAPTURE)) { ++s->n_batches; s->n_queries += c.nq; }
    int launches = 0;
    if (c.stats) { c.stats->uncertified = 0; c.stats->candidates = 0; c.stats->scan_ctas = 0; }

    // choose the scan kernel
    int kernel = 0, kp = 0;
    if (!(c.flags & VM_FLAG_FORCE_EXACT) && s->size > 0) {
        int kp_tc = tc_list_len(c.k);
        int kp_simt = c.k <= 24 ? (c.k + 8 > 16 ? ((c.k + 8 + 7) & ~7) : 16) : 0;
        bool tc_ok = kp_tc > 0 && scan_tc_supported(s->dtype, s->dim, c.nq, kp_tc);
        // The tcgen05 scan is the default at every size: it streams big shards at the HBM roofline (the CUDA-core
        // kernel reaches ~half of it) and is also the lower-latency choice for a few queries over a small store
        // (measured fp32, 1-8 queries: 5 K rows 39 vs 45-54 us, 60 K rows 55-57 vs 74-123 us).  The CUDA-core kernel
        // serves the shapes the tensor path does not fit (k > 48, dims beyond its shared memory) and cross-checks it.
        bool want_tc = !(c.flags & VM_FLAG_FORCE_SIMT);
        if (want_tc && tc_ok) { kernel = 2; kp = kp_tc; }
        else if (kp_simt > 0) { kernel = 1; kp = kp_simt; }
        else if (tc_ok) { kernel = 2; kp = kp_tc; }
    }
    if (kernel == 0) {
        int rc = k_exact(ex, st, false);
        if (rc != VM_OK) return rc;
        launches += 2;
        if (c.h.idx) {
            if ((rc = pack_out_enqueue(c)) != VM_OK) return rc;
            VM_CUDA_CHECK(wait_stream(st, s));
            unpack_to_host(w.h_pack, c.nq, c.k, c.h);
        }
        if (c.stats) { c.stats->scan_kernel = 0; c.stats->scan_launches += launches; }
        return VM_OK;
    }

    int nq_pad = kernel == 2 ? ((c.nq + 15) & ~15) : c.nq;
    // bf16 store: feed the query as hi + lo bf16 terms (two MMAs per K slice) whenever that layout fits shared memory
    // -- free up to 48 queries per pass (measured, 12.5 M x 384: 1.34 ms either way); at 64 the doubled MMA count makes
    // the tensor pipe the pacing unit (+4..10 %), and since a wide band is settled inside the rescoring kernel anyway
    // the single-term query is the default there (VM_FLAG_SPLIT forces the split, VM_FLAG_NO_SPLIT forbids it)
    const int split = (kernel == 2 && s->dtype == VM_BF16 && !(c.flags & VM_FLAG_NO_SPLIT) &&
                       (c.nq <= 48 || (c.flags & VM_FLAG_SPLIT)) && scan_tc_supported(s->dtype, s->dim, c.nq, kp, 1)) ? 1 : 0;
    // The kernels of one call are chained with programmatic dependent launch (common.cuh): each one's launch and
    // prologue overlap its predecessor's drain -- also inside the captured graph of the host-buffer path (5 K-row store, 30
    // queries: 74.4 -> 70.5 us per call; 1 M rows: no change).  Off while events bracket the scan (VM_FLAG_TIMING).
#ifdef VIDMEM_NO_GRAPH_PDL
    const bool pdl = !(c.flags & (VM_FLAG_TIMING | FLAG_INTERNAL_CAPTURE));   // A/B build: plain edges inside the captured graph
#else
    const bool pdl = !(c.flags & VM_FLAG_TIMING);   // also while a graph is captured: the launches become programmatic edges
#endif
    int rc = k_normalize_queries(q_dev, c.q_dtype, c.nq, nq_pad, s->dim, s->ld, (float *)w.q_f32.p,
                                 (kernel == 2 && s->dtype == VM_BF16) ? w.q_bf16.p : nullptr,
                                 (int32_t *)w.flags.p + c.nq, kernel == 2 ? (uint32_t *)w.seed.p : nullptr,
                                 kernel == 2 ? (int)(w.seed.bytes / 4) : 0, kernel == 2 && s->dtype == VM_F32, split, pdl, st);
    if (rc != VM_OK) return rc;
    ++launches;
    const double eps = scan_eps(kernel, s->dtype, s->dim, split, s->rows_exact != nullptr);

    ScanArgs a;
    ScanInfo sinfo;
    a.rows = s->rows; a.inv_norms = s->inv_norms; a.dtype = s->dtype; a.n = s->size; a.dim = s->dim; a.ld = s->ld;
    a.queries = (const float *)w.q_f32.p; a.nq = c.nq; a.kp = kp; a.cand = (uint64_t *)w.cand.p; a.stream = st;
    a.slab = (uint64_t *)w.cand.p; a.scnt = (int *)w.scnt.p;
    a.ubuf = (uint64_t *)w.ubuf.p; a.ucnt = (int *)w.seed.p + SEED_TAB_WORDS + 2 * MAXQ; a.ucap = SCAN_UNION_CAP;
    a.band = nextafterf((float)(2.0 * eps), INFINITY); a.ksel = c.k; a.split = split; a.pdl = pdl;
    const bool timing = (c.flags & VM_FLAG_TIMING) != 0;
    if (timing) {
        s->ev_cur = s->ev_next;
        s->ev_next = (s->ev_next + 1) % vm_store::EV_RING;
        if (s->ev_pending < vm_store::EV_RING) ++s->ev_pending;
        if (!s->evr[s->ev_cur][0]) { VM_CUDA_CHECK(cudaEventCreate(&s->evr[s->ev_cur][0])); VM_CUDA_CHECK(cudaEventCreate(&s->evr[s->ev_cur][1])); }
        VM_CUDA_CHECK(cudaEventRecord(s->evr[s->ev_cur][0], st));
    }
    if (kernel == 1) {
        int64_t need = (s->size + 31) / 32;
        a.ctas = (int)imin64(need, 2 * s->sm_count);
        rc = launch_scan_simt(a);
        launches += (c.nq + 7) / 8;
    } else {
        int64_t tiles = (s->size + 127) / 128;
        a.ctas = (int)imin64(tiles, s->sm_count);

        // small store: too few tiles per CTA for a threshold to form -> rank every row's key instead
        a.dump = tiles <= s->sm_count && tiles * SCAN_DUMP_TILE <= SCAN_DUMP_MAX_KEYS &&
                 (size_t)tiles * c.nq * SCAN_DUMP_TILE * 8 <= w.cand.bytes &&
                 select_rescore_fits((int)tiles, SCAN_DUMP_TILE, kp, s->exact_dtype(), s->dim, s->ld);
        s->last_band_ctas = a.dump ? 0 : a.ctas; s->last_band_nq = c.nq;   // dump mode keeps every row: no band counters
        rc = launch_scan_tc(a, s->dtype == VM_BF16 ? w.q_bf16.p : w.q_f32.p, (uint32_t *)w.seed.p, (int *)w.flags.p + c.nq + 1, nullptr, &sinfo);
        launches += 1;
    }
    if (rc != VM_OK) return rc;
    if (timing) { VM_CUDA_CHECK(cudaEventRecord(s->evr[s->ev_cur][1], st)); s->timed = true; }

    int32_t *flags = (int32_t *)w.flags.p;
    int32_t *uncert = flags + c.nq;  // counter sits right after the nq flags (zeroed by the normalise kernel)
    RescoreArgs rs{(const uint64_t *)w.merged.p, kp, s->exact_rows(), s->inv_norms, s->exact_dtype(), s->ld, s->dim, s->size, q_dev,
                   c.q_dtype, c.nq, eps, c.sum_mode, fin, flags, uncert, s->extreme,
                   kernel == 2 ? (float *)w.col_thr.p : nullptr, s->cum};
    // where the candidates are: the union buffer of the tcgen05 scan (complete band), its dumped tiles (every row),
    // or the per-CTA top-kp lists of the CUDA-core scan
    SelectArgs sel;
    const bool union_src = kernel == 2 && !a.dump;
    if (union_src) {
        sel.slab = a.slab; sel.scnt = a.scnt; sel.ctas = a.ctas; sel.ubuf = a.ubuf; sel.ucnt = a.ucnt; sel.ucap = a.ucap;
        sel.seed_tab = a.ctas <= 256 ? (const uint32_t *)w.seed.p : nullptr; sel.nq_pad = nq_pad; sel.ksel = c.k; sel.band = a.band;
    } else { sel.cand = a.cand; sel.lists = a.ctas; sel.list_len = a.dump ? SCAN_DUMP_TILE : kp; sel.complete = a.dump ? 1 : 0; }
    rc = k_select_rescore(sel, rs, st, pdl);   // fused selection + exact rescoring + band settlement
    if (rc == VM_ERR_UNSUPPORTED && !a.dump) {  // rows too large for shared memory: two kernels
        if (union_src) rc = k_slab_top(sel, c.nq, kp, (uint64_t *)w.merged.p, (int *)w.sel_inc.p, st);
        else rc = k_merge_candidates(a.cand, a.ctas, c.nq, kp, (uint64_t *)w.merged.p, st);
        if (rc != VM_OK) return rc;
        rc = k_rescore(rs, st, union_src ? (const int *)w.sel_inc.p : nullptr);
        ++launches;
    }
    if (rc != VM_OK) return rc;
    launches += 1;

    ex.flags = flags;
    int n_uncert = 0, n_full = -1;
    // Second chance for uncertified queries of the tensor-core scan: one more scan in collect mode
    // (every row within 2 eps of the exact k-th candidate score) + exact rescoring of what it gathered.
    // Both kernels exit at once when nothing is flagged.  Whatever they cannot settle (buffer overflow,
    // stores with out-of-range rows) is left to the binary64 scan of every row.
    auto run_collect = [&]() -> int {
        VM_CUDA_CHECK(cudaMemsetAsync(w.col_cnt.p, 0, (size_t)c.nq * 4, st));
        ScanCollect sc{(const float *)w.col_thr.p, (uint64_t *)w.col_buf.p, (int *)w.col_cnt.p, COLLECT_CAP, uncert};
        int r = launch_scan_tc(a, s->dtype == VM_BF16 ? w.q_bf16.p : w.q_f32.p, nullptr, nullptr, &sc);
        if (r != VM_OK) return r;
        return k_collect_rescore((const uint64_t *)w.col_buf.p, (const int *)w.col_cnt.p, COLLECT_CAP, rs, st);
    };
    if (c.flags & VM_FLAG_ASYNC) {
        if (c.flags & FLAG_INTERNAL_CAPTURE) {
            // graph replay carries only the common path; the uncertified count goes to the host, which
            // re-runs the batch through the plain path in the rare case it is non-zero
            VM_CUDA_CHECK(cudaMemcpyAsync(w.h_uncert, uncert, 4, cudaMemcpyDeviceToHost, st));
        } else {
            rc = k_exact(ex, st, pdl);  // ONE conditional launch: exits at once when nothing is flagged
            if (rc != VM_OK) return rc;
            launches += 1;
        }
        n_uncert = -1;
    } else {
        VM_CUDA_CHECK(cudaMemcpyAsync(w.h_uncert, uncert, 4, cudaMemcpyDeviceToHost, st));
        if (c.h.idx && (rc = pack_out_enqueue(c)) != VM_OK) return rc;
        VM_CUDA_CHECK(wait_stream(st, s));
        n_uncert = *w.h_uncert;
        n_full = 0;
        if (n_uncert > 0) {
            int left = n_uncert;
            if (kernel == 2) {
                if ((rc = run_collect()) != VM_OK) return rc;
                launches += 2;
                VM_CUDA_CHECK(cudaMemcpyAsync(w.h_uncert, uncert, 4, cudaMemcpyDeviceToHost, st));
                VM_CUDA_CHECK(wait_stream(st, s));
                left = *w.h_uncert;
            }
            n_full = left;
            if (left > 0) {
                rc = k_exact(ex, st, false);
                if (rc != VM_OK) return rc;
                launches += 1;
            }
            if (c.h.idx) {
                if ((rc = pack_out_enqueue(c)) != VM_OK) return rc;
                VM_CUDA_CHECK(wait_stream(st, s));
            }
        }
        if (c.h.idx) unpack_to_host(w.h_pack, c.nq, c.k, c.h);
    }
    if (c.stats) {
        c.stats->scan_kernel = kernel;
        c.stats->scan_launches += launches;
        c.stats->uncertified += n_uncert > 0 ? n_uncert : 0;
        c.stats->full_rescans = n_full;
        c.stats->candidates = kp;
        c.stats->scan_ctas = a.ctas;
        c.stats->scan_stages = kernel == 2 ? sinfo.stages : 0;
        c.stats->scan_variant = kernel == 2 ? sinfo.variant : 0;
    }
    return VM_OK;
}

// topk_graph: the call is not one for the graph path
static constexpr int GRAPH_SKIPPED = 1;

// Captures the pipeline of the one-batch host-buffer call c into cache entry ge: H2D of the pinned queries ->
// normalise -> scan -> select/rescore -> D2H of the uncertified-query count and of the result block.
static int graph_capture(const TopkCall &c, vm_store::GraphEntry *ge)
{
    vm_store *s = c.s;
    Workspace &w = s->ws;
    vm_topk_stats cs{};
    TopkCall cc = c;
    cc.queries = w.q_raw.p; cc.q_mem = VM_MEM_DEVICE; cc.flags |= VM_FLAG_ASYNC | FLAG_INTERNAL_CAPTURE;
    cc.d = ResultBlock::at(w.o_idx.p, c.nq, c.k); cc.st = s->gstream; cc.stats = &cs;
    const size_t qbytes = (size_t)c.nq * s->dim * dtype_size(c.q_dtype);
    cudaGraph_t graph = nullptr;
    VM_CUDA_CHECK(cudaStreamBeginCapture(s->gstream, cudaStreamCaptureModeRelaxed));
    int rc = VM_OK;
    if (cudaMemcpyAsync(w.q_raw.p, w.h_q, qbytes, cudaMemcpyHostToDevice, s->gstream) != cudaSuccess) rc = VM_ERR_CUDA;
    if (rc == VM_OK) rc = topk_batch(cc);
    if (rc == VM_OK && cudaMemcpyAsync(w.h_pack, cc.d.idx, result_bytes(c.nq, c.k), cudaMemcpyDeviceToHost, s->gstream) != cudaSuccess)
        rc = VM_ERR_CUDA;
    cudaError_t ce = cudaStreamEndCapture(s->gstream, &graph);
    if (rc != VM_OK || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        if (rc == VM_OK) { set_error("graph capture failed: %s", cudaGetErrorString(ce)); rc = VM_ERR_CUDA; }
        cudaGetLastError();
        return rc;
    }
    ce = cudaGraphInstantiate(&ge->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) { ge->exec = nullptr; set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); return VM_ERR_CUDA; }
    ge->version = s->version; ge->nq = c.nq; ge->k = c.k; ge->flags = c.flags; ge->score_mode = c.score_mode;
    ge->sum_mode = c.sum_mode; ge->q_dtype = c.q_dtype; ge->min_score = c.min_score; ge->row_offset = c.row_offset; ge->stats = cs;
    return VM_OK;
}

// CUDA-graph fast path: one graph launch runs the whole pipeline of the call (graph_capture), and the
// device-conditional exact re-scan is replaced by a host re-run of the rare uncertified batch.  Host buffers, one
// batch, caller on the legacy default stream (the graph runs on a library-owned blocking stream, which the legacy
// stream orders with).  The graph bakes in row count and TMA descriptors, so it is keyed on the store version.
// c describes the whole call; returns GRAPH_SKIPPED when the call must take the batch loop instead.
static int topk_graph(const TopkCall &c, int out_mem, bool sharded, const ResultBlock &out)
{
    vm_store *s = c.s;
    Workspace &w = s->ws;
    static const bool no_graph = getenv("VIDMEM_NO_GRAPH") != nullptr;
    // capturing costs a few hundred microseconds: only worth it for a store that is being queried, not
    // one that is mutated every few calls (streaming inserts)
    if (s->seen_version == s->version) { if (s->stable_calls < 1 << 20) ++s->stable_calls; }
    else { s->seen_version = s->version; s->stable_calls = 0; }
    if (no_graph || s->stable_calls < 16 || sharded || c.st != nullptr || c.q_mem != VM_MEM_HOST || out_mem != VM_MEM_HOST ||
        (c.flags & (VM_FLAG_ASYNC | VM_FLAG_TIMING | VM_FLAG_FORCE_EXACT)) || s->size == 0 ||
        c.nq > queries_per_pass(s, c.k, c.flags))
        return GRAPH_SKIPPED;
    if (!s->gstream) VM_CUDA_CHECK(cudaStreamCreate(&s->gstream));
    vm_store::GraphEntry *ge = nullptr;
    for (auto &e : s->graphs)
        if (e.exec && e.version == s->version && e.nq == c.nq && e.k == c.k && e.flags == c.flags && e.score_mode == c.score_mode &&
            e.sum_mode == c.sum_mode && e.q_dtype == c.q_dtype && e.row_offset == c.row_offset &&
            memcmp(&e.min_score, &c.min_score, sizeof(double)) == 0) { ge = &e; break; }  // bitwise: a NaN bound must match itself
    if (!ge) {  // capture into the oldest entry
        ge = &s->graphs[s->graph_next];
        s->graph_next = (s->graph_next + 1) & 3;
        if (ge->exec) { cudaGraphExecDestroy(ge->exec); ge->exec = nullptr; }
        const int rc = graph_capture(c, ge);
        if (rc != VM_OK) return rc;
    }
    memcpy(w.h_q, c.queries, (size_t)c.nq * s->dim * dtype_size(c.q_dtype));
    ++s->n_batches; s->n_queries += c.nq;
    VM_CUDA_CHECK(cudaGraphLaunch(ge->exec, s->gstream));
    VM_CUDA_CHECK(wait_stream(s->gstream, s));
    const int uncertified = ge->stats.scan_kernel != 0 ? *w.h_uncert : 0;  // the exact-only pipeline writes no count
    if (uncertified > 0) {
        // some query was not certified: run this batch through the plain path (collect pass / exact scan)
        TopkCall rerun = c;
        rerun.d = ResultBlock::at(w.o_idx.p, c.nq, c.k); rerun.st = s->gstream; rerun.h = out;
        return topk_batch(rerun);
    }
    unpack_to_host(w.h_pack, c.nq, c.k, out);
    if (c.stats) { *c.stats = ge->stats; c.stats->uncertified = uncertified; }
    return VM_OK;
}

// offset of this rank's result slot of exchange generation gen in the peer-mapped buffer (two slots alternate)
static size_t xchg_slot_off(unsigned long long gen) { return (size_t)(gen & 1) * XCHG_SLOT_BYTES; }

// where the local pass of a batch writes its results: this rank's exchange slot (p2p), the all-gather send buffer
// (NCCL), the caller's arrays (device outputs) or the workspace block (host outputs)
static ResultBlock batch_dest(vm_store *s, const vm_comm *comm, bool sharded, int out_mem, const ResultBlock &out, int nb, int k)
{
    if (sharded && comm->p2p) return ResultBlock::at((char *)comm->peer[comm->rank] + xchg_slot_off(comm->gen), nb, k);
    if (sharded) return ResultBlock::at(s->ws.gather_send.p, nb, k);
    return out_mem == VM_MEM_DEVICE ? out : ResultBlock::at(s->ws.o_idx.p, nb, k);
}

// Exchanges the local results of one sharded batch between the ranks -- peer-mapped slots, or ONE all-gather of the
// result blocks -- and merges them into m
static int exchange_merge(vm_store *s, vm_comm *comm, int nb, int k, const ResultBlock &m, cudaStream_t st)
{
    if (comm->p2p) {
        const int rc = k_p2p_publish((char *)comm->peer[comm->rank] + XCHG_FLAG_OFF, comm->gen, st);
        if (rc != VM_OK) return rc;
        return k_merge_topk_p2p(comm->peer, comm->nranks, xchg_slot_off(comm->gen), XCHG_FLAG_OFF, comm->gen, nb, k, m.idx, m.score,
                                m.count, st);
    }
    const Workspace &w = s->ws;
    VM_NCCL_CHECK(g_nccl.AllGather(w.gather_send.p, w.gather_recv.p, packed_bytes(nb, k), /*ncclInt8*/ 0, comm->nccl, st));
    const ResultBlock r = ResultBlock::at(w.gather_recv.p, nb, k);
    return k_merge_topk_lists(r.idx, r.score, r.count, packed_bytes(nb, k), comm->nranks, nb, k, m.idx, m.score, m.count, st);
}

static int topk_common(vm_store *s, vm_comm *comm, int64_t row_offset, const void *queries, int q_dtype, int q_mem, int nq,
                       int k, double min_score, int score_mode, int sum_mode, int flags, int64_t *out_idx,
                       double *out_score, int32_t *out_count, int out_mem, vm_topk_stats *stats, void *stream)
{
    VM_REQUIRE(s, VM_ERR_BADARG, "store is NULL");
    VM_REQUIRE(nq >= 0, VM_ERR_BADARG, "nq < 0");
    VM_REQUIRE(k >= 1 && k <= MAXK, VM_ERR_BADARG, "k %d outside [1, %d]", k, MAXK);
    VM_REQUIRE(q_dtype == VM_F32 || q_dtype == VM_BF16 || q_dtype == VM_F64, VM_ERR_BADARG, "bad query dtype");
    VM_REQUIRE(score_mode == VM_SCORE_RAW || score_mode == VM_SCORE_NEO4J, VM_ERR_BADARG, "bad score_mode");
    VM_REQUIRE(sum_mode == VM_SUM_NAIVE || sum_mode == VM_SUM_NEUMAIER, VM_ERR_BADARG, "bad sum_mode");
    VM_REQUIRE(!(flags & VM_FLAG_ASYNC) || (out_mem == VM_MEM_DEVICE && q_mem == VM_MEM_DEVICE), VM_ERR_BADARG,
               "VM_FLAG_ASYNC needs device queries and device outputs");
    if (stats) memset(stats, 0, sizeof(*stats));
    if (nq == 0) return VM_OK;
    VM_REQUIRE(queries && out_idx && out_score && out_count, VM_ERR_BADARG, "NULL buffer");
    DeviceGuard g(s->device);
    VM_REQUIRE(g.ok, VM_ERR_CUDA, "cannot select device %d", s->device);
    int rc = ws_prepare(s);
    if (rc != VM_OK) return rc;
    const bool sharded = comm && comm->nranks > 1;
    const ResultBlock out{out_idx, out_score, out_count};
    const TopkCall call{s, queries, q_dtype, q_mem, nq, k, min_score, score_mode, sum_mode, flags, row_offset, {}, (cudaStream_t)stream,
                        stats};
    if ((rc = topk_graph(call, out_mem, sharded, out)) != GRAPH_SKIPPED) return rc;

    Workspace &w = s->ws;
    const int bq = queries_per_pass(s, k, flags);
    for (int q0 = 0; q0 < nq; q0 += bq) {
        const int nb = nq - q0 < bq ? nq - q0 : bq;
        const ResultBlock out_b = out.from(q0, k);
        if (sharded && comm->p2p) {
            ++comm->gen;  // a fresh exchange slot and flag value for this batch
        } else if (sharded) {
            if ((rc = w.gather_send.ensure(packed_bytes(nb, k))) != VM_OK) return rc;
            if ((rc = w.gather_recv.ensure(packed_bytes(nb, k) * comm->nranks)) != VM_OK) return rc;
        }
        TopkCall c = call;
        c.queries = (const char *)queries + (size_t)q0 * s->dim * dtype_size(q_dtype);
        c.nq = nb;
        c.d = batch_dest(s, comm, sharded, out_mem, out_b, nb, k);
        if (out_mem == VM_MEM_HOST) {
            // Sharded call with host outputs: enqueue the local pass without a host round trip (uncertified queries
            // are settled by the device-conditional binary64 scan), so scan -> exchange -> merge -> one packed D2H run
            // back to back and the ranks reach the exchange together; the only synchronisation is the final one.
            if (sharded) c.flags |= VM_FLAG_ASYNC;
            else c.h = out_b;
        }
        if ((rc = topk_batch(c)) != VM_OK) return rc;
        if (!sharded) continue;
        const ResultBlock ws = ResultBlock::at(w.o_idx.p, nb, k);
        if ((rc = exchange_merge(s, comm, nb, k, out_mem == VM_MEM_DEVICE ? out_b : ws, c.st)) != VM_OK) return rc;
        if (stats) stats->scan_launches += 2;
        if (out_mem == VM_MEM_HOST) {
            VM_CUDA_CHECK(cudaMemcpyAsync(w.h_pack, ws.idx, result_bytes(nb, k), cudaMemcpyDeviceToHost, c.st));
            VM_CUDA_CHECK(wait_stream(c.st, s));
            unpack_to_host(w.h_pack, nb, k, out_b);
        }
    }
    return VM_OK;
}

extern "C" int vm_topk(vm_store *s, const void *queries, int q_dtype, int q_mem, int nq, int k, double min_score,
                       int score_mode, int sum_mode, int flags, int64_t *out_idx, double *out_score, int32_t *out_count,
                       int out_mem, vm_topk_stats *stats, void *stream)
{
    return topk_common(s, nullptr, 0, queries, q_dtype, q_mem, nq, k, min_score, score_mode, sum_mode, flags, out_idx,
                       out_score, out_count, out_mem, stats, stream);
}

extern "C" int vm_topk_sharded(vm_store *s, vm_comm *comm, int64_t row_offset, const void *queries, int q_dtype, int q_mem,
                               int nq, int k, double min_score, int score_mode, int sum_mode, int flags, int64_t *out_idx,
                               double *out_score, int32_t *out_count, int out_mem, vm_topk_stats *stats, void *stream)
{
    VM_REQUIRE(comm, VM_ERR_BADARG, "comm is NULL");
    return topk_common(s, comm, row_offset, queries, q_dtype, q_mem, nq, k, min_score, score_mode, sum_mode, flags, out_idx,
                       out_score, out_count, out_mem, stats, stream);
}

extern "C" int vm_merge_topk_lists(int device, const int64_t *idx_dev, const double *score_dev, const int32_t *count_dev,
                                   int nlists, int nq, int k, int64_t *out_idx_dev, double *out_score_dev,
                                   int32_t *out_count_dev, void *stream)
{
    VM_REQUIRE(idx_dev && score_dev && count_dev && out_idx_dev && out_score_dev && out_count_dev, VM_ERR_BADARG, "NULL buffer");
    VM_REQUIRE(nlists >= 1 && nq >= 1 && k >= 1, VM_ERR_BADARG, "bad shape");
    DeviceGuard g(device);
    // the merge kernel steps from list to list with one stride for all three arrays, so the counts ([nlists][nq]) are
    // copied out to the stride of the idx and score lists
    size_t stride = (size_t)nq * k * 8;
    VM_REQUIRE(device >= 0 && device < MAX_DEVICES, VM_ERR_BADARG, "device index %d outside [0, %d)", device, MAX_DEVICES);
    static thread_local Buf cnt_wide_dev[MAX_DEVICES];  // scratch is device memory: one per device
    Buf &cnt_wide = cnt_wide_dev[device];
    int rc = cnt_wide.ensure(stride * nlists);
    if (rc != VM_OK) return rc;
    VM_CUDA_CHECK(cudaMemcpy2DAsync(cnt_wide.p, stride, count_dev, (size_t)nq * 4, (size_t)nq * 4, nlists,
                                    cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return k_merge_topk_lists(idx_dev, score_dev, cnt_wide.p, stride, nlists, nq, k, out_idx_dev, out_score_dev,
                              out_count_dev, (cudaStream_t)stream);
}

extern "C" int vm_merge_topk_packed(int device, const void *packed_dev, int nlists, int nq, int k, int64_t *out_idx_dev,
                                    double *out_score_dev, int32_t *out_count_dev, void *stream)
{
    VM_REQUIRE(packed_dev && out_idx_dev && out_score_dev && out_count_dev, VM_ERR_BADARG, "NULL buffer");
    VM_REQUIRE(nlists >= 1 && nq >= 1 && k >= 1, VM_ERR_BADARG, "bad shape");
    DeviceGuard g(device);
    const ResultBlock r = ResultBlock::at(const_cast<void *>(packed_dev), nq, k);
    return k_merge_topk_lists(r.idx, r.score, r.count, packed_bytes(nq, k), nlists, nq, k, out_idx_dev, out_score_dev,
                              out_count_dev, (cudaStream_t)stream);
}

extern "C" int vm_merge_max_by_id(int device, const int64_t *idx_dev, const double *score_dev, const int32_t *count_dev,
                                  int nq, int k, int k2, int64_t *out_idx_dev, double *out_score_dev, int32_t *out_count_dev,
                                  void *stream)
{
    VM_REQUIRE(idx_dev && score_dev && count_dev && out_idx_dev && out_score_dev && out_count_dev, VM_ERR_BADARG, "NULL buffer");
    VM_REQUIRE(nq >= 1 && k >= 1 && k2 >= 1, VM_ERR_BADARG, "bad shape");
    DeviceGuard g(device);
    return k_merge_max_by_id(idx_dev, score_dev, count_dev, nq, k, k2, out_idx_dev, out_score_dev, out_count_dev,
                             (cudaStream_t)stream);
}

// ---- scalar cosine seams ----------------------------------------------------------------------
extern "C" int vm_cosine_pairs(int device, const void *a, const void *b, int dtype, int mem, int64_t n, int dim, int zero_rule,
                               int sum_mode, double *out, int out_mem, void *stream)
{
    VM_REQUIRE(n >= 0 && dim >= 0, VM_ERR_BADARG, "bad shape");
    VM_REQUIRE(dtype == VM_F32 || dtype == VM_F64, VM_ERR_BADARG, "dtype must be VM_F32 or VM_F64");
    VM_REQUIRE(zero_rule >= 0 && zero_rule <= 2, VM_ERR_BADARG, "zero_rule %d outside [0, 2]", zero_rule);
    if (n == 0) return VM_OK;
    VM_REQUIRE(a && b && out, VM_ERR_BADARG, "NULL buffer");
    int rc = check_arch(device, nullptr);
    if (rc != VM_OK) return rc;
    DeviceGuard g(device);
    cudaStream_t st = (cudaStream_t)stream;
    VM_REQUIRE(device >= 0 && device < MAX_DEVICES, VM_ERR_BADARG, "device index %d outside [0, %d)", device, MAX_DEVICES);
    static thread_local Buf scratch[MAX_DEVICES][3];  // scratch is device memory: one set per device
    Buf &da = scratch[device][0], &db = scratch[device][1], &dout = scratch[device][2];
    size_t bytes = (size_t)n * dim * dtype_size(dtype);
    const void *pa = a, *pb = b;
    if (mem == VM_MEM_HOST) {
        if ((rc = da.ensure(bytes ? bytes : 8)) != VM_OK || (rc = db.ensure(bytes ? bytes : 8)) != VM_OK) return rc;
        VM_CUDA_CHECK(cudaMemcpyAsync(da.p, a, bytes, cudaMemcpyHostToDevice, st));
        VM_CUDA_CHECK(cudaMemcpyAsync(db.p, b, bytes, cudaMemcpyHostToDevice, st));
        pa = da.p; pb = db.p;
    }
    double *po = out;
    if (out_mem == VM_MEM_HOST) {
        if ((rc = dout.ensure((size_t)n * 8)) != VM_OK) return rc;
        po = (double *)dout.p;
    }
    rc = k_cosine_pairs(pa, pb, dtype, n, dim, zero_rule, sum_mode, po, st);
    if (rc != VM_OK) return rc;
    if (out_mem == VM_MEM_HOST) {
        VM_CUDA_CHECK(cudaMemcpyAsync(out, po, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        VM_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    return VM_OK;
}

// ---- all-pairs --------------------------------------------------------------------------------
extern "C" int vm_pairs_above(int device, const void *x_dev, int dtype, int64_t n, int dim, float threshold, int64_t cap,
                              int64_t *out_i_dev, int64_t *out_j_dev, float *out_score_dev, int64_t *out_count_dev, int part,
                              int nparts, int flags, void *stream)
{
    VM_REQUIRE(x_dev && out_count_dev, VM_ERR_BADARG, "NULL buffer");
    VM_REQUIRE(cap == 0 || (out_i_dev && out_j_dev && out_score_dev), VM_ERR_BADARG, "NULL output with cap > 0");
    VM_REQUIRE(dtype == VM_F32 || dtype == VM_BF16, VM_ERR_BADARG, "dtype must be VM_F32 or VM_BF16");
    VM_REQUIRE(n >= 0 && n < (1LL << 31), VM_ERR_BADARG, "n outside [0, 2^31)");
    VM_REQUIRE(dim >= 1 && dim <= 4096, VM_ERR_BADARG, "dim outside [1, 4096]");
    VM_REQUIRE(nparts >= 1 && part >= 0 && part < nparts, VM_ERR_BADARG, "bad part/nparts");
    int rc = check_arch(device, nullptr);
    if (rc != VM_OK) return rc;
    DeviceGuard g(device);
    return k_pairs_above(device, x_dev, dtype, n, dim, ld_for_dim(dim), threshold, cap, out_i_dev, out_j_dev, out_score_dev,
                         out_count_dev, part, nparts, flags, (cudaStream_t)stream);
}

extern "C" int vm_pairs_above_sharded(vm_comm *comm, void *x_dev, int dtype, int64_t n, int dim, float threshold, int64_t cap,
                                      int64_t *out_i_dev, int64_t *out_j_dev, float *out_score_dev, int64_t *out_count_dev,
                                      int root, int flags, void *stream)
{
    VM_REQUIRE(comm, VM_ERR_BADARG, "comm is NULL");
    VM_REQUIRE(x_dev && out_count_dev, VM_ERR_BADARG, "NULL buffer");
    VM_REQUIRE(cap >= 1 && out_i_dev && out_j_dev && out_score_dev, VM_ERR_BADARG, "cap < 1 or NULL output");
    VM_REQUIRE(dtype == VM_F32 || dtype == VM_BF16, VM_ERR_BADARG, "dtype must be VM_F32 or VM_BF16");
    VM_REQUIRE(n >= 0 && n < (1LL << 31), VM_ERR_BADARG, "n outside [0, 2^31)");
    VM_REQUIRE(dim >= 1 && dim <= 4096, VM_ERR_BADARG, "dim outside [1, 4096]");
    VM_REQUIRE(root >= -1 && root < comm->nranks, VM_ERR_BADARG, "root %d outside [-1, %d)", root, comm->nranks);
    int rc = check_arch(comm->device, nullptr);
    if (rc != VM_OK) return rc;
    DeviceGuard g(comm->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int G = comm->nranks, ld = ld_for_dim(dim);
    // 1. replicate the operand: ONE broadcast from `root` over NVLink (root < 0: every rank already holds it)
    if (root >= 0 && G > 1 && n > 0)
        VM_NCCL_CHECK(g_nccl.Broadcast(x_dev, x_dev, (size_t)n * ld * dtype_size(dtype), /*ncclInt8*/ 0, root, comm->nccl, st));
    // 2. this rank's share of the upper-triangular tile grid (dealt cyclically) -> local hit lists
#define ENS(b, bytes) if ((rc = (b).ensure(bytes)) != VM_OK) return rc
    ENS(comm->pl_i, (size_t)cap * 8); ENS(comm->pl_j, (size_t)cap * 8); ENS(comm->pl_s, (size_t)cap * 4);
    ENS(comm->pl_cnt, 8); ENS(comm->pg_cnt, (size_t)G * 8);
    if (!comm->h_counts) VM_CUDA_CHECK(cudaMallocHost((void **)&comm->h_counts, 16 * 8));
    rc = k_pairs_above(comm->device, x_dev, dtype, n, dim, ld, threshold, cap, (int64_t *)comm->pl_i.p, (int64_t *)comm->pl_j.p,
                       (float *)comm->pl_s.p, (int64_t *)comm->pl_cnt.p, comm->rank, G, 0, st);
    if (rc != VM_OK) return rc;
    // 3. exchange: all-gather of the counts, then ONE all-gather of the lists padded to `slot` entries per rank.
    //    Default: the counts are read back (8 bytes per rank) so the slot is the largest count -- no padding
    //    traffic.  VM_FLAG_ASYNC: no host round trip at all, the slot is the full capacity.
    VM_NCCL_CHECK(g_nccl.AllGather(comm->pl_cnt.p, comm->pg_cnt.p, 8, /*ncclInt8*/ 0, comm->nccl, st));
    int64_t slot = cap;
    if (!(flags & VM_FLAG_ASYNC)) {
        VM_CUDA_CHECK(cudaMemcpyAsync(comm->h_counts, comm->pg_cnt.p, (size_t)G * 8, cudaMemcpyDeviceToHost, st));
        VM_CUDA_CHECK(cudaStreamSynchronize(st));
        int64_t mx = 0, total = 0;
        for (int r = 0; r < G; ++r) { mx = comm->h_counts[r] > mx ? comm->h_counts[r] : mx; total += comm->h_counts[r]; }
        if (mx > cap || total > cap) {
            VM_CUDA_CHECK(cudaMemcpyAsync(out_count_dev, &total, 8, cudaMemcpyHostToDevice, st));
            VM_CUDA_CHECK(cudaStreamSynchronize(st));
            set_error("%lld pairs above the threshold exceed cap=%lld", (long long)total, (long long)cap);
            return VM_ERR_OVERFLOW;
        }
        slot = mx;
    }
    if (slot == 0) { VM_CUDA_CHECK(cudaMemsetAsync(out_count_dev, 0, 8, st)); return VM_OK; }
    // [i slot*8 | j slot*8 | s slot*4], padded to a multiple of 8 bytes: with an odd slot the next rank's int64 arrays
    // would start on a 4-byte boundary (found when a new tile-to-rank dealing made the largest per-rank count odd)
    const size_t per_rank = ((size_t)slot * 20 + 7) & ~(size_t)7;
    ENS(comm->pg_send, per_rank); ENS(comm->pg_recv, per_rank * G);
#undef ENS
    char *sb = (char *)comm->pg_send.p;
    VM_CUDA_CHECK(cudaMemcpyAsync(sb, comm->pl_i.p, (size_t)slot * 8, cudaMemcpyDeviceToDevice, st));
    VM_CUDA_CHECK(cudaMemcpyAsync(sb + (size_t)slot * 8, comm->pl_j.p, (size_t)slot * 8, cudaMemcpyDeviceToDevice, st));
    VM_CUDA_CHECK(cudaMemcpyAsync(sb + (size_t)slot * 16, comm->pl_s.p, (size_t)slot * 4, cudaMemcpyDeviceToDevice, st));
    VM_NCCL_CHECK(g_nccl.AllGather(comm->pg_send.p, comm->pg_recv.p, per_rank, /*ncclInt8*/ 0, comm->nccl, st));
    // 4. concatenate the per-rank lists in rank order on the device (identical on every rank)
    return k_pairs_concat(comm->pg_recv.p, per_rank, slot, (const int64_t *)comm->pg_cnt.p, G, cap, out_i_dev, out_j_dev,
                          out_score_dev, out_count_dev, st);
}

// ---- communicator -----------------------------------------------------------------------------
extern "C" int vm_comm_unique_id(void *out128)
{
    VM_REQUIRE(out128, VM_ERR_BADARG, "out is NULL");
    int rc = nccl_load();
    if (rc != VM_OK) return rc;
    VM_NCCL_CHECK(g_nccl.GetUniqueId(out128));
    return VM_OK;
}

extern "C" int vm_comm_init_rank(vm_comm **out, int device, int nranks, int rank, const void *id128)
{
    VM_REQUIRE(out && id128, VM_ERR_BADARG, "NULL argument");
    VM_REQUIRE(nranks >= 1 && nranks <= 16 && rank >= 0 && rank < nranks, VM_ERR_BADARG, "bad rank %d / nranks %d (at most 16 ranks)", rank, nranks);
    int rc = nccl_load();
    if (rc != VM_OK) return rc;
    DeviceGuard g(device);
    VM_CUDA_CHECK(cudaSetDevice(device));
    vm_comm *c = new (std::nothrow) vm_comm();
    VM_REQUIRE(c, VM_ERR_OOM, "host allocation failed");
    Id128 id;
    memcpy(id.b, id128, 128);
    int r = g_nccl.CommInitRank(&c->nccl, nranks, id, rank);
    if (r != 0) {
        set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
        delete c;
        return VM_ERR_NCCL;
    }
    c->nranks = nranks; c->rank = rank; c->device = device;
    *out = c;
    return VM_OK;
}

extern "C" size_t vm_comm_exchange_bytes(void) { return XCHG_BYTES; }

extern "C" int vm_comm_attach_peer_buffers(vm_comm *c, void *const *bufs, int nranks)
{
    VM_REQUIRE(c && bufs, VM_ERR_BADARG, "NULL argument");
    VM_REQUIRE(nranks == c->nranks && nranks <= 16, VM_ERR_BADARG, "peer buffers for %d ranks, communicator has %d (max 16)", nranks, c->nranks);
    for (int r = 0; r < nranks; ++r) {
        VM_REQUIRE(bufs[r] && ((uintptr_t)bufs[r] & 255) == 0, VM_ERR_BADARG, "peer buffer %d is NULL or not 256-byte aligned", r);
        c->peer[r] = bufs[r];
    }
    c->p2p = true;
    c->gen = 0;
    return VM_OK;
}

extern "C" int vm_comm_destroy(vm_comm *c)
{
    if (!c) return VM_OK;
    if (c->nccl && g_nccl.CommDestroy) g_nccl.CommDestroy(c->nccl);
    {
        DeviceGuard g(c->device);
        Buf *all[] = {&c->pl_i, &c->pl_j, &c->pl_s, &c->pl_cnt, &c->pg_cnt, &c->pg_send, &c->pg_recv};
        for (Buf *b : all) b->release();
        if (c->h_counts) cudaFreeHost(c->h_counts);
    }
    delete c;
    return VM_OK;
}
extern "C" int vm_comm_nranks(const vm_comm *c) { return c ? c->nranks : -1; }
extern "C" int vm_comm_rank(const vm_comm *c) { return c ? c->rank : -1; }

// ---- synthetic data ---------------------------------------------------------------------------
extern "C" int vm_synth_fill(int device, void *rows_dev, int dtype, uint64_t seed, int64_t row0, int64_t n, int dim,
                             uint64_t dup_period, void *stream)
{
    VM_REQUIRE(rows_dev, VM_ERR_BADARG, "rows is NULL");
    VM_REQUIRE(dtype == VM_F32 || dtype == VM_BF16, VM_ERR_BADARG, "dtype must be VM_F32 or VM_BF16");
    DeviceGuard g(device);
    return k_synth_fill(rows_dev, dtype, seed, row0, n, dim, ld_for_dim(dim), dup_period, (cudaStream_t)stream);
}
