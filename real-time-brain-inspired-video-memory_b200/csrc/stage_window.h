// stage_window.h -- shared-memory layout of the rescoring kernels (select.cu): the staged-row window of stage_and_chain,
// the band capacity of select_rescore_kernel and the window of collect_rescore_kernel.  Kept in a header of plain integer
// arithmetic so that the SAME code is compiled for the host by tests/test_stage_window_cpu.py, which checks over every
// shape the API accepts that the layout fits, that the chunks tile each row and that the three slots never overlap.
#pragma once
#include <stddef.h>
#ifdef __CUDACC__
#define VM_STAGE_FN __host__ __device__ __forceinline__
#else
#define VM_STAGE_FN inline
#endif

namespace vm {

static constexpr int SELECT_KEY_CAP = 4096;      // band keys the rescoring kernel stages per query after the final filter
static constexpr int SCAN_DUMP_TILE = 128;       // rows (= keys per query) per dumped tile
static constexpr int SCAN_DUMP_MAX_KEYS = 9472;  // per query: what the fused select kernel ranks in shared memory (148 x 64)
static constexpr int COLLECT_CAP = 4096;         // rows per query the collect pass may gather

static constexpr int SR_THREADS = 512;
static constexpr size_t SR_SMEM_LIMIT = 180 * 1024;  // dynamic shared memory of select_rescore_kernel
static constexpr size_t CR_SMEM_LIMIT = 200 * 1024;  // dynamic shared memory of collect_rescore_kernel
static constexpr int CR_ROWS = 32;                   // rows collect_rescore_kernel stages at a time

// Rows of one query's near-tie band the rescoring kernel settles itself: as many as shared memory leaves room for
// (12 bytes each), between BAND_CAP_MIN and BAND_CAP_MAX.  Settling 2048 rows costs ~0.3 ms for the batch (64 staged
// sub-batches per query, the queries in parallel) and no extra pass over the store; larger bands of up to COLLECT_CAP
// rows are left to the collect pass (a second streaming scan + its own rescoring), anything larger to the binary64 scan.
static constexpr int BAND_CAP_MIN = 1024, BAND_CAP_MAX = 2048;

// Chunk c of a row of gpr 16-byte groups cut into `chunks` chunks spans the groups [stage_chunk_lo(c), stage_chunk_lo(c+1)).
VM_STAGE_FN int stage_chunk_lo(int c, int gpr, int chunks) { return c * gpr / chunks; }
// Chunk c is staged into slot c % 3 of a window of `win` groups per staged row; the slot starts at this group.
VM_STAGE_FN int stage_slot_lo(int c, int win) { return (c % 3) * win / 3; }

// The staged-row window of stage_and_chain for `rows` rows of `ld` elements of `elem_bytes` bytes in `room` bytes of
// shared memory: whole rows in three chunks when they fit (one 16-byte group of padding per row), else the fewest chunks
// whose three slots fit.  The windowed pitch is an odd number of 16-byte groups, as whole fp32 / binary64 rows are, so
// that the chains, each walking its own row at the same column, spread over the shared-memory banks.  chunks == 0: not
// even one group per slot fits.
struct StageWindow { int pitch, chunks; };
VM_STAGE_FN StageWindow stage_window(int rows, int elem_bytes, int ld, size_t room)
{
    const int gpr = ld * elem_bytes / 16;                    // 16-byte groups per row
    if ((size_t)rows * (gpr + 1) * 16 <= room) return {(gpr + 1) * 16, 3};
    for (int chunks = 4; chunks <= gpr; ++chunks) {
        const int s = (gpr + chunks - 1) / chunks;           // groups of the widest chunk
        const int win = 3 * s + (s & 1);                     // three slots of >= s groups, win + 1 odd
        if ((size_t)rows * (win + 1) * 16 <= room) return {(win + 1) * 16, chunks};
    }
    return {0, 0};
}

// Shared memory of select_rescore_kernel: keys, list maxima, query and the staged-row window, sized to leave room for at
// least BAND_CAP_MIN band rows; then as many band rows (12 bytes each) as fit, up to BAND_CAP_MAX.  band_cap == 0: the
// shape does not fit.
struct SelectLayout { StageWindow win; int band_cap; size_t smem; };
VM_STAGE_FN SelectLayout select_layout(int key_cap, int lists, int kp, int elem_bytes, int dim, int ld)
{
    const size_t fixed = (size_t)key_cap * 8 + (size_t)((lists + 3) & ~3) * 4 + (size_t)((dim + 1) & ~1) * 8 + 16 + 32;
    const size_t need = fixed + (size_t)BAND_CAP_MIN * 12;
    SelectLayout L{{0, 0}, 0, 0};
    if (need > SR_SMEM_LIMIT) return L;
    L.win = stage_window(kp, elem_bytes, ld, SR_SMEM_LIMIT - need);
    if (L.win.chunks == 0) return L;
    const size_t base = fixed + (size_t)kp * L.win.pitch;
    const size_t cap = ((SR_SMEM_LIMIT - base) / 12) & ~(size_t)63;
    L.band_cap = (int)(cap < (size_t)BAND_CAP_MAX ? cap : (size_t)BAND_CAP_MAX);
    L.smem = base + (size_t)L.band_cap * 12;
    return L;
}
// key_cap keys per query: SELECT_KEY_CAP in slab mode (lists == 0), lists x list length in list mode
VM_STAGE_FN bool select_layout_fits(int key_cap, int lists, int kp, int elem_bytes, int dim, int ld)
{
    return select_layout(key_cap, lists, kp, elem_bytes, dim, ld).band_cap >= BAND_CAP_MIN && kp <= 64 && 2 * kp + 1 <= SR_THREADS;
}

// Shared memory of collect_rescore_kernel: query, scores and row ids of the `cap` gathered rows, then the staged-row
// window of CR_ROWS rows.  win.chunks == 0: the shape does not fit.
struct CollectLayout { StageWindow win; size_t smem; };
VM_STAGE_FN CollectLayout collect_layout(int cap, int elem_bytes, int dim, int ld)
{
    const size_t fixed = (size_t)((dim + 1) & ~1) * 8 + (size_t)cap * 8 + (size_t)((cap + 3) & ~3) * 4 + 64;
    const StageWindow win = fixed < CR_SMEM_LIMIT ? stage_window(CR_ROWS, elem_bytes, ld, CR_SMEM_LIMIT - fixed) : StageWindow{0, 0};
    return {win, fixed + (size_t)CR_ROWS * win.pitch};
}

}  // namespace vm
