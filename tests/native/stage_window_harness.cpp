// Host build of csrc/stage_window.h for tests/test_stage_window_cpu.py and tests/test_rescore_window_gpu.py: the
// shared-memory layout of the rescoring kernels for a range of dims, and a walk over the chunks and slots of a
// staged-row window with the same index formulas stage_and_chain uses.
#include "stage_window.h"

// Layout of select_rescore_kernel for kp candidate rows of elem_bytes-byte elements, for every dim in [dim_lo, dim_hi).
// lists == 0: slab mode (SELECT_KEY_CAP keys); else list mode, lists x list_len keys.
// out[dim - dim_lo] = {fits, gpr, pitch, chunks, band_cap, smem}.
extern "C" void select_stage(int elem_bytes, int kp, int lists, int list_len, int dim_lo, int dim_hi, long long *out)
{
    const int key_cap = lists > 0 ? lists * list_len : vm::SELECT_KEY_CAP;
    for (int dim = dim_lo; dim < dim_hi; ++dim, out += 6) {
        const int ld = (dim + 7) & ~7;
        const vm::SelectLayout L = vm::select_layout(key_cap, lists, kp, elem_bytes, dim, ld);
        out[0] = vm::select_layout_fits(key_cap, lists, kp, elem_bytes, dim, ld) ? 1 : 0;
        out[1] = ld * elem_bytes / 16;
        out[2] = L.win.pitch;
        out[3] = L.win.chunks;
        out[4] = L.band_cap;
        out[5] = (long long)L.smem;
    }
}

// Layout of collect_rescore_kernel (CR_ROWS rows at a time, COLLECT_CAP gathered rows) for every dim in [dim_lo, dim_hi).
// out[dim - dim_lo] = {rows, gpr, pitch, chunks, smem}.
extern "C" void collect_stage(int elem_bytes, int dim_lo, int dim_hi, long long *out)
{
    for (int dim = dim_lo; dim < dim_hi; ++dim, out += 5) {
        const int ld = (dim + 7) & ~7;
        const vm::CollectLayout L = vm::collect_layout(vm::COLLECT_CAP, elem_bytes, dim, ld);
        out[0] = vm::CR_ROWS;
        out[1] = ld * elem_bytes / 16;
        out[2] = L.win.pitch;
        out[3] = L.win.chunks;
        out[4] = (long long)L.smem;
    }
}

// The constants the layouts are built from: {SELECT_KEY_CAP, SCAN_DUMP_TILE, SCAN_DUMP_MAX_KEYS, COLLECT_CAP,
// SR_SMEM_LIMIT, CR_SMEM_LIMIT, BAND_CAP_MIN, BAND_CAP_MAX, CR_ROWS}.
extern "C" void stage_constants(long long *out)
{
    const long long v[] = {vm::SELECT_KEY_CAP, vm::SCAN_DUMP_TILE, vm::SCAN_DUMP_MAX_KEYS, vm::COLLECT_CAP, (long long)vm::SR_SMEM_LIMIT,
                           (long long)vm::CR_SMEM_LIMIT, vm::BAND_CAP_MIN, vm::BAND_CAP_MAX, vm::CR_ROWS};
    for (int i = 0; i < (int)(sizeof(v) / sizeof(v[0])); ++i) out[i] = v[i];
}

// Walks the window (pitch, chunks) of a row of gpr 16-byte groups.  Returns 0 when it is sound, else the first rule
// broken: 1 the chunks do not tile [0, gpr) in order; 2 a chunk is wider than its slot; 3 the slots overlap or leave
// the win = pitch / 16 - 1 groups of a staged row; 4 whole rows (chunks == 3, win == gpr) are not staged in their own
// columns.  chunk_lo / slot_lo [chunks + 1] receive the first group of every chunk (+ gpr) and of its slot.
extern "C" int stage_walk(int gpr, int pitch, int chunks, int *chunk_lo, int *slot_lo)
{
    const int win = pitch / 16 - 1;
    auto slot_hi = [&](int b) { return b == 2 ? win : vm::stage_slot_lo(b + 1, win); };
    for (int b = 0; b < 3; ++b) {
        const int lo = vm::stage_slot_lo(b, win), hi = slot_hi(b);
        if (lo < 0 || hi > win || lo > hi) return 3;
        if (b > 0 && lo < slot_hi(b - 1)) return 3;
    }
    for (int c = 0; c <= chunks; ++c) {
        chunk_lo[c] = vm::stage_chunk_lo(c, gpr, chunks);
        slot_lo[c] = vm::stage_slot_lo(c, win);
    }
    if (chunk_lo[0] != 0 || chunk_lo[chunks] != gpr) return 1;
    for (int c = 0; c < chunks; ++c) {
        if (chunk_lo[c + 1] < chunk_lo[c]) return 1;
        if (chunk_lo[c + 1] - chunk_lo[c] > slot_hi(c % 3) - slot_lo[c]) return 2;
    }
    if (chunks == 3 && win == gpr)
        for (int c = 0; c < 3; ++c)
            if (slot_lo[c] != chunk_lo[c]) return 4;
    return 0;
}
