// reg_row.cu -- instantiates the whole-transform-in-one-CTA kernels (KIND_ROW).  Compiled per precision: -DPHAST_T=double|float.
// push_row adds, beside each kernel, its builds for batched real transforms (MODE_C2R_IN, MODE_R2C_OUT; registry.h).  Its two
// arguments after the id are the minimum-blocks bounds of those builds (f64 : f32): the plain build's resident CTAs per SM on
// sm_100 (from its `-Xptxas -v` register count, shared memory and block size), so the extra registers of the real build cannot
// cost occupancy -- or 0 (no bound) where ptxas would spill under that bound; DESIGN.md section 3 lists what those builds get.
#include "registry.h"

#ifndef PHAST_T
#error "compile with -DPHAST_T=double|float"
#endif

namespace phast {

template <>
void add_row_kernels<PHAST_T>(std::vector<KernelEntry<PHAST_T>>& v) {
    using T = PHAST_T;
    constexpr bool F64 = sizeof(T) == 8;
    push_row<T, 64, 64, 0, 0, 0, 32, 32, 2>(v);
    push_row<T, 64, 64, 0, 0, 0, F64 ? 0 : 32, 32, 4>(v);
    push_row<T, 64, 64, 0, 0, 0, 0, F64 ? 21 : 32, 8>(v);
    push_row<T, 32, 32, 0, 0, 0, F64 ? 0 : 32, F64 ? 25 : 32, 16>(v);
    push_row<T, 16, 64, 0, 0, 0, 0, F64 ? 0 : 25, 4, 8>(v);
    push_row<T, 8, 64, 0, 0, 0, F64 ? 18 : 0, F64 ? 18 : 25, 8, 8>(v);
    push_row<T, 4, 64, 0, 0, 0, 0, F64 ? 12 : 21, 16, 8>(v);
    push_row<T, 2, 64, 0, 0, 0, F64 ? 18 : 0, F64 ? 18 : 25, 4, 8, 8>(v);
    push_row<T, 1, 64, 0, 0, 0, F64 ? 16 : 0, F64 ? 16 : 25, 8, 8, 8>(v);
    push_row<T, 1, 128, 0, 0, 0, 0, F64 ? 0 : 10, 16, 8, 8>(v);
    push_row<T, 1, 256, 0, 0, 0, F64 ? 4 : 6, F64 ? 4 : 6, 4, 8, 8, 8>(v);
    push_row<T, 1, 256, 0, 0, 0, F64 ? 2 : 5, F64 ? 2 : 5, 8, 8, 8, 8>(v);
    if constexpr (sizeof(T) == 4) push_row<T, 1, 512, 0, 0, 0, 2, 2, 16, 8, 8, 8>(v);
    push_row<T, 1, 256, 0, 0, 70, F64 ? 2 : 3, F64 ? 2 : 3, 16, 16, 16>(v);
    push_row<T, 1, 128, 0, 0, 70, F64 ? 4 : 7, F64 ? 4 : 7, 8, 16, 16>(v);
    push_row<T, 1, 64, 0, 0, 70, F64 ? 9 : 14, F64 ? 9 : 14, 4, 16, 16>(v);
    push_row<T, 2, 32, 0, 0, 70, F64 ? 0 : 28, F64 ? 23 : 28, 16, 16>(v);
    // ids 80/81: one-CTA kernels for BATCHES of small transforms (2^24 points per call): 4..16 points split in two
    // stages so the lanes of a warp run along the row (coalesced) instead of one row per lane -- n=16 f64 259 -> 121 us;
    // 512 / 1024 points with ONE shared-memory exchange (32x16, 32x32) -- f32 n=1024 86 -> 52 us; 2048 points as 16x16x8.
    push_row<T, 64, 128, 0, 0, 80, 16, 16, 2, 2>(v);
    push_row<T, 64, 128, 0, 0, 80, F64 ? 0 : 16, 16, 2, 4>(v);
    push_row<T, 32, 128, 0, 0, 80, F64 ? 0 : 16, 16, 4, 4>(v);
    push_row<T, 16, 64, 0, 0, 81, F64 ? 0 : 32, 32, 4, 4>(v);
    push_row<T, 2, 32, 0, 0, 81, F64 ? 12 : 16, F64 ? 12 : 16, 32, 16>(v);
    push_row<T, 2, 64, 0, 0, 81, F64 ? 6 : 8, F64 ? 6 : 8, 32, 32>(v);
    push_row<T, 1, 128, 0, 0, 81, F64 ? 5 : 0, F64 ? 5 : 0, 16, 16, 8>(v);
    // MODE_ROW_BULK builds of the batch kernels (tile in and out by cp.async.bulk, for batches that lie back to back in planar
    // arrays; opt-in, PHASTFT_ROW_BULK=1 -- bit-identical, measured equal or slower, profiles/r02_exp_row_bulk.txt): same radices / C / id as the kernel pick_row_batch_kernel chooses for that size, NT = stage-1 tasks per CTA where
    // the plain kernel makes two trips (the landing zone is read in a single trip)
    {
        constexpr int M6 = MODE_ROW_BULK;
        v.push_back(make_entry_async<T, KIND_ROW, 64, 128, M6, 0, 0, 80, 2, 2>());
        v.push_back(make_entry_async<T, KIND_ROW, 64, 256, M6, 0, 0, 80, 2, 4>());
        if constexpr (F64) v.push_back(make_entry_async<T, KIND_ROW, 32, 128, M6, 0, 0, 80, 4, 4>());
        else v.push_back(make_entry_async<T, KIND_ROW, 16, 64, M6, 0, 0, 81, 4, 4>());
        v.push_back(make_entry_async<T, KIND_ROW, 16, 128, M6, 0, 0, 0, 4, 8>());
        v.push_back(make_entry_async<T, KIND_ROW, 8, 64, M6, 0, 0, 0, 8, 8>());
        v.push_back(make_entry_async<T, KIND_ROW, 4, 64, M6, 0, 0, 0, 16, 8>());
        v.push_back(make_entry_async<T, KIND_ROW, 2, 32, M6, 0, 0, 70, 16, 16>());
        if constexpr (F64) v.push_back(make_entry_async<T, KIND_ROW, 1, 64, M6, 0, 0, 0, 8, 8, 8>());
        else v.push_back(make_entry_async<T, KIND_ROW, 2, 32, M6, 0, 0, 81, 32, 16>());
        v.push_back(make_entry_async<T, KIND_ROW, 1, 128, M6, 0, 0, 0, 16, 8, 8>());
        if constexpr (F64) v.push_back(make_entry_async<T, KIND_ROW, 1, 128, M6, 0, 0, 81, 16, 16, 8>());
        else v.push_back(make_entry_async<T, KIND_ROW, 1, 256, M6, 0, 0, 70, 8, 16, 16>());
        v.push_back(make_entry_async<T, KIND_ROW, 1, 256, M6, 0, 0, 70, 16, 16, 16>());
    }
    // (ids 82 / 83 -- the 16..128-point kernels with 2x / 4x the transforms per CTA -- measured equal within 2 %, profiles/r02_exp_tiny.txt,
    // and are not compiled: those sizes are bound by the load / store INSTRUCTION rate, 128 bytes per f32 warp access, not by CTA count)
    // id 90: the largest transforms ONE CTA can hold (128 KB tile): 2^13 f64, 2^14 f32 -- for batches one HBM round trip
    // instead of two passes (the north star's "<= 2^14 points entirely in one block")
    if constexpr (sizeof(T) == 8) {
        push_row<T, 1, 512, 0, 1, 90, 1, 1, 16, 8, 8, 8>(v);     // 8192 points
        push_row<T, 1, 256, 0, 1, 91, 1, 1, 32, 16, 16>(v);
    } else {
        push_row<T, 1, 1024, 0, 1, 90, 1, 1, 16, 16, 8, 8>(v);   // 16384 points
        push_row<T, 1, 512, 0, 1, 91, 1, 1, 32, 16, 32>(v);
        push_row<T, 1, 512, 0, 1, 91, 1, 1, 16, 16, 32>(v);      // 8192 points, two exchanges
    }
}

}  // namespace phast
