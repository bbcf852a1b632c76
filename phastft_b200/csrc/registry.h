// registry.h -- the table of compiled kernels the planner chooses from.
//
// The kernels are instantiated in several translation units so the library builds in parallel
// (__graft_entry__.build()): reg_strided.cu (COL / TRANS passes, compiled once per precision and kind),
// reg_row.cu (whole-transform-in-one-CTA kernels), reg_multi.cu (cluster and pipelined two-pass launches).
// phastft_cuda.cu holds the planner, the launcher and the C ABI and only sees these descriptors.
#pragma once
#include <string>
#include <vector>

#include "fft_kernels.cuh"

namespace phast {

template <typename T>
struct KernelEntry {
    int kind, R, C, NT, first_radix, stages, variant;
    int mode = 0;          // MODE_PLAIN, MODE_TMA_IN / MODE_BULK_IN (asynchronous tile input), MODE_C2R_IN (c2r pre-processing on load)
                           // or MODE_ROW_BULK (one-CTA batch kernel, tile in and out by cp.async.bulk)
    int rads[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // the stage radices (the planner builds the one-CTA kernels' [i][m] stage-twiddle tables from them)
    size_t smem;
    const void* fn;        // fft_pass_kernel<...>; NULL for the passes of a cluster launch (they only exist inside it)
    std::string radices;   // for describe(): the radices plus the mode / variant tags
    std::string rl;        // the radices alone ("16x16"): same tile, same tables
};

// Both passes of a 2-pass plan in ONE launch by a K-CTA thread-block cluster, intermediate exchanged through
// distributed shared memory (fft_cluster2_kernel).
template <typename T>
struct ClusterEntry {
    int log2n, K, NT, minb, variant;
    KernelEntry<T> k1, k2;    // descriptors of the two pass bodies (kind, R, C, first radix) for the planner's tables
    const void* fn;
    size_t smem;
};

// Both passes of a 2-pass plan in one persistent launch, intermediates in an L2-resident ring (fft_pipe2_kernel).
// Matched to a plan by the descriptors of its two pass kernels.
template <typename T>
struct PipeEntry {
    int mode = 0;          // 0: plain pass bodies; 1: asynchronous tile input (TMA boxes of the planar input / bulk rows of the ring)
    int R1, C1, NT1, R2, C2, NT2;
    std::string rad1, rad2;
    const void* fn;
    int NT;
    size_t smem;
};

// Tile width in columns for the strided (HBM-facing) kinds: C * sizeof(T) = 32 B (CH), 64 B (CN) or 128 B (CW).
template <typename T> struct TileC;
template <> struct TileC<double> { static constexpr int CH = 4, CN = 8, CW = 16; };
template <> struct TileC<float> { static constexpr int CH = 8, CN = 16, CW = 32; };

template <class RL> std::string radix_string() {
    std::string r;
    for (int i = 0; i < RL::S; ++i) r += (i ? "x" : "") + std::to_string(RL::rad(i));
    return r;
}

template <typename T, int KIND, int C, int NT, int VARIANT, int MINB, int ID, int... Rs>
KernelEntry<T> make_entry_v() {
    using RL = RadixList<Rs...>;
    using PK = PassKernel<T, RL, C, NT, KIND, 0, VARIANT>;
    static_assert(NT % 32 == 0, "whole warps");
    static_assert(KIND != KIND_COL || NT % C == 0, "a COL thread keeps its column");
    static_assert(PK::SMEM_BYTES <= 227 * 1024, "tile exceeds the 227 KB shared memory of an sm_100 CTA");
    KernelEntry<T> e;
    e.kind = KIND; e.R = RL::R(); e.C = C; e.NT = NT; e.first_radix = RL::rad(0); e.stages = RL::S; e.variant = ID;
    for (int q = 0; q < RL::S && q < 8; ++q) e.rads[q] = RL::rad(q);
    e.smem = PK::SMEM_BYTES;
    e.fn = reinterpret_cast<const void*>(&fft_pass_kernel<T, RL, C, NT, KIND, VARIANT, MINB>);
    e.radices = e.rl = radix_string<RL>();
    if (ID) e.radices += ",v" + std::to_string(ID);
    return e;
}
// pass kernels with an asynchronous tile input (cp.async.bulk.tensor / cp.async.bulk + mbarrier)
template <typename T, int KIND, int C, int NT, int MODE, int VARIANT, int MINB, int ID, int... Rs>
KernelEntry<T> make_entry_async() {
    using RL = RadixList<Rs...>;
    using PK = PassKernel<T, RL, C, NT, KIND, MODE, VARIANT>;
    static_assert(NT % 32 == 0, "whole warps");
    static_assert(KIND != KIND_COL || NT % C == 0, "a COL thread keeps its column");
    static_assert(PK::SMEM_BYTES <= 227 * 1024, "tile exceeds the 227 KB shared memory of an sm_100 CTA");
    KernelEntry<T> e;
    e.kind = KIND; e.R = RL::R(); e.C = C; e.NT = NT; e.first_radix = RL::rad(0); e.stages = RL::S; e.variant = ID; e.mode = MODE;
    e.smem = PK::SMEM_BYTES;
    e.fn = reinterpret_cast<const void*>(&fft_pass_async_kernel<T, RL, C, NT, KIND, MODE, VARIANT, MINB>);
    e.rl = radix_string<RL>();
    e.radices = e.rl + (MODE == MODE_TMA_IN ? ",tma" : MODE == MODE_BULK_IN ? ",bulk" : MODE == MODE_C2R_IN ? ",c2r" :
                        MODE == MODE_R2C_OUT ? ",r2c" : ",bulk-io");
    for (int q = 0; q < RL::S && q < 8; ++q) e.rads[q] = RL::rad(q);
    if (ID) e.radices += ",v" + std::to_string(ID);
    return e;
}

// a default entry plus, for first-pass (COL) tiles, the same kernel with the c2r pre-processing folded into its loads
template <typename T, int KIND, int C, int NT, int VARIANT, int MINB, int ID, int... Rs>
void push_entry(std::vector<KernelEntry<T>>& v) {
    v.push_back(make_entry_v<T, KIND, C, NT, VARIANT, MINB, ID, Rs...>());
    if constexpr (KIND == KIND_COL) v.push_back(make_entry_async<T, KIND, C, NT, MODE_C2R_IN, VARIANT, MINB, ID, Rs...>());
}

// a one-CTA kernel plus the builds of the same tile for batched real transforms: c2r pre-processing on load (every tile) and
// r2c untangle on store (tiles with a shared-memory stage to untangle from, S >= 2).  MINB_C2R / MINB_R2C: their
// minimum-blocks bounds, the plain build's resident CTAs per SM so that they keep its occupancy (0 where that would spill)
template <typename T, int C, int NT, int VARIANT, int MINB, int ID, int MINB_C2R, int MINB_R2C, int... Rs>
void push_row(std::vector<KernelEntry<T>>& v) {
    static_assert((MINB_C2R == 0 || MINB_C2R >= MINB) && (MINB_R2C == 0 || MINB_R2C >= MINB), "a real build keeps the plain build's bound");
    v.push_back(make_entry_v<T, KIND_ROW, C, NT, VARIANT, MINB, ID, Rs...>());
    v.push_back(make_entry_async<T, KIND_ROW, C, NT, MODE_C2R_IN, VARIANT, MINB_C2R ? MINB_C2R : MINB, ID, Rs...>());
    if constexpr (sizeof...(Rs) >= 2)
        v.push_back(make_entry_async<T, KIND_ROW, C, NT, MODE_R2C_OUT, VARIANT, MINB_R2C ? MINB_R2C : MINB, ID, Rs...>());
}

template <typename T, int KIND, int C, int NT, int... Rs>
KernelEntry<T> make_entry() { return make_entry_v<T, KIND, C, NT, 0, 0, 0, Rs...>(); }

// defined in the reg_*.cu translation units
template <typename T> void add_row_kernels(std::vector<KernelEntry<T>>& v);
template <typename T, int KIND> void add_strided_kernels(std::vector<KernelEntry<T>>& v);
template <typename T> const std::vector<PipeEntry<T>>& pipe_registry();
template <typename T> const std::vector<ClusterEntry<T>>& cluster_registry();

}  // namespace phast
