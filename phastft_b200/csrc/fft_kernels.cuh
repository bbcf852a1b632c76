// fft_kernels.cuh -- the three sm_100a pass kernels of the B200 FFT.
//
// One launch = one "pass" over the whole signal: every CTA owns an R x C tile (R-point
// sub-transform x C adjacent columns/rows), runs all log2(R) butterfly stages on it with
// the tile held in shared memory between register-resident radix-4/8/16 stages, and
// touches HBM exactly once for the read and once for the write.  A transform of
// N = R_1 * R_2 [* R_3] points is 1, 2 or 3 such launches (DESIGN.md section 3).
//
// What this replaces in the reference (all CPU, one sweep over memory per radix-2 stage):
//   algorithms/dit.rs:33-164   recursive cache-blocked DIT driver      -> the pass decomposition
//   algorithms/bravo.rs:82-251 BRAVO / CO-BRAVO bit-reversal           -> folded into addressing:
//        digit-reversed placement into shared memory on load (stage 1) and the transposed
//        store of the last pass; no separate permutation pass exists on the GPU
//   kernels/dit.rs:971-1115    fft_dit_chunk_n (planner-twiddle stage) -> stage twiddles from the
//        per-pass W_R table, inter-pass twiddles from a two-level W_N table built by the planner
//   algorithms/dit.rs:325-331  inverse 1/N scaling loop                -> fused into the last store
//
// Kernel kinds
//   KIND_COL   first / middle pass: tile rows are strided (stride B), columns contiguous.
//              load [r][c] -> store [k][c], same addresses (layout preserving, in-place safe).
//   KIND_TRANS last pass of a multi-pass plan: tile rows are contiguous sub-sequences, the C rows
//              of a tile are C adjacent values of the slowest input digit; the store is the
//              digit-reversing transpose, written as C-element contiguous runs.
//   KIND_ROW   whole transform in one CTA (N <= 4096 f64 / 8192 f32): rows contiguous in and out.
#pragma once
#ifndef PHAST_EXP_STAGE_TW
#define PHAST_EXP_STAGE_TW 0
#endif
#include <cuda.h>
#include <type_traits>

#include "fft_device.cuh"

namespace phast {

enum { KIND_COL = 0, KIND_TRANS = 1, KIND_ROW = 2 };

template <typename T>
struct PassParams {
    const T* in_re;                // planar input (or interleaved (re,im) pairs if in_interleaved)
    const T* in_im;                // (no __restrict__: in-place passes alias in and out)
    T* out_re;                     // planar output (or interleaved if out_interleaved)
    T* out_im;
    long long in_bstride;          // elements between consecutive transforms of the batch
    long long out_bstride;
    int batch;                     // number of transforms (KIND_ROW: may not be a multiple of C)
    int in_interleaved;            // 1: in_re points at N (re,im) pairs (r2c first pass); 2: pairs, re/im swapped
    int out_interleaved;           // 1: out_re points at N pairs; 2: pairs with re/im swapped (c2r)
    // geometry
    int log2A;                     // A = number of sub-transform groups before this digit
    int log2B;                     // B = stride of this pass's digit = product of later pass sizes
    int log2R1;                    // KIND_TRANS: size of the first pass digit (tile columns run over it)
    int log2Rprev;                 // size of the previous pass digit (0 if no inter-pass twiddle)
    int blk_offset;                // KIND_COL: first linear tile index of this launch (L2-blocked sub-range of `a`)
    int kt_base;                   // KIND_TRANS: first k1 tile of this launch ...
    int log2_ktn;                  // ... and log2 of the number of k1 tiles it covers
    int pdl;                       // launched with programmatic stream serialization
    int has_tw;                    // apply inter-pass twiddle on load
    int tw_shift;                  // exponent scale: e_N = e_L << tw_shift   (N / L)
    Tw2 tw2;                       // two-level W_N table
    const cx<T>* __restrict__ tw_stage;  // W_R^e, e < R           (stage twiddles)
    const cx<T>* __restrict__ tw_stage_im;  // KIND_ROW: per stage s >= 1 the table [i][m] = W_L^(m*i), L = Ns(s)*rad(s), concatenated
                                         // (lanes run along m in a one-CTA kernel: consecutive lanes read consecutive entries)
    const cx<T>* __restrict__ tw_wc;     // KIND_TRANS, 2-pass plans: W_L^(c*m), [c][m] layout
    T scale;                       // multiplied into the stored result (1/N for the inverse)
    // cluster exchange (XCH = 1 producer only): the consuming pass's tile is [CB rows][P2 points]
    int xch_log2P2;                // log2 of the consumer's row length (= its R)
    int xch_log2CB;                // log2 of the consumer's rows per CTA (= its C)
    // ring of workspace slots (fft_pipe2_kernel): transform b's intermediate lives in slot b % ring (ring a power of two; 0 = none)
    int out_ring;                  // KIND_COL: applied to the batch index of the OUTPUT address
    int in_ring;                   // KIND_TRANS: applied to the batch index of the INPUT address
    // c2r pre-processing on load (MODE_C2R_IN only): in_re / in_im are the N/2 + 1 bins of the half-spectrum, the pass's
    // input element k is built from bins k and N/2 - k with the twiddle W_N^k out of this table
    // (MODE_R2C_OUT: the same W_N table, for the untangle of the one-CTA kernel's result)
    Tw2 pre_tw2;
    int pre_log2half;              // log2(N/2); 0 = no pre-processing
    int r2c_out;                   // host only: launch the MODE_R2C_OUT build of the one-CTA kernel
    double2 pre_wc[32];            // W_(2 R1)^i, i < R1 = the kernel's first radix
    // TMA tile input (MODE_TMA_IN only): one tensor map per planar array, dims {B columns, R rows, batch}
    alignas(64) CUtensorMap tmap_re;
    alignas(64) CUtensorMap tmap_im;
};

// Shared-memory tile addressing (units: complex elements).
//   CFAST kernels (COL, TRANS): [pos][c'] with c' = c ^ swz(pos)  (swz == 0 for COL)
//   ROW kernel: [c][pos'] with pos' = pos ^ swz(pos)
// swz(pos) takes the bits of `pos` in which the low bits of the *memory-order* index of stage 1
// land after digit reversal, so that the stage-1 scatter of a coalesced global read is
// bank-conflict free; later stages address whole rows / aligned runs and are unaffected.
template <class RL, int C, int KIND, typename T>
struct TileAddr {
    static constexpr int R = RL::R();
    static constexpr int LOG2R = ilog2_c(R);
    static constexpr int RS_LAST = RL::rad(RL::S - 1);
    static constexpr int SWZ_SHIFT = LOG2R - ilog2_c(RS_LAST);
    // 16-byte (f64) / 8-byte (f32) complex elements: a 128-byte wavefront holds 8 / 16 of them
    static constexpr int LANES_PER_WF = 128 / (2 * (int)sizeof(T));
    static constexpr int SWZ_MASK_WANT = LANES_PER_WF - 1;
    static constexpr int SWZ_MASK_TRANS = (C - 1) < SWZ_MASK_WANT ? (C - 1) : SWZ_MASK_WANT;
    static constexpr int SWZ_MASK_ROW = (R >= 4 * LANES_PER_WF) ? SWZ_MASK_WANT : 0;
    static __device__ __forceinline__ int at(int pos, int c) {
        if constexpr (KIND == KIND_COL) {
            return pos * C + c;
        } else if constexpr (KIND == KIND_TRANS) {
            return pos * C + (c ^ ((pos >> SWZ_SHIFT) & SWZ_MASK_TRANS));
        } else {
            return c * R + (pos ^ ((pos >> SWZ_SHIFT) & SWZ_MASK_ROW));
        }
    }
};

// ---------------------------------------------------------------------------------------------
// r2c / c2r arithmetic, the one copy: called by the elementwise kernels at the end of this file and by the pass kernels that
// fold it into their loads (MODE_C2R_IN) or their last store (MODE_R2C_OUT).  c_h + i s_h = wkr + i wki = 0.5 * W_N^k.
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void half_twiddle(const Tw2& tw2, uint32_t k, T& c_h, T& s_h) {
    const double2 wd = tw2.get(k);
    c_h = T(0.5 * wd.x); s_h = T(0.5 * wd.y);
}
// r2c untangle of bin 0 (r2c.rs:161-166): Z[0] = (a0 + i b0) in, the real bins X[0] and X[N/2] out
template <typename T>
__device__ __forceinline__ void r2c_untangle_ends(T a0, T b0, T& r0, T& rh) {
    r0 = a0 + b0; rh = a0 - b0;
}
// r2c untangle of the self pair k = N/4 (r2c.rs:233-236): Z[N/4] = (a + ib) in, X[N/4] out
template <typename T>
__device__ __forceinline__ void r2c_untangle_self(T a, T b, T wkr, T wki, T& rq, T& iq) {
    rq = a + T(2) * wkr * b;
    iq = T(2) * wki * b;
}
// r2c untangle of the bin pair (k, m = N/2 - k), k != 0, N/4 (r2c.rs:167-232): (a + ib) = Z[k], (c + id) = Z[m] of the
// half-length transform in, X[k] and X[m] out
template <typename T>
__device__ __forceinline__ void r2c_untangle_pair(T a, T b, T c, T d, T wkr, T wki, T& rk, T& ik, T& rm, T& im) {
    T s_re = T(0.5) * (a + c), s_im = T(0.5) * (b - d);
    T t_re = b + d, t_im = c - a;
    T wzr = wkr * t_re - wki * t_im;
    T wzi = wkr * t_im + wki * t_re;
    rk = s_re + wzr; ik = s_im + wzi;
    rm = s_re - wzr; im = wzi - s_im;
}
// c2r pre-processing of element k (r2c.rs:263-347): bins k = (re_f + i im_f) and conj(bin N/2 - k) = (re_s + i im_s) in,
// element k of the half-length inverse transform's input out
template <typename T>
__device__ __forceinline__ cx<T> c2r_element(T re_f, T im_f, T re_s, T im_s, T c_h, T s_h) {
    T zx_re = T(0.5) * (re_f + re_s), zx_im = T(0.5) * (im_f + im_s);
    T dr = re_f - re_s, di = im_f - im_s;
    T zy_re = c_h * dr + s_h * di;
    T zy_im = c_h * di - s_h * dr;
    return make_cx<T>(zx_re - zy_im, zx_im + zy_re);
}

// ---------------------------------------------------------------------------------------------
// The pass kernel.
// ---------------------------------------------------------------------------------------------
// Cluster exchange helpers (thread-block clusters + distributed shared memory, sm_90+):
//   cluster_sync()        barrier.cluster arrive(release) + wait(acquire) by every thread of every CTA of the cluster
//   st_cluster(addr, v)   store into the shared memory of CTA `rank` of the cluster (mapa + st.shared::cluster)
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned cluster_ctarank() {
    unsigned r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ unsigned map_to_rank(unsigned smem_addr, unsigned rank) {
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster(unsigned addr, const double2& v) {
    asm volatile("st.shared::cluster.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void st_cluster(unsigned addr, const float2& v) {
    asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}

// TMA / mbarrier helpers (sm_90+; SASS: UTMALDG for the tensor copy, UBLKCP for the 1-D bulk copy, SYNCS for the mbarrier)
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned mbar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n"
        "DONE_%=:\n\t}" ::"r"(mbar), "r"(parity) : "memory");
}
// 3-D tensor tile (box fixed in the map) global -> shared, completion counted on `mbar`
__device__ __forceinline__ void tma_load_3d(unsigned smem_dst, const CUtensorMap* map, int x, int y, int z, unsigned mbar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_dst), "l"(map), "r"(x), "r"(y), "r"(z), "r"(mbar) : "memory");
}
// contiguous bytes global -> shared (16-byte aligned, size a multiple of 16)
__device__ __forceinline__ void bulk_load_1d(unsigned smem_dst, const void* gsrc, unsigned bytes, unsigned mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_dst), "l"(gsrc), "r"(bytes), "r"(mbar) : "memory");
}

// XCH (how this pass gets its input tile / where its last stage puts its results):
//   0  plain pass: global memory in, global memory out
//   1  producer (KIND_COL): the LAST stage does not store to global memory; every thread keeps its results in
//      registers across a cluster barrier and then scatters them into the shared-memory tiles of the CTAs that own
//      the rows in the next pass, in the layout [row c'][t] that pass's global loads would have read
//   2  consumer (KIND_TRANS): stage 1 reads that tile instead of global memory (all threads first, then a
//      __syncthreads, then the tile is overwritten in the pass's own layout)
//   3  TMA tile input (KIND_COL, first pass, planar input): one thread issues cp.async.bulk.tensor copies of the tile's
//      R x C boxes of the re and im arrays straight into the tile's shared memory (no per-thread address generation, no
//      LSU sector waste on the 32-byte runs of a 4-column f64 tile -- which is what lets a 1024-row tile be 64 KB and three
//      CTAs share an SM); the threads wait on the mbarrier, read their stage-1 inputs out of the landing zone, and go on as usual
//   4  bulk tile input (KIND_TRANS, interleaved intermediates): the tile's C rows are contiguous in the workspace -- C
//      cp.async.bulk copies land them as [c][t], then as mode 2
//   5  c2r pre-processing on load (first pass of the half-length inverse transform inside c2r): the input element k is
//      computed from bins k and N/2 - k of the half-spectrum while it is being loaded (the reference's separate sweep
//      r2c.rs:764-780 and its scratch round trip disappear: one HBM pass less per c2r)
//   6  bulk tile input AND output (KIND_ROW, batches whose transforms lie back to back in planar arrays): the CTA's C transforms
//      are one contiguous run per plane -- two cp.async.bulk copies bring them in (landing zone = the tile, planar [c][r]), the
//      last stage writes its results into a second planar staging area and two cp.async.bulk copies take them out.  The
//      per-lane 4/8-byte accesses of the plain kernel (128 bytes per f32 warp instruction, the bound of the 16..128-point
//      batches) become two asynchronous copies per CTA.
//   7  r2c untangle on store (KIND_ROW, batched r2c): the row is a member's N reals read as N/2 complex pairs; the last stage
//      puts its results back into the tile, and after a barrier each thread takes one bin pair (k, N/2 - k) of one member out
//      of shared memory and stores the untangled bins N/2 + 1 straight to the planar outputs.  The separate untangle sweep
//      and its HBM round trip disappear.
enum { MODE_PLAIN = 0, MODE_XCH_PRODUCE = 1, MODE_XCH_CONSUME = 2, MODE_TMA_IN = 3, MODE_BULK_IN = 4, MODE_C2R_IN = 5, MODE_ROW_BULK = 6,
       MODE_R2C_OUT = 7 };
template <typename T, class RL, int C, int NT, int KIND, int XCH = 0, int VARIANT = 0>
struct PassKernel {
    static constexpr int S = RL::S;
    static constexpr int R = RL::R();
    static constexpr int LOG2R = ilog2_c(R);
    static constexpr int TILE_C = C;               // tile width (columns for COL, rows for TRANS / ROW)
    static constexpr int R1 = RL::rad(0);          // first-stage radix
    static constexpr int M = R / R1;               // stage-1 tasks per column
    static constexpr int LOG2C = ilog2_c(C);
    using Addr = TileAddr<RL, C, KIND, T>;
    // shared memory: tile (only if S >= 2) + Um[M] + G[C][R1]
    static constexpr int TILE_ELEMS = (S >= 2) ? R * C : 0;
    static constexpr int G_ELEMS = (KIND == KIND_TRANS) ? C * R1 : R1;
    static constexpr bool ASYNC_IN = (XCH == MODE_TMA_IN || XCH == MODE_BULK_IN || XCH == MODE_ROW_BULK);
    static constexpr size_t TABLE_END = sizeof(cx<T>) * (size_t)(TILE_ELEMS + M + G_ELEMS);
    static constexpr size_t MBAR_OFF = (TABLE_END + 15) & ~size_t(15);
    static constexpr size_t OUT_OFF = (MBAR_OFF + 16 + 127) & ~size_t(127);      // MODE_ROW_BULK: planar output staging [2][C][R]
    static constexpr size_t SMEM_BYTES = XCH == MODE_ROW_BULK ? OUT_OFF + sizeof(cx<T>) * (size_t)TILE_ELEMS : ASYNC_IN ? MBAR_OFF + 16 : TABLE_END;
    static_assert(XCH == 0 || XCH == MODE_C2R_IN || S >= 2, "an exchanging pass needs a shared-memory tile");
    static_assert(XCH != MODE_R2C_OUT || KIND == KIND_ROW, "r2c untangle on store: one-CTA kernels");
    static_assert(XCH != 1 || KIND == KIND_COL, "the producer of a cluster exchange is a COL pass");
    static_assert(XCH != 2 || KIND == KIND_TRANS, "the consumer of a cluster exchange is a TRANS pass");
    static_assert(XCH != MODE_TMA_IN || (KIND == KIND_COL && C * sizeof(T) >= 16), "TMA tile input: COL pass, rows of >= 16 bytes");
    static_assert(XCH != MODE_BULK_IN || KIND == KIND_TRANS, "bulk tile input: TRANS pass");
    static_assert(XCH != MODE_ROW_BULK || KIND == KIND_ROW, "bulk tile input and output: one-CTA kernels");

    // ---- global element access -------------------------------------------------------------
    static __device__ __forceinline__ void gload(const PassParams<T>& p, long long idx, T& re, T& im) {
        if (p.in_interleaved) {
            cx<T> v = reinterpret_cast<const cx<T>*>(p.in_re)[idx];
            if (p.in_interleaved == 1) { re = v.x; im = v.y; } else { re = v.y; im = v.x; }
        } else {
            re = p.in_re[idx];
            im = p.in_im[idx];
        }
    }
    static __device__ __forceinline__ void gstore(const PassParams<T>& p, long long idx, T re, T im) {
        if (p.scale != T(1)) { re *= p.scale; im *= p.scale; }
        if (p.out_interleaved == 0) {
            p.out_re[idx] = re;
            p.out_im[idx] = im;
        } else if (p.out_interleaved == 1) {
            reinterpret_cast<cx<T>*>(p.out_re)[idx] = make_cx<T>(re, im);
        } else {
            reinterpret_cast<cx<T>*>(p.out_re)[idx] = make_cx<T>(im, re);
        }
    }

    // N strided elements at once.  The layout test is hoisted out of the unrolled loop so each layout gets
    // its own straight-line block behind a uniform branch: with the test inside the loop the compiler
    // predicates both layouts into one stream (every launch then issues the other layout's dead loads and
    // selects, and the selects of the interleaved path split its loads into two dependent batches).
    // Layout class: 0 planar, 1 interleaved (re, im), 2 interleaved swapped (im, re), -1 = test at run time.
    // MODE_C2R_IN: element k of the half-length inverse transform's input, built on the fly from the half-spectrum
    // (same arithmetic, in the same order, as c2r_preprocess_kernel below; r2c.rs:263-347).  The inverse runs as a forward
    // transform of the swapped parts (r2c.rs:782), so the kernel is handed (im, re).
    template <int N>
    static __device__ __forceinline__ void gload_c2r(const PassParams<T>& p, long long mb, long long k0, long long step, cx<T> (&x)[N]) {
        // mb: the member's first bin in in_re / in_im; element i is bin k = k0 + i * step of that member, with
        // step = (N/2) / R1 (first pass: R * B = N/2; one-CTA kernel: M = R / R1), so its twiddle
        // W_N^k = W_N^k0 * W_(2 R1)^i: one table lookup per task, the second factors are launch constants (pre_wc).
        // Loads in groups of 8 (f64): 4 scalars per element, all of a group in flight at once.
        const long long half = 1LL << p.pre_log2half;
        const T* __restrict__ fr = p.in_re + mb + k0;
        const T* __restrict__ fi = p.in_im + mb + k0;
        const T* __restrict__ sr = p.in_re + mb + (half - k0);
        const T* __restrict__ si = p.in_im + mb + (half - k0);
        const double2 wb = p.pre_tw2.get((uint32_t)k0);
        constexpr int G = (sizeof(T) == 8 && N > 8) ? 8 : N;
#pragma unroll
        for (int g0 = 0; g0 < N; g0 += G) {
            T re_f[G], im_f[G], re_s[G], im_s[G];
#pragma unroll
            for (int i = 0; i < G; ++i) {
                const long long off = (long long)(g0 + i) * step;
                re_f[i] = fr[off]; im_f[i] = fi[off];
                re_s[i] = sr[-off]; im_s[i] = -si[-off];
            }
#pragma unroll
            for (int i = 0; i < G; ++i) {
                const double2 wd = (g0 + i == 0) ? wb : cmul_d(wb, p.pre_wc[g0 + i]);
                const T c_h = T(0.5 * wd.x), s_h = T(0.5 * wd.y);
                const cx<T> z = c2r_element<T>(re_f[i], im_f[i], re_s[i], im_s[i], c_h, s_h);
                x[g0 + i] = make_cx<T>(z.y, z.x);
            }
        }
    }
    // mb (MODE_C2R_IN only): offset of the element's batch member, a0 - mb its index inside the member
    template <int N, int IL = -1>
    static __device__ __forceinline__ void gload_n(const PassParams<T>& p, long long a0, long long step, cx<T> (&x)[N],
                                                   [[maybe_unused]] long long mb = 0) {
        if constexpr (XCH == MODE_C2R_IN) {
            gload_c2r<N>(p, mb, a0 - mb, step, x);
        } else if constexpr (IL < 0) {
            if (p.in_interleaved == 0) gload_n<N, 0>(p, a0, step, x);
            else if (p.in_interleaved == 1) gload_n<N, 1>(p, a0, step, x);
            else gload_n<N, 2>(p, a0, step, x);
        } else if constexpr (IL == 0) {
            const T* pr = p.in_re + a0;
            const T* pi = p.in_im + a0;
#pragma unroll
            for (int i = 0; i < N; ++i) x[i] = make_cx<T>(pr[(long long)i * step], pi[(long long)i * step]);
        } else {
            const cx<T>* pc = reinterpret_cast<const cx<T>*>(p.in_re) + a0;
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const cx<T> v = pc[(long long)i * step];
                x[i] = (IL == 1) ? v : make_cx<T>(v.y, v.x);
            }
        }
    }
    template <int N, int OL = -1>
    static __device__ __forceinline__ void gstore_n(const PassParams<T>& p, long long a0, long long step, cx<T> (&x)[N]) {
        if constexpr (OL < 0) {
            if (p.out_interleaved == 0) gstore_n<N, 0>(p, a0, step, x);
            else if (p.out_interleaved == 1) gstore_n<N, 1>(p, a0, step, x);
            else gstore_n<N, 2>(p, a0, step, x);
        } else {
            if (p.scale != T(1)) {
#pragma unroll
                for (int i = 0; i < N; ++i) x[i] = cscale<T>(x[i], p.scale);
            }
            if constexpr (OL == 0) {
                T* pr = p.out_re + a0;
                T* pi = p.out_im + a0;
#pragma unroll
                for (int i = 0; i < N; ++i) { pr[(long long)i * step] = x[i].x; pi[(long long)i * step] = x[i].y; }
            } else {
                cx<T>* pc = reinterpret_cast<cx<T>*>(p.out_re) + a0;
#pragma unroll
                for (int i = 0; i < N; ++i) pc[(long long)i * step] = (OL == 1) ? x[i] : make_cx<T>(x[i].y, x[i].x);
            }
        }
    }

    // OL: output layout class of the LAST stage's stores (see gload_n); the test is made once
    // per stage (run_stages), outside the task loop, so each layout is a straight-line loop.
    template <int s, int OL = -1>
    static __device__ __forceinline__ void stage_from_tile(const PassParams<T>& p, cx<T>* tile, long long out_base,
                                                           long long out_kstride, int tile_rows_valid, int tid) {
        constexpr int RAD = RL::rad(s);
        constexpr int NS = RL::Ns(s);
        constexpr int J = R / RAD;                      // tasks per column
        constexpr int TW_SHIFT = LOG2R - ilog2_c(NS * RAD);
        constexpr bool LAST = (s == S - 1);
        constexpr int NTASK = J * C;
        constexpr int TRIPS = (NTASK + NT - 1) / NT;
#pragma unroll((VARIANT & 1) ? TRIPS : 1)
        for (int t = tid; t < NTASK; t += NT) {
            int c, j;
            if constexpr (KIND == KIND_ROW) { j = t % J; c = t / J; } else { c = t % C; j = t / C; }
            const int m = j & (NS - 1);
            const int g = j / NS;
            const int base = g * NS * RAD + m;
            cx<T> x[RAD];
#pragma unroll
            for (int i = 0; i < RAD; ++i) x[i] = tile[Addr::at(base + i * NS, c)];
            if constexpr ((VARIANT & 2) && RAD == 8) {
                // 3 table loads (W^m, W^2m, W^4m), the other four twiddles by complex products
                cx<T> w1 = __ldg(p.tw_stage + ((m * 1) << TW_SHIFT));
                cx<T> w2 = __ldg(p.tw_stage + ((m * 2) << TW_SHIFT));
                cx<T> w4 = __ldg(p.tw_stage + ((m * 4) << TW_SHIFT));
                cx<T> w3 = ctwid<T>(w1, w2), w5 = ctwid<T>(w1, w4), w6 = ctwid<T>(w2, w4);
                cx<T> w7 = ctwid<T>(w3, w4);
                const cx<T> ws[8] = {w1, w1, w2, w3, w4, w5, w6, w7};
#pragma unroll
                for (int i = 1; i < RAD; ++i) x[i] = ctwid<T>(x[i], ws[i]);
            } else if constexpr (KIND == KIND_ROW) {
                // One-CTA kernels run their lanes along the row, so m differs from lane to lane: W_R^(m*i) out of the plain W_R table is
                // a 32-way gather (15 of them per radix-16 task: measured 40-50 % of these kernels' time, profiles/r02_tuning.md section 7).
                // The per-stage table in [i][m] order makes every one of those loads a contiguous run.
                constexpr int TW_OFF = tw_im_offset<RL>(s);
                const cx<T>* tws = p.tw_stage_im + TW_OFF + m;
                // only the rows i = 1, 2, 4, 8, ... are loaded; W^(m*i) for the other i is the product of two earlier ones
                // (i = hi + lo, hi the top bit: at most popcount(i) - 1 <= 3 products deep for radix 16): 4 loads + 11 products
                // instead of 15 loads per radix-16 task
                cx<T> w[RAD];
#pragma unroll
                for (int i = 1; i < RAD; ++i) {
                    const int hi = 1 << (31 - __builtin_clz((unsigned)i));
                    if (i == hi) w[i] = __ldg(tws + i * NS);
                    else w[i] = ctwid<T>(w[hi], w[i - hi]);
                    x[i] = ctwid<T>(x[i], w[i]);
                }
            } else {
#if PHAST_EXP_STAGE_TW == 1      // experiment: no stage twiddles (wrong results; prices them: profiles/r02_exp_tw_pass.txt)
#elif PHAST_EXP_STAGE_TW == 2    // experiment: the round-1 form, one table load per twiddle
#pragma unroll
                for (int i = 1; i < RAD; ++i) x[i] = ctwid<T>(x[i], __ldg(p.tw_stage + ((m * i) << TW_SHIFT)));
#else
                // Lanes run along c here, so a warp holds 32 / C distinct m: each W_R^(m*i) load is a 2...8-way gather with a
                // stride that grows with i.  Loads for i = 1, 2, 4, ... only, the others by products as above: 2-6 % of the
                // whole transform (2^26 f64 1082 -> 1025 us; without any stage twiddles it would be 993).
                cx<T> w[RAD];
#pragma unroll
                for (int i = 1; i < RAD; ++i) {
                    const int hi = 1 << (31 - __builtin_clz((unsigned)i));
                    if (i == hi) w[i] = __ldg(p.tw_stage + ((m * i) << TW_SHIFT));
                    else w[i] = ctwid<T>(w[hi], w[i - hi]);
                    x[i] = ctwid<T>(x[i], w[i]);
                }
#endif
            }
            DftC<T, RAD>::run(x);
            if constexpr (!LAST || XCH == MODE_R2C_OUT) {
                // (MODE_R2C_OUT: the last stage's outputs kr = m + k*NS go back to their natural positions for the untangle)
#pragma unroll
                for (int k = 0; k < RAD; ++k) tile[Addr::at(base + k * NS, c)] = x[k];
            } else if constexpr (XCH == 1) {
                // last stage of the producing pass of a cluster exchange.  Output row h = m + k*NS of this CTA's column
                // tcol belongs, in the next pass, to CTA h / CB of the cluster, which wants it at [h % CB][tcol] of its tile
                // (the layout its global loads would have read from the workspace).  All tiles of the cluster are still
                // being read by this very stage, so: results stay in registers, cluster barrier, then the scatter.
                // Lanes run along c, so one store instruction writes 32 consecutive elements of one destination row.
                static_assert(TRIPS == 1 && NTASK == NT, "the exchanging stage must be a single trip: one task per thread");
                cluster_sync();
                const unsigned tile_s = (unsigned)__cvta_generic_to_shared(tile);
                const unsigned tcol = (unsigned)out_base + (unsigned)c;     // body() passes the tile's first column in out_base
                const unsigned cb_mask = (1u << p.xch_log2CB) - 1u;
#pragma unroll
                for (int k = 0; k < RAD; ++k) {
                    const unsigned h = (unsigned)(m + k * NS);
                    const unsigned off = ((h & cb_mask) << p.xch_log2P2) + tcol;
                    st_cluster(map_to_rank(tile_s + off * (unsigned)sizeof(cx<T>), h >> p.xch_log2CB), x[k]);
                }
            } else {
                // last stage: g == 0, natural-order outputs kr = m + k*NS
                if (KIND == KIND_ROW && c >= tile_rows_valid) continue;
                if constexpr (XCH == MODE_ROW_BULK) {
                    // natural-order planar staging; the bulk copies at the end of body() take it out
                    T* ore = reinterpret_cast<T*>(reinterpret_cast<unsigned char*>(tile) + OUT_OFF) + c * R + m;
                    T* oim = ore + C * R;
                    const T sc = p.scale;
#pragma unroll
                    for (int k = 0; k < RAD; ++k) { ore[k * NS] = x[k].x * sc; oim[k * NS] = x[k].y * sc; }
                } else
                if constexpr (KIND == KIND_ROW) gstore_n<RAD, OL>(p, out_base + (long long)c * p.out_bstride + m, (long long)NS, x);
                else gstore_n<RAD, OL>(p, out_base + (long long)m * out_kstride + c, (long long)NS * out_kstride, x);
            }
        }
    }

    template <int s>
    static __device__ __forceinline__ void run_stages(const PassParams<T>& p, cx<T>* tile, long long out_base,
                                                      long long out_kstride, int rows_valid, int tid) {
        if constexpr (s < S) {
            __syncthreads();
            if constexpr (s == S - 1) {
                if (p.out_interleaved == 0) stage_from_tile<s, 0>(p, tile, out_base, out_kstride, rows_valid, tid);
                else if (p.out_interleaved == 1) stage_from_tile<s, 1>(p, tile, out_base, out_kstride, rows_valid, tid);
                else stage_from_tile<s, 2>(p, tile, out_base, out_kstride, rows_valid, tid);
            } else {
                stage_from_tile<s>(p, tile, out_base, out_kstride, rows_valid, tid);
            }
            run_stages<s + 1>(p, tile, out_base, out_kstride, rows_valid, tid);
        }
    }

    // ---- the kernel body ------------------------------------------------------------------------
    // `tile_index` is the linear tile id (blockIdx.x for a plain launch; a fused launch loops over tiles).
    // Threads with threadIdx.x >= NT (a fused launch whose other pass needs more threads) take part in
    // the barriers only: their task index starts beyond every task count.
    static __device__ __forceinline__ void body(const PassParams<T>& p, unsigned tile_index) {
        extern __shared__ __align__(128) unsigned char smem_raw[];
        cx<T>* tile = reinterpret_cast<cx<T>*>(smem_raw);
        cx<T>* s_um = tile + TILE_ELEMS;   // [M]       per-CTA  W_L^(kp*B*m')
        cx<T>* s_g = s_um + M;             // [C][R1] or [R1]     W_L^(kp(c)*M*B*i)

        const int tid = (threadIdx.x < NT) ? (int)threadIdx.x : (1 << 28);
        // Programmatic dependent launch (sm_90+): this grid may have been scheduled while the previous
        // pass is still draining; wait for its memory to be visible before touching global data, and
        // let the next pass's CTAs be scheduled as soon as every CTA of this grid is resident.
        // With an asynchronous tile input only the thread that issues the copies waits: the others build the
        // twiddle tables meanwhile and meet the data at the mbarrier (every later access depends on that data).
        if (p.pdl) {
            asm volatile("griddepcontrol.launch_dependents;");
            if constexpr (!ASYNC_IN) asm volatile("griddepcontrol.wait;" ::: "memory");
        }
        long long in_base, out_base, out_kstride;
        long long in_rstride;          // element stride of the tile row index r (COL) / 1 (ROW, TRANS)
        long long in_cstride;          // element stride between tile columns
        int rows_valid = C;
        uint32_t kp0 = 0;              // previous-pass output digit of column c = 0
        uint32_t kp_cstep = 0;         // ... and its increment per column
        uint32_t bcol0 = 0;            // flat index of the remaining digits for column 0 (COL only)
        [[maybe_unused]] long long in_mbase = 0;   // COL, MODE_C2R_IN: first element of the tile's batch member

        if constexpr (KIND == KIND_COL) {
            const int tilesB = 1 << (p.log2B - LOG2C);
            const unsigned blk = tile_index + (unsigned)p.blk_offset;
            const int bt = blk & (tilesB - 1);
            const int rest = blk >> (p.log2B - LOG2C);
            const int a = rest & ((1 << p.log2A) - 1);
            const int batch = rest >> p.log2A;
            const long long off = ((long long)a << (LOG2R + p.log2B)) + ((long long)bt << LOG2C);
            in_mbase = (long long)batch * p.in_bstride;
            in_base = in_mbase + off;
            out_base = (long long)(p.out_ring ? (batch & (p.out_ring - 1)) : batch) * p.out_bstride + off;
            in_rstride = 1LL << p.log2B;
            in_cstride = 1;
            out_kstride = in_rstride;
            kp0 = a & ((1u << p.log2Rprev) - 1u);
            bcol0 = (uint32_t)bt << LOG2C;
            if constexpr (XCH == 1) out_base = (long long)bcol0;   // no global output: the last stage wants the tile's first column
        } else if constexpr (KIND == KIND_TRANS) {
            // rows of the tile: a(c) = (k0 + c) * rest_n + rest, rest_n = A / R1
            const int log2restn = p.log2A - p.log2R1;
            const int tilesK = 1 << p.log2_ktn;
            const int kt = p.kt_base + (tile_index & (tilesK - 1));
            const int tmp = tile_index >> p.log2_ktn;
            const int rest = tmp & ((1 << log2restn) - 1);
            const int batch = tmp >> log2restn;
            const int k0 = kt << LOG2C;
            in_base = (long long)(p.in_ring ? (batch & (p.in_ring - 1)) : batch) * p.in_bstride + ((((long long)k0 << log2restn) + rest) << LOG2R);
            in_rstride = 1;
            in_cstride = 1LL << (log2restn + LOG2R);
            // out[(k0 + c) + R1*rest + A*kr]
            out_base = (long long)batch * p.out_bstride + k0 + ((long long)rest << p.log2R1);
            out_kstride = 1LL << p.log2A;
            const uint32_t rprev_mask = (1u << p.log2Rprev) - 1u;
            kp0 = (uint32_t)(((long long)k0 << log2restn) + rest) & rprev_mask;
            kp_cstep = (log2restn == 0) ? 1u : 0u;   // 2-pass plan: kp = k1 = k0 + c ; 3-pass: kp = k2
        } else {
            const long long first = (long long)tile_index * C;
            rows_valid = (int)min((long long)C, (long long)p.batch - first);
            in_base = first * p.in_bstride;
            out_base = first * p.out_bstride;
            in_rstride = 1;
            in_cstride = p.in_bstride;
            out_kstride = 1;
        }

        // ---- asynchronous tile input: thread 0 puts the whole tile in flight --------------------------------------
        [[maybe_unused]] const unsigned mbar = (unsigned)__cvta_generic_to_shared(smem_raw + MBAR_OFF);
        if constexpr (ASYNC_IN) {
            if (tid == 0) {
                mbar_init(mbar, 1);
                if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
                mbar_expect_tx(mbar, XCH == MODE_ROW_BULK ? (unsigned)(2 * rows_valid * R * sizeof(T)) : (unsigned)(TILE_ELEMS * sizeof(cx<T>)));
                const unsigned tile_s = (unsigned)__cvta_generic_to_shared(tile);
                if constexpr (XCH == MODE_TMA_IN) {
                    // boxes of at most 256 rows.  Planar input: re plane [R][C] then im plane [R][C].  Interleaved input (the
                    // workspace of a 3-pass plan): one map over the pairs, the landing zone is the tile itself, [R][C] complex.
                    constexpr int BOX_ROWS = R < 256 ? R : 256;
                    const int blkq = (int)(tile_index + (unsigned)p.blk_offset);
                    const int col0 = (blkq & ((1 << (p.log2B - LOG2C)) - 1)) << LOG2C;
                    const int bz = blkq >> (p.log2B - LOG2C);          // = a + A * batch: the map's third dimension
                    if (p.in_interleaved) {
#pragma unroll
                        for (int r0 = 0; r0 < R; r0 += BOX_ROWS)
                            tma_load_3d(tile_s + (unsigned)(r0 * C * sizeof(cx<T>)), &p.tmap_re, 2 * col0, r0, bz, mbar);
                    } else {
#pragma unroll
                        for (int r0 = 0; r0 < R; r0 += BOX_ROWS) {
                            tma_load_3d(tile_s + (unsigned)(r0 * C * sizeof(T)), &p.tmap_re, col0, r0, bz, mbar);
                            tma_load_3d(tile_s + (unsigned)((R + r0) * C * sizeof(T)), &p.tmap_im, col0, r0, bz, mbar);
                        }
                    }
                } else if constexpr (XCH == MODE_ROW_BULK) {
                    const unsigned bytes = (unsigned)(rows_valid * R * sizeof(T));
                    bulk_load_1d(tile_s, p.in_re + in_base, bytes, mbar);
                    bulk_load_1d(tile_s + (unsigned)(C * R * sizeof(T)), p.in_im + in_base, bytes, mbar);
                } else {
                    const cx<T>* src = reinterpret_cast<const cx<T>*>(p.in_re) + in_base;
#pragma unroll
                    for (int c = 0; c < C; ++c)
                        bulk_load_1d(tile_s + (unsigned)(c * R * sizeof(cx<T>)), src + (long long)c * in_cstride, (unsigned)(R * sizeof(cx<T>)), mbar);
                }
            }
        }

        // ---- PRELOAD: when every thread owns exactly one stage-1 task, issue its global loads NOW so
        // they are in flight while the twiddle tables below are built (their two-level lookups are two
        // dependent L2 round trips that would otherwise sit in front of the first data load).
        constexpr bool PRELOAD = (M * C <= NT);
        static_assert((XCH != 2 && !ASYNC_IN) || PRELOAD, "a pass that reads its input out of its own tile must do stage 1 in a single trip (every thread holds its task's inputs across the barrier)");
        cx<T> pre[PRELOAD ? R1 : 1];
        if constexpr (PRELOAD) {
            const int t = tid;
            if (t < M * C) {
                int c, mp;
                if constexpr (KIND == KIND_COL) { c = t % C; mp = t / C; } else { mp = t % M; c = t / M; }
                if constexpr (ASYNC_IN) {
                    // filled in below, once the tile has landed
                } else if constexpr (XCH == 2) {
                    // the previous pass's CTAs left this tile as [c][t], t = mp + i*M (what the global loads would have read)
                    const cx<T>* src = tile + c * R + mp;
#pragma unroll
                    for (int i = 0; i < R1; ++i) pre[i] = src[i * M];
                } else if ((KIND != KIND_ROW) || (c < rows_valid)) {
                    const long long a0 = in_base + (long long)c * in_cstride + (long long)mp * in_rstride;
                    const long long mb = (KIND == KIND_ROW) ? in_base + (long long)c * in_cstride : in_mbase;
                    gload_n<R1>(p, a0, (long long)M * in_rstride, pre, mb);
                } else {
#pragma unroll
                    for (int i = 0; i < R1; ++i) pre[i] = make_cx<T>(T(0), T(0));
                }
            }
        }

        // ---- per-CTA inter-pass twiddle factors (two-level lookups, f64, once per CTA) ----------
        // tw(r, c) = W_L^( kp(c) * (r*B + bcol(c)) ),  r = m' + i*M
        //          = W_L^(kp*B*m') * W_L^(kp*bcol) * W_L^(kp*M*B*i)  =  Um[m'] * V[c] * G[c][i]
        cx<T> vreg = make_cx<T>(T(1), T(0));
        const bool has_tw = (KIND != KIND_ROW) && p.has_tw;
        if (has_tw) {
            const int log2B = (KIND == KIND_COL) ? p.log2B : 0;
            for (int mp = tid; mp < M; mp += NT) {
                uint32_t e = (kp0 * (uint32_t)mp) << log2B;
                s_um[mp] = to_cx<T>(p.tw2.get(e << p.tw_shift));
            }
            constexpr int LOG2M = ilog2_c(M);
            for (int q = tid; q < G_ELEMS; q += NT) {
                const int i = q % R1;
                const int c = q / R1;
                uint32_t kp = kp0 + kp_cstep * (uint32_t)c;
                uint32_t e = (kp * (uint32_t)i) << (LOG2M + log2B);
                s_g[q] = to_cx<T>(p.tw2.get(e << p.tw_shift));
            }
            if constexpr (KIND == KIND_COL) {
                const int c = tid % C;   // NT % C == 0: a thread keeps its column for the whole kernel
                uint32_t e = kp0 * (bcol0 + (uint32_t)c);
                vreg = to_cx<T>(p.tw2.get(e << p.tw_shift));
            }
            __syncthreads();
        } else if constexpr (XCH == 2 || ASYNC_IN) {
            __syncthreads();     // every thread has read its inputs out of the exchanged tile before stage 1 overwrites it
        }                        // (asynchronous input: thread 0's mbarrier init is visible to all)
        if constexpr (ASYNC_IN) {
            mbar_wait(mbar, 0);
            const int t = tid;
            if (t < M * C) {
                int c, mp;
                if constexpr (KIND == KIND_COL) { c = t % C; mp = t / C; } else { mp = t % M; c = t / M; }
                if constexpr (XCH == MODE_ROW_BULK) {
                    const T* re_pl = reinterpret_cast<const T*>(tile) + c * R + mp;
                    const T* im_pl = re_pl + C * R;
                    if (c < rows_valid) {
#pragma unroll
                        for (int i = 0; i < R1; ++i) pre[i] = make_cx<T>(re_pl[i * M], im_pl[i * M]);
                    } else {
#pragma unroll
                        for (int i = 0; i < R1; ++i) pre[i] = make_cx<T>(T(0), T(0));
                    }
                } else if constexpr (XCH == MODE_TMA_IN) {
                    if (p.in_interleaved) {
                        const cx<T>* src = tile + mp * C + c;
#pragma unroll
                        for (int i = 0; i < R1; ++i) pre[i] = src[i * M * C];
                    } else {
                        const T* re_pl = reinterpret_cast<const T*>(tile) + mp * C + c;
                        const T* im_pl = re_pl + R * C;
#pragma unroll
                        for (int i = 0; i < R1; ++i) pre[i] = make_cx<T>(re_pl[i * M * C], im_pl[i * M * C]);
                    }
                } else {
                    const cx<T>* src = tile + c * R + mp;
#pragma unroll
                    for (int i = 0; i < R1; ++i) pre[i] = src[i * M];
                }
            }
            __syncthreads();     // the landing zone is free: stage 1 may overwrite it
        }

        // ---- stage 1: global -> registers -> (twiddle, DFT) -> tile (or global when S == 1) ------
        // The input layout is tested once, outside the task loop (see gload_n).
        auto stage1 = [&](auto il_tag) {
            [[maybe_unused]] constexpr int IL = decltype(il_tag)::value;
            constexpr int NTASK = M * C;
            constexpr int TRIPS1 = (NTASK + NT - 1) / NT;
#pragma unroll((VARIANT & 4) ? TRIPS1 : 1)
            for (int t = tid; t < NTASK; t += NT) {
                int c, mp;
                if constexpr (KIND == KIND_COL) { c = t % C; mp = t / C; } else { mp = t % M; c = t / M; }
                cx<T> x[R1];
                [[maybe_unused]] const bool valid = (KIND != KIND_ROW) || (c < rows_valid);
                if constexpr (PRELOAD) {
#pragma unroll
                    for (int i = 0; i < R1; ++i) x[i] = pre[i];
                } else if (valid) {
                    const long long a0 = in_base + (long long)c * in_cstride + (long long)mp * in_rstride;
                    const long long mb = (KIND == KIND_ROW) ? in_base + (long long)c * in_cstride : in_mbase;
                    gload_n<R1, IL>(p, a0, (long long)M * in_rstride, x, mb);
                } else {
#pragma unroll
                    for (int i = 0; i < R1; ++i) x[i] = make_cx<T>(T(0), T(0));
                }
                if (has_tw) {
                    cx<T> pt = s_um[mp];
                    if constexpr (KIND == KIND_COL) {
                        pt = ctwid<T>(pt, vreg);
                    } else {
                        if (kp_cstep) pt = ctwid<T>(pt, __ldg(p.tw_wc + c * M + mp));
                    }
                    const cx<T>* g = (KIND == KIND_TRANS) ? (s_g + c * R1) : s_g;
                    x[0] = ctwid<T>(x[0], pt);
#pragma unroll
                    for (int i = 1; i < R1; ++i) x[i] = ctwid<T>(x[i], ctwid<T>(pt, g[i]));
                }
                DftC<T, R1>::run(x);
                if constexpr (S >= 2) {
                    const int j = rev_tail<RL>(mp);
#pragma unroll
                    for (int k = 0; k < R1; ++k) tile[Addr::at(j * R1 + k, c)] = x[k];
                } else {
                    if (valid) {
                        if constexpr (KIND == KIND_ROW) gstore_n<R1>(p, out_base + (long long)c * p.out_bstride, 1LL, x);
                        else gstore_n<R1>(p, out_base + c, out_kstride, x);
                    }
                }
            }
        };
        if constexpr (PRELOAD || XCH == MODE_C2R_IN) stage1(std::integral_constant<int, 0>{});
        else if (p.in_interleaved == 0) stage1(std::integral_constant<int, 0>{});
        else if (p.in_interleaved == 1) stage1(std::integral_constant<int, 1>{});
        else stage1(std::integral_constant<int, 2>{});
        // ---- stages 2..S -------------------------------------------------------------------------
        run_stages<1>(p, tile, out_base, out_kstride, rows_valid, tid);
        if constexpr (XCH == MODE_R2C_OUT) {
            // Z = the tile's row c (the half-length transform of member c's reals as pairs).  Task (c, k), k < R/2: bins k and
            // R - k; k == 0 also does bins 0, R and the self pair R/2 (as r2c_untangle_kernel).  Consecutive lanes take
            // consecutive k, so the stores of bins k (ascending) and R - k (descending) are both warp-contiguous.
            __syncthreads();
            constexpr int Q = R / 2;
            for (int t = tid; t < C * Q; t += NT) {
                const int c = t / Q, k = t % Q;
                if (c >= rows_valid) break;
                T* ore = p.out_re + out_base + (long long)c * p.out_bstride;
                T* oim = p.out_im + out_base + (long long)c * p.out_bstride;
                if (k == 0) {
                    const cx<T> z0 = tile[Addr::at(0, c)];
                    T r0, rh;
                    r2c_untangle_ends<T>(z0.x, z0.y, r0, rh);
                    ore[0] = r0; oim[0] = T(0);
                    ore[R] = rh; oim[R] = T(0);
                    T wkr, wki;
                    half_twiddle<T>(p.pre_tw2, (uint32_t)Q, wkr, wki);
                    const cx<T> zq = tile[Addr::at(Q, c)];
                    r2c_untangle_self<T>(zq.x, zq.y, wkr, wki, ore[Q], oim[Q]);
                } else {
                    T wkr, wki;
                    half_twiddle<T>(p.pre_tw2, (uint32_t)k, wkr, wki);
                    const cx<T> zk = tile[Addr::at(k, c)], zm = tile[Addr::at(R - k, c)];
                    r2c_untangle_pair<T>(zk.x, zk.y, zm.x, zm.y, wkr, wki, ore[k], oim[k], ore[R - k], oim[R - k]);
                }
            }
        }
        if constexpr (XCH == MODE_ROW_BULK) {
            // the staging area was written through the generic proxy: make it visible to the asynchronous proxy, then one thread
            // copies the two planes out and waits until the copies have READ shared memory before the CTA may exit
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (tid == 0) {
                const unsigned stage_s = (unsigned)__cvta_generic_to_shared(smem_raw + OUT_OFF);
                const unsigned bytes = (unsigned)(rows_valid * R * sizeof(T));
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(p.out_re + out_base), "r"(stage_s), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(p.out_im + out_base), "r"(stage_s + (unsigned)(C * R * sizeof(T))), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            }
        }
    }

};

template <typename T, class RL, int C, int NT, int KIND, int VARIANT = 0, int MINB = 0>
__global__ void __launch_bounds__(NT, MINB) fft_pass_kernel(const __grid_constant__ PassParams<T> p) {
    PassKernel<T, RL, C, NT, KIND, 0, VARIANT>::body(p, blockIdx.x);
}
// the same pass with an asynchronous tile input (MODE_TMA_IN / MODE_BULK_IN) or another MODE_* of its loads / stores
template <typename T, class RL, int C, int NT, int KIND, int MODE, int VARIANT = 0, int MINB = 0>
__global__ void __launch_bounds__(NT, MINB) fft_pass_async_kernel(const __grid_constant__ PassParams<T> p) {
    PassKernel<T, RL, C, NT, KIND, MODE, VARIANT>::body(p, blockIdx.x);
}

// ---------------------------------------------------------------------------------------------
// One HBM pass for transforms that fit the shared memory of a thread-block cluster (2^13..2^17 points): the K CTAs of a
// cluster run pass 1 (PK1, KIND_COL, each CTA P2/K adjacent columns of the P1 x P2 view of the signal) out of global
// memory, exchange the intermediate through distributed shared memory (every CTA scatters its results into the tiles of
// the CTAs that own those rows in pass 2 -- the transpose that a two-launch plan does through a global workspace), and
// run pass 2 (PK2, KIND_TRANS, P1/K rows each) out of shared memory into global memory.  HBM sees the signal once in
// and once out; grid = transforms x K, cluster dimension K (launch attribute).
// Replaces, for these sizes, the L1-resident leaf of the reference's recursion (algorithms/dit.rs:27-93).
// ---------------------------------------------------------------------------------------------
template <class PK1, class PK2, typename T, int NT, int MINB>
__global__ void __launch_bounds__(NT, MINB) fft_cluster2_kernel(const __grid_constant__ PassParams<T> p1,
                                                                const __grid_constant__ PassParams<T> p2) {
    PK1::body(p1, blockIdx.x);      // ends with: cluster barrier, scatter into the cluster's tiles
    cluster_sync();                 // every CTA's scatter has landed; nobody writes another CTA's tile after this
    PK2::body(p2, blockIdx.x);
}

// ---------------------------------------------------------------------------------------------
// Both passes of a two-pass plan in ONE persistent launch with the intermediates in an L2-resident ring.
//
// A two-launch plan writes the whole batch's intermediate to HBM and reads it back: 2x the compulsory traffic, which
// caps it at half the roofline however good each pass is (round 1: 4096 x 2^16 f32 at 0.47 with both passes at
// 0.92-0.96).  Here one grid runs both passes at once, its CTAs drawing pass-1 and pass-2 tiles from one ordered ticket queue.
// Pass 1 of transform b writes slot b % ring of a workspace of `ring` transforms (sized to stay in the 126 MB L2, 24-32 MiB),
// pass 2 of transform b reads it back while it is still in L2, and the slot is rewritten (or discarded) before its dirty
// lines are evicted, so HBM sees the batch once in and once out (tools/dsmem_bench.cu `ring`: 5.4 TB/s of
// compulsory traffic against 3.4 TB/s for the HBM round trip).  Dependencies are per-transform counters:
//     a pass-2 tile of transform b waits for done1[b] == tiles1   (all of its rows have been produced)
//     a pass-1 tile of transform b waits for done2[b - ring] == tiles2   (its slot has been drained)
// released with red.release.gpu after a block barrier and acquired with ld.acquire.gpu by thread 0 before a block barrier.
// With batch == 1 this is a fused two-pass launch of a lone transform (replaces round 1's cooperative-launch + grid-barrier
// experiment).
// ---------------------------------------------------------------------------------------------
struct PipeCtl {
    unsigned* ticket;              // next work item (zeroed before the launch, like done1 / done2)
    unsigned* done1;               // [batch] pass-1 tiles finished per transform
    unsigned* done2;               // [batch] pass-2 tiles finished per transform
    unsigned tiles1, tiles2;       // tiles per transform in pass 1 / pass 2
    unsigned batch, ring, delay;   // ring: workspace slots (transforms), a power of two; pass 2 runs `delay` < ring transforms behind
    int discard;                   // pass 2 tells L2 to drop its input lines once read (discard.global.L2): no write-back of the ring
};
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_gpu(unsigned* p, unsigned v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void wait_count(const unsigned* p, unsigned want) {
    if (threadIdx.x == 0)
        while (ld_acquire_gpu(p) < want) __nanosleep(64);
    __syncthreads();
}

// One CTA = one tile.  The tile is NOT derived from blockIdx: the CTA draws a ticket when it starts running, so tickets are
// held by resident CTAs only and every wait below is for a smaller ticket -- forward progress without assuming anything about
// the order in which the hardware dispatches CTAs (the decoupled-look-back argument).  Ticket order:
//     step s  =  [pass-1 tiles of transform s]  then  [pass-2 tiles of transform s - delay]
// so pass 1 runs `delay` transforms ahead of pass 2 and both kinds of tile are in flight on every SM.  No loop around the
// pass bodies: each keeps (about) the register allocation it has as a kernel of its own.
template <class PK, typename T>
__device__ __forceinline__ void pipe_discard_rows(const PassParams<T>& p, unsigned bq, unsigned kt) {
    // this tile's input rows (C rows of R contiguous interleaved elements each) will not be read again: let L2 drop them
    constexpr int LINES_PER_ROW = (int)(PK::R * sizeof(cx<T>) / 128);
    const char* rows = reinterpret_cast<const char*>(reinterpret_cast<const cx<T>*>(p.in_re) + (long long)bq * p.in_bstride +
                                                     (long long)kt * PK::TILE_C * PK::R);
    for (int q = threadIdx.x; q < PK::TILE_C * LINES_PER_ROW; q += blockDim.x)
        asm volatile("discard.global.L2 [%0], 128;" ::"l"(rows + (size_t)q * 128) : "memory");
}

template <class PK1, class PK2, typename T, int NTF, int MINB>
__global__ void __launch_bounds__(NTF, MINB) fft_pipe2_kernel(const __grid_constant__ PassParams<T> p1,
                                                             const __grid_constant__ PassParams<T> p2,
                                                             const __grid_constant__ PipeCtl c) {
    __shared__ unsigned s_ticket;
    if (threadIdx.x == 0) s_ticket = atomicAdd(c.ticket, 1u);
    __syncthreads();
    const unsigned t = s_ticket;
    const unsigned L = c.tiles1 + c.tiles2;
    const unsigned step = t / L, j = t - step * L;
    if (j < c.tiles1) {
        if (step >= c.batch) return;
        if (step >= c.ring) wait_count(c.done2 + (step - c.ring), c.tiles2);          // the slot has been drained
        PK1::body(p1, step * c.tiles1 + j);
        __syncthreads();
        if (threadIdx.x == 0) red_release_gpu(c.done1 + step, 1u);
    } else {
        if (step < c.delay || step - c.delay >= c.batch) return;
        const unsigned b = step - c.delay, kt = j - c.tiles1;
        wait_count(c.done1 + b, c.tiles1);                                             // all rows of the transform have been produced
        PK2::body(p2, b * c.tiles2 + kt);
        __syncthreads();
        if (c.discard) { pipe_discard_rows<PK2, T>(p2, b & (c.ring - 1), kt); __syncthreads(); }
        if (threadIdx.x == 0) red_release_gpu(c.done2 + b, 1u);
    }
}

// ---------------------------------------------------------------------------------------------
// r2c post-processing (reference: simd_untangle_inplace_*, algorithms/r2c.rs:150-242) and c2r
// pre-processing (simd_c2r_preprocess_*, r2c.rs:263-432).  Elementwise over bin pairs (k, half-k).
// The planner's w[k] = 0.5 * W_N^k table (planner.rs:120-162, an O(N) rotation recurrence on the
// CPU) is replaced by a two-level lookup: consecutive k hit consecutive `lo` entries (coalesced)
// and one broadcast `hi` entry.
// ---------------------------------------------------------------------------------------------
template <typename T>
struct RealParams {
    T* __restrict__ re;         // untangle: in/out (length half+1).  preprocess: z_re out (length half)
    T* __restrict__ im;
    const T* __restrict__ in_re;  // preprocess only: spectrum (length half+1)
    const T* __restrict__ in_im;
    long long bstride;          // elements between batch members in re/im
    long long in_bstride;
    int log2half;
    Tw2 tw2;                    // two-level table for W_N, N = 2*half
};

// Bin pair k of one member (k <= N/4; k == 0 also does bin N/2), in place on its half+1 slots.
template <typename T>
__device__ __forceinline__ void r2c_untangle_at(T* re, T* im, long long k, long long half, const Tw2& tw2) {
    const long long q = half >> 1;
    if (k == 0) {
        T a0 = re[0], b0 = im[0], r0, rh;
        r2c_untangle_ends<T>(a0, b0, r0, rh);
        re[0] = r0; im[0] = T(0);
        re[half] = rh; im[half] = T(0);
        return;
    }
    T wkr, wki;
    half_twiddle<T>(tw2, (uint32_t)k, wkr, wki);
    if (k == q) {
        T a = re[q], b = im[q];
        r2c_untangle_self<T>(a, b, wkr, wki, re[q], im[q]);
        return;
    }
    const long long m = half - k;
    T a = re[k], b = im[k], c = re[m], d = im[m];
    r2c_untangle_pair<T>(a, b, c, d, wkr, wki, re[k], im[k], re[m], im[m]);
}

template <typename T>
__global__ void __launch_bounds__(256) r2c_untangle_kernel(const __grid_constant__ RealParams<T> p) {
    const long long half = 1LL << p.log2half;
    const long long q = half >> 1;
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    T* re = p.re + (long long)blockIdx.y * p.bstride;
    T* im = p.im + (long long)blockIdx.y * p.bstride;
    if (k > q) return;
    r2c_untangle_at<T>(re, im, k, half, p.tw2);
}

// The same untangle over `members` members of a batch with the (member, k) pairs flattened into grid.x: every thread has
// work whatever N is (r2c_untangle_kernel gives each member whole 256-thread blocks, of which N/4 + 1 threads are active).
template <typename T>
__global__ void __launch_bounds__(256) r2c_untangle_batch_kernel(const __grid_constant__ RealParams<T> p, long long members) {
    const long long half = 1LL << p.log2half;
    const long long q1 = (half >> 1) + 1;            // pairs k = 0 .. N/4 per member
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= members * q1) return;
    const long long b = g / q1, k = g - b * q1;
    r2c_untangle_at<T>(p.re + b * p.bstride, p.im + b * p.bstride, k, half, p.tw2);
}

template <typename T>
__global__ void __launch_bounds__(256) c2r_preprocess_kernel(const __grid_constant__ RealParams<T> p) {
    const long long half = 1LL << p.log2half;
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= half) return;
    const T* ire = p.in_re + (long long)blockIdx.y * p.in_bstride;
    const T* iim = p.in_im + (long long)blockIdx.y * p.in_bstride;
    T* zre = p.re + (long long)blockIdx.y * p.bstride;
    T* zim = p.im + (long long)blockIdx.y * p.bstride;
    const long long m = half - k;
    T c_h, s_h;
    half_twiddle<T>(p.tw2, (uint32_t)k, c_h, s_h);
    // r2c.rs:263-347
    T re_f = ire[k], im_f = iim[k];
    T re_s = ire[m], im_s = -iim[m];
    const cx<T> z = c2r_element<T>(re_f, im_f, re_s, im_s, c_h, s_h);
    zre[k] = z.x;
    zim[k] = z.y;
}

}  // namespace phast
