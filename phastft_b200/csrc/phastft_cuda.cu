// phastft_cuda.cu -- planner, launcher and C ABI of libphastft_cuda.so (see include/phastft_cuda.h).
//
// Reference items replaced (QuState/PhastFT @ 8cd3a39, paths under /root/reference/src):
//   planner.rs:34-114   PlannerDit{64,32}: per-stage cos/sin tables, total 2(N-64) entries
//        -> Plan<T>: pass decomposition N = R_1*R_2[*R_3], a two-level W_N table (2*sqrt(N)
//           f64 entries) for the inter-pass twiddles and one W_R table per pass
//   planner.rs:164-212  PlannerR2c{64,32}                      -> PlanR2c<T>
//   algorithms/dit.rs:263-401 fft_*_dit_with_planner_and_opts  -> run_c2c(): 1-3 kernel launches
//   algorithms/r2c.rs:521-895 r2c / c2r entry points            -> r2c_dev() / c2r_dev()
//   options.rs:10-43    Options                                 -> accepted, no effect on the GPU
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <algorithm>
#include <functional>
#include <vector>

#include "../../include/phastft_cuda.h"
#include "registry.h"

using namespace phast;

// =================================================================================================
// errors
// =================================================================================================
namespace {

thread_local std::string g_last_error;
std::atomic<uint64_t> g_launches{0};

int32_t fail(int32_t code, const std::string& detail = std::string()) {
    g_last_error = phastft_status_message(code);
    if (!detail.empty()) { g_last_error += ": "; g_last_error += detail; }
    return code;
}

#define CUDA_TRY(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) {                                                                        \
            int32_t _code = (_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver ||            \
                             _e == cudaErrorInvalidDevice)                                              \
                                ? PHASTFT_ERR_NO_DEVICE                                                 \
                                : PHASTFT_ERR_CUDA;                                                     \
            (void)cudaGetLastError(); /* clear it: the next kernel-launch check must not see a stale error */ \
            return fail(_code, std::string(#expr) + " -> " + cudaGetErrorString(_e));                   \
        }                                                                                               \
    } while (0)

inline bool is_pow2(size_t n) { return n != 0 && (n & (n - 1)) == 0; }
inline int ilog2(size_t n) { int l = 0; while (n >>= 1) ++l; return l; }

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};


// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
encode_tiled_fn tensor_map_encoder() {
    static encode_tiled_fn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        (void)cudaGetLastError();
        return reinterpret_cast<encode_tiled_fn>(p);
    }();
    return fn;
}
// {cols (contiguous), rows (stride row_stride elements), batch (stride bstride elements)} of T; box {box_cols, box_rows, 1}
template <typename T>
bool encode_tile_map(CUtensorMap* map, const T* base, size_t cols, size_t rows, size_t row_stride, size_t batch, size_t bstride,
                     unsigned box_cols, unsigned box_rows) {
    encode_tiled_fn enc = tensor_map_encoder();
    if (!enc) return false;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || ((row_stride * sizeof(T)) & 15) || ((bstride * sizeof(T)) & 15)) return false;
    cuuint64_t dims[3] = {cols, rows, batch};
    cuuint64_t strides[2] = {row_stride * sizeof(T), bstride * sizeof(T)};
    if (batch == 1) strides[1] = strides[0] * rows;      // unused dimension: any legal stride
    cuuint32_t box[3] = {box_cols, box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUtensorMapDataType dt = sizeof(T) == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    return enc(map, dt, 3, const_cast<T*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// =================================================================================================
// kernel registry (the kernels themselves are instantiated in reg_strided.cu / reg_row.cu / reg_multi.cu)
// =================================================================================================
template <typename T>
const std::vector<KernelEntry<T>>& registry() {
    static const std::vector<KernelEntry<T>> reg = [] {
        std::vector<KernelEntry<T>> v;
        add_row_kernels<T>(v);                       // whole transform in one CTA (rows contiguous in and out)
        add_strided_kernels<T, KIND_COL>(v);         // first / middle passes
        add_strided_kernels<T, KIND_TRANS>(v);       // last pass
        return v;
    }();
    return reg;
}

const char* kind_name(int k) { return k == KIND_COL ? "COL" : k == KIND_TRANS ? "TRANS" : "ROW"; }

// =================================================================================================
// twiddle generation (host, extended precision, octant-reduced so symmetric entries are exact)
// =================================================================================================
void root_of_unity(uint64_t k, uint64_t n, double& re, double& im) {
    // W_n^k = exp(-2*pi*i*k/n), n a power of two
    k &= (n - 1);
    if (n < 8) {
        // n in {1, 2, 4}
        static const double c4[4] = {1, 0, -1, 0}, s4[4] = {0, -1, 0, 1};
        uint64_t q = k * (4 / n);
        re = c4[q]; im = s4[q];
        return;
    }
    const uint64_t eighth = n / 8;
    const uint64_t oct = k / eighth, rem = k % eighth;
    auto cs = [&](uint64_t j, long double& c, long double& s) {
        if (j == 0) { c = 1.0L; s = 0.0L; return; }
        if (j == eighth) { c = s = 0.70710678118654752440084436210484903928L; return; }
        long double a = 2.0L * 3.14159265358979323846264338327950288L * (long double)j / (long double)n;
        c = cosl(a); s = sinl(a);
    };
    long double c, s, co, si;
    switch (oct) {
        case 0: cs(rem, c, s); co = c; si = s; break;
        case 1: cs(eighth - rem, c, s); co = s; si = c; break;
        case 2: cs(rem, c, s); co = -s; si = c; break;
        case 3: cs(eighth - rem, c, s); co = -c; si = s; break;
        case 4: cs(rem, c, s); co = -c; si = -s; break;
        case 5: cs(eighth - rem, c, s); co = -s; si = -c; break;
        case 6: cs(rem, c, s); co = s; si = -c; break;
        default: cs(eighth - rem, c, s); co = c; si = -s; break;
    }
    re = (double)co;
    im = (double)(-si);
    if (re == 0.0) re = 0.0;
    if (im == 0.0) im = 0.0;
}

// =================================================================================================
// plans
// =================================================================================================
constexpr int MAX_PASSES = 3;

// First 256 bytes of a plan's table blob: what the rest of the blob was laid out for.  Offsets and the W_L^(c*m)
// tables depend on the pass decomposition and on each pass's kernel (tile width, first radix), which can differ
// between ranks (PlannerMode::Tune, PHASTFT_* overrides): import / broadcast compare headers first.
constexpr size_t BLOB_HEADER_BYTES = 256;
struct BlobHeader {
    uint64_t magic;        // "PHASTFT2"
    uint64_t bytes;        // whole blob, header included
    uint64_t n;
    uint32_t precision_bits, num_passes;
    uint64_t layout_sig;   // FNV-1a of the plan description (factors, kernels, radices, variants)
};
static_assert(sizeof(BlobHeader) <= BLOB_HEADER_BYTES, "header fits its slot");
constexpr uint64_t BLOB_MAGIC = 0x3254464854534150ull;
inline uint64_t fnv1a(const std::string& str) {
    uint64_t h = 1469598103934665603ull;
    for (unsigned char c : str) { h ^= c; h *= 1099511628211ull; }
    return h;
}
constexpr int ALT_ROW_PASS = -1;   // launch_pass(): use Plan::alt_row

template <typename T>
struct PassDesc {
    const KernelEntry<T>* k = nullptr;    // kernel for a lone transform
    const KernelEntry<T>* kb = nullptr;   // kernel when the call carries many transforms (multi-wave grids)
    const KernelEntry<T>* kt = nullptr;   // 2-pass plans of lone transforms: the pass with an asynchronous (TMA) tile input
    const KernelEntry<T>* kc = nullptr;   // first pass only: `k` with the c2r pre-processing folded into its loads (MODE_C2R_IN)
    const KernelEntry<T>* kcb = nullptr;  // ... the same for batched c2r calls: `kb`'s build (first COL pass: any build of the same R)
    const KernelEntry<T>* kf = nullptr;   // one-CTA kernels: `k` / `kb` with the r2c untangle on store (MODE_R2C_OUT), if they have
    const KernelEntry<T>* kfb = nullptr;  // a shared-memory stage
    const KernelEntry<T>* kr = nullptr;   // one-CTA plans: `kb` with its tile moved in and out by cp.async.bulk (MODE_ROW_BULK)
    size_t tw_wc_off_t = (size_t)-1;      // W_L^(c*m) table for `kt`
    size_t tw_im_off = (size_t)-1;        // one-CTA kernels: the per-stage [i][m] stage-twiddle tables for `k` ...
    size_t tw_im_off_b = (size_t)-1;      // ... and for `kb`
    int log2R = 0, log2A = 0, log2B = 0, log2R1 = 0, log2Rprev = 0, has_tw = 0, tw_shift = 0;
    size_t tw_stage_off = 0;  // byte offsets into the table blob
    size_t tw_wc_off = (size_t)-1;
    size_t tw_wc_off_b = (size_t)-1;      // same table for `kb` (depends on its C and first radix)
};

template <typename T>
struct Plan {
    size_t n = 0;
    int log2n = 0;
    int device = 0;
    int num_passes = 0;
    PassDesc<T> pass[MAX_PASSES];
    PassDesc<T> alt_row;               // multi-pass N that one CTA can hold (<= 128 KB): the one-CTA kernel, used for batches
    size_t alt_row_min_batch = 4;
    bool tma_lone = false;             // 2-pass plans: lone transforms through the asynchronous-input pair pass[].kt (PHASTFT_TMA=1)
    bool tma_batch = false;            // ... and batched calls (batch * N >= 2^21): the default where the pair exists (PHASTFT_TMA_BATCH=0 disables)
    const ClusterEntry<T>* cl = nullptr;   // both passes in ONE launch by a thread-block cluster (exchange through DSMEM)
    PassDesc<T> cl_pass[2];
    size_t cl_min_batch = 0;           // calls with at least this many transforms use the cluster launch
    int cl_max_active = 0;             // cudaOccupancyMaxActiveClusters of that launch on this device
    // 2-pass plans: both passes in one persistent launch, intermediates in an L2-resident ring (fft_pipe2_kernel)
    const PipeEntry<T>* pipe_b = nullptr;   // for batched calls (pairs pass[0].kb / pass[1].kb)
    const PipeEntry<T>* pipe_1 = nullptr;   // for a lone transform (pairs pass[0].k / pass[1].k); off unless PHASTFT_PIPE_LONE=1
    int pipe_grid_b = 0, pipe_grid_1 = 0;   // co-resident CTAs of those launches on this device
    mutable unsigned char* pipe_state = nullptr;   // ticket + done1[batch] + done2[batch], zeroed per call
    mutable size_t pipe_state_batch = 0;
    // table blob: [tw2_hi][tw2_lo][per pass W_R][wc]
    std::vector<unsigned char> blob_host;
    unsigned char* blob_dev = nullptr;
    size_t hi_off = 0, lo_off = 0;
    int lo_bits = 0;
    // workspace (multi-pass only) and host-API staging, grown lazily under `mu`
    mutable std::mutex mu;
    mutable std::mutex host_mu;         // held for a whole *_host call: staging buffers + the plan's streams are per plan
    mutable T* ws_re = nullptr;
    mutable T* ws_im = nullptr;
    mutable size_t ws_elems = 0;        // per array; ONE allocation of 2*ws_elems, ws_im = ws_re + ws_elems
    int ws_il = -1;                     // layout of the intermediates between passes: 0 planar, 1 interleaved
                                        // complex, -1 = interleaved for 3-pass plans and large batches (run_c2c)
    T* ws2_re = nullptr;                // 3-pass plans: L2-resident scratch for one k1 group (see run_c2c)
    T* ws2_im = nullptr;
    long long l2_group = 0;             // k1 values per group
    mutable T* stage_re = nullptr;      // host-API staging (N each, or 2N for interleaved in stage_re)
    mutable T* stage_im = nullptr;
    mutable size_t stage_elems = 0;
    mutable cudaStream_t stream = nullptr;   // used by the *_host entry points
    mutable cudaStream_t stream_h2d = nullptr;   // copy streams of the pipelined batch host path (created lazily)
    mutable cudaStream_t stream_d2h = nullptr;
    mutable cudaEvent_t ws_free = nullptr;   // orders workspace reuse across streams
    mutable cudaStream_t ws_last_stream = nullptr;
    mutable bool ws_used = false;
    std::string description;

    ~Plan() {
        DeviceGuard g(device);
        if (blob_dev) cudaFree(blob_dev);
        if (ws_re) cudaFree(ws_re);
        if (pipe_state) cudaFree(pipe_state);
        if (ws2_re) cudaFree(ws2_re);
        if (ws2_im) cudaFree(ws2_im);
        if (stage_re) cudaFree(stage_re);
        if (stage_im) cudaFree(stage_im);
        if (ws_free) cudaEventDestroy(ws_free);
        if (stream) cudaStreamDestroy(stream);
        if (stream_h2d) cudaStreamDestroy(stream_h2d);
        if (stream_d2h) cudaStreamDestroy(stream_d2h);
    }
};

// Layout of the intermediates between passes: planar (two halves of the workspace) or interleaved
// complex.  Interleaved makes every access a 16-byte (f64) element, so a 64-byte run needs half as many
// columns: the 1024-row middle tile of 2^25..2^26 shrinks from 128 KB to 64 KB and two CTAs share an SM
// (2^26 f64 middle pass 646 -> 513 us, profiles/r01_tune25*.txt); streaming passes gain 2-9 % (tune24/25), single
// L2-resident transforms lose 2-7 %, hence the automatic rule.  PHASTFT_WS_IL=0|1 forces a layout.
inline int ws_interleaved_mode() {
    const char* e = getenv("PHASTFT_WS_IL");
    return e ? (atoi(e) != 0 ? 1 : 0) : -1;
}

// An explicit plan choice (PlannerMode::Tune tries several and keeps the fastest); consulted by
// choose_factors / pick_kernel before the heuristics, like the PHASTFT_FACTORS / PHASTFT_PASS_C env overrides.
struct PlanChoice {
    std::vector<int> factors;   // log2 of each pass size
    std::vector<int> pass_c;    // tile columns per pass (0 = heuristic)
};
thread_local const PlanChoice* g_choice = nullptr;

// pass sizes (log2) for a transform of 2^n points -------------------------------------------------
template <typename T>
std::vector<int> choose_factors(int n) {
    if (g_choice && !g_choice->factors.empty()) return g_choice->factors;
    // override: PHASTFT_FACTORS="20:10,10;26:9,9,8"  (applies to both precisions; tuning aid)
    if (const char* env = getenv("PHASTFT_FACTORS")) {
        std::string s(env);
        size_t pos = 0;
        while (pos < s.size()) {
            size_t end = s.find(';', pos);
            if (end == std::string::npos) end = s.size();
            std::string item = s.substr(pos, end - pos);
            size_t colon = item.find(':');
            if (colon != std::string::npos && atoi(item.substr(0, colon).c_str()) == n) {
                std::vector<int> f;
                int sum = 0;
                size_t p = colon + 1;
                while (p < item.size()) {
                    size_t q = item.find(',', p);
                    if (q == std::string::npos) q = item.size();
                    f.push_back(atoi(item.substr(p, q - p).c_str()));
                    sum += f.back();
                    p = q + 1;
                }
                if (sum == n && !f.empty() && (int)f.size() <= MAX_PASSES) return f;
            }
            pos = end + 1;
        }
    }
    // A lone transform is one CTA only while that beats two many-CTA passes (profiles/r02_exp_lone_row.txt, after the stage
    // twiddles of the one-CTA kernels became contiguous loads + products: f64 2^11 3.3 us in one CTA vs 4.1 us as {5,6}, 2^12 4.7 vs
    // 4.5; f32 2^12 3.1 us, 2^13 5.0 vs 5.6 as {6,7}).  Batches of <= 2^13 (f64) / 2^14 (f32) points always use a one-CTA
    // kernel (Plan::alt_row): one launch, one HBM round trip.
    const int single_max = sizeof(T) == 8 ? 11 : 13;
    if (n <= single_max) return {n};
    // two passes while both tiles stay <= 1024 points long; the ends of a 3-pass plan are kept at
    // 2^8 so they can use 128-byte runs in a 64 KB tile, the middle pass takes the rest (<= 2^10)
    // measured-best splits (profiles/r01_tune7*.txt, profiles/r01_tuning.md)
    if (n <= 16) { int a = n / 2; return {a, n - a}; }
    if (n <= 20) { int a = (n + 1) / 2; return {a, n - a}; }
    if (n <= 22) return {7, n - 14, 7};
    if (n <= 26) return {8, n - 16, 8};
    // beyond 2^26 an end pass has to grow too: the 1024-row pass goes in the middle (its tile arrives by TMA at 0.84 of the peak), the
    // smaller end first (256-row first pass with 128-byte runs): 2^27 as {8,10,9} 2323 us vs 2743 us as {9,9,9} (f64), 1282 vs 1461 (f32),
    // profiles/r02_exp_mid_batch.txt
    // (2^28: {8,10,10} 4856 / 2595 us against 5589 / 2908 as {9,10,9} and 5842 / 2993 as {10,9,9})
    if (n == 27) return {8, 10, 9};
    if (n == 28) return {8, 10, 10};
    if (n == 29) return {9, 10, 10};
    int a = (n + 2) / 3, b = (n - a + 1) / 2;
    return {a, n - a - b, b};
}

// `l2_resident`: the whole signal fits L2 (a few MiB .. 64 MiB).  There the passes are launch- and
// latency-bound single waves and the tile width is chosen by a wave model (profiles/r01_tune15*.txt, r01_tune16:
// 2^18 f64 8.8 us with 4-column tiles vs 12.2 us with 8; 2^20 f32 16.6 us with 8 columns vs 25.4 us
// with 16; 2^20 f64 stays at 8 columns because its 1024-row tile holds only one CTA per SM).
template <typename T>
const KernelEntry<T>* pick_kernel(int kind, int R, int max_c, int pass_index, bool hbm_strided, bool l2_resident = false,
                                  size_t rows_total = 0, int pref_c = 0, int pref_variant = 0) {
    int want_c = pref_c, want_variant = pref_variant;
    auto nth = [&](const char* name, int& out) {
        if (const char* env = getenv(name)) {
            std::string sv(env);
            size_t pos = 0;
            for (int i = 0; pos <= sv.size(); ++i) {
                size_t q = sv.find(',', pos);
                if (q == std::string::npos) q = sv.size();
                if (i == pass_index) out = atoi(sv.substr(pos, q - pos).c_str());
                pos = q + 1;
            }
        }
    };
    if (const char* env = getenv("PHASTFT_TILE_C")) want_c = atoi(env);
    if (const char* env = getenv("PHASTFT_VARIANT")) want_variant = atoi(env);
    nth("PHASTFT_PASS_C", want_c);                 // e.g. "16,8,16"
    if (g_choice && pass_index >= 0 && pass_index < (int)g_choice->pass_c.size() && g_choice->pass_c[pass_index] > 0)
        want_c = g_choice->pass_c[pass_index];
    nth("PHASTFT_PASS_VARIANT", want_variant);     // e.g. "0,5,0"
    const int CH = TileC<T>::CH, CN = TileC<T>::CN, CW = TileC<T>::CW;
    const size_t tile_limit = 72 * 1024;           // keep >= 3 CTAs/SM worth of shared memory
    const KernelEntry<T>* best = nullptr;
    int best_rank = 1 << 30;
    for (const auto& e : registry<T>()) {
        if (e.kind != kind || e.R != R || e.mode != MODE_PLAIN) continue;
        if (kind != KIND_ROW && e.C > max_c) continue;
        if (e.variant != want_variant) continue;
        int rank;
        if (kind == KIND_ROW) rank = 0;
        else if (want_c) rank = (e.C == want_c) ? 0 : 10 + abs(e.C - want_c);
        else if (l2_resident) {
            // cost ~ (waves of CTAs) x (points per tile): a pass over an L2-resident signal is one or two
            // latency-bound waves, so smaller tiles win until they no longer fit the chip in one wave
            if (e.C != CH && e.C != CN && e.C != CW) continue;
            int occ = 1, sms = 148, dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            cudaFuncSetAttribute(e.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e.smem);
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, e.fn, e.NT, e.smem) != cudaSuccess || occ < 1) occ = 1;
            const size_t ctas = std::max<size_t>(1, rows_total / (size_t)e.C);
            const size_t waves = (ctas + (size_t)sms * occ - 1) / ((size_t)sms * occ);
            rank = (int)std::min<size_t>(waves * (size_t)e.R * e.C, 1u << 24) * 4 - ilog2(e.C);   // tie -> wider tile
        }
        else if (hbm_strided) rank = (e.C == CW && e.smem <= tile_limit) ? 0 : (e.C == CN) ? 1 : (e.C == CW) ? 2 : (e.C == CH) ? 4 : 3;
        else rank = (e.C == CN) ? 0 : (e.C == CW && e.smem <= tile_limit) ? 1 : (e.C == CH) ? 2 : 3;
        if (rank < best_rank) { best = &e; best_rank = rank; }
    }
    if (!best && want_variant != 0) {   // requested variant does not exist for this tile: fall back to the default
        for (const auto& e : registry<T>())
            if (e.kind == kind && e.R == R && e.variant == 0 && e.mode == MODE_PLAIN && (kind == KIND_ROW || e.C <= max_c) && !best) best = &e;
    }
    return best;
}

// One-CTA kernels: for a batch the radix-16 builds win at some sizes (profiles/r01_tune19*.txt: 2^8 6.7 vs 4.5 TB/s,
// f32 2^11 3.4 vs 2.2 TB/s, f64 2^11/2^12 3.4 vs 2.9 TB/s) while a lone transform prefers the default.
template <typename T>
const KernelEntry<T>* pick_row_batch_kernel(int R, const KernelEntry<T>* dflt) {
    if (const char* env = getenv("PHASTFT_ROW_VARIANT")) {        // re-tuning override
        const int want = atoi(env);
        for (const auto& e : registry<T>())
            if (e.kind == KIND_ROW && e.R == R && e.variant == want) return &e;
    }
    // measured per size, batches of 2^24 points, after the stage twiddles of these kernels became contiguous loads + products
    // (profiles/r02_exp_row2.txt; round 1's choices: profiles/r01_tune19*.txt, r01_tune29*.txt); 0 = the lone-transform kernel is
    // also the best batch kernel (f64 2^9 / 2^10: 82.7 / 83.1 us = 0.98-0.99 of the measured HBM peak)
    const bool f64 = sizeof(T) == 8;
    int want = 0;
    switch (R) {
        case 4: case 8: want = 80; break;
        case 16: want = f64 ? 80 : 81; break;
        case 256: want = 70; break;
        case 512: want = f64 ? 0 : 81; break;
        case 1024: want = 0; break;
        case 2048: want = f64 ? 81 : 70; break;
        case 4096: want = 70; break;
        case 8192: want = f64 ? 90 : 0; break;
        case 16384: want = 91; break;
        default: break;
    }
    for (const auto& e : registry<T>())        // want == 0: the plain build (the lone-transform choice may be another variant)
        if (e.kind == KIND_ROW && e.R == R && e.variant == want && e.mode == MODE_PLAIN) return &e;
    return dflt;
}

// The MODE_ROW_BULK build of a one-CTA batch kernel (same radices, C and id; NT may differ), or NULL.  Opt-in (PHASTFT_ROW_BULK=1):
// bit-identical and measured equal or slower at every size (profiles/r02_exp_row_bulk.txt: f32 2^5 82.9 vs 77.5 us per 2^24
// points, f64 2^12 169 vs 93 with the doubled shared memory) -- these kernels are not bound by their per-lane global accesses.
template <typename T>
const KernelEntry<T>* find_row_bulk(const KernelEntry<T>* kb) {
    if (!kb || kb->kind != KIND_ROW) return nullptr;
    const char* env = getenv("PHASTFT_ROW_BULK");
    if (!env || atoi(env) == 0) return nullptr;
    for (const auto& e : registry<T>())
        if (e.mode == MODE_ROW_BULK && e.kind == KIND_ROW && e.R == kb->R && e.C == kb->C && e.variant == kb->variant && e.rl == kb->rl) return &e;
    return nullptr;
}

// The build of `k`'s tile (same kind, radices, C, NT and id) with the given MODE_*, or NULL (the last registered, if several).
template <typename T>
const KernelEntry<T>* find_mode(const KernelEntry<T>* k, int mode) {
    const KernelEntry<T>* found = nullptr;
    if (!k) return found;
    for (const auto& e : registry<T>())
        if (e.mode == mode && e.kind == k->kind && e.R == k->R && e.C == k->C && e.NT == k->NT && e.variant == k->variant && e.rl == k->rl) found = &e;
    return found;
}
// the MODE_C2R_IN / MODE_R2C_OUT builds of a one-CTA pass's kernels (batched real transforms)
template <typename T>
void find_real_modes(PassDesc<T>& d) {
    d.kc = find_mode(d.k, MODE_C2R_IN); d.kcb = find_mode(d.kb, MODE_C2R_IN);
    d.kf = find_mode(d.k, MODE_R2C_OUT); d.kfb = find_mode(d.kb, MODE_R2C_OUT);
}

// Entries of the concatenated per-stage [i][m] stage-twiddle tables of a one-CTA kernel (stage q >= 1 owns Ns(q) * rad(q)).
template <typename T>
size_t tw_im_entries(const KernelEntry<T>* k) {
    size_t tot = 0, ns = (size_t)k->rads[0];
    for (int q = 1; q < k->stages; ++q) { tot += ns * (size_t)k->rads[q]; ns *= (size_t)k->rads[q]; }
    return tot;
}

template <typename T>
int32_t build_plan(size_t n, int device, Plan<T>** out) {
    if (!out) return fail(PHASTFT_ERR_INVALID_ARG, "out == NULL");
    *out = nullptr;
    if (!is_pow2(n)) return fail(PHASTFT_ERR_NOT_POW2);          // planner.rs:66
    if (n > (size_t(1) << 30)) return fail(PHASTFT_ERR_INVALID_ARG, "num_points > 2^30 not supported");
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count == 0) return fail(PHASTFT_ERR_NO_DEVICE, ce != cudaSuccess ? cudaGetErrorString(ce) : "");
    if (device < 0 || device >= count) return fail(PHASTFT_ERR_NO_DEVICE, "device ordinal out of range");
    DeviceGuard guard(device);

    std::unique_ptr<Plan<T>> pl(new Plan<T>());
    pl->n = n;
    pl->log2n = ilog2(n);
    pl->device = device;
    const int ln = pl->log2n;

    std::vector<int> f = ln == 0 ? std::vector<int>{} : choose_factors<T>(ln);
    pl->num_passes = (int)f.size();
    pl->ws_il = ws_interleaved_mode();
    const bool il3 = pl->num_passes == 3 && pl->ws_il != 0;   // the middle pass reads and writes interleaved data
    // two-level W_N table
    pl->lo_bits = (ln + 1) / 2;
    const size_t n_lo = size_t(1) << pl->lo_bits, n_hi = size_t(1) << (ln - pl->lo_bits);
    size_t off = BLOB_HEADER_BYTES;
    pl->hi_off = off; off += n_hi * sizeof(double2);
    pl->lo_off = off; off += n_lo * sizeof(double2);

    int acc = 0;
    for (int p = 0; p < pl->num_passes; ++p) {
        PassDesc<T>& d = pl->pass[p];
        d.log2R = f[p];
        d.log2A = acc;
        d.log2B = ln - acc - f[p];
        d.log2R1 = f[0];
        acc += f[p];
        const bool last = (p == pl->num_passes - 1);
        const int kind = pl->num_passes == 1 ? KIND_ROW : (last ? KIND_TRANS : KIND_COL);
        const int max_c = kind == KIND_COL ? (1 << d.log2B) : kind == KIND_TRANS ? (1 << f[0]) : (1 << 30);
        // wide (128-byte) runs pay off once the signal no longer lives in L2; below that more, smaller CTAs win
        const bool big = ln >= 21;     // above 2^20 the passes are multi-wave streams, below single latency-bound waves
        const bool wide = (p == 0 || last) && big;
        // interleaved 1024-row middle pass: half-width (64-byte-run) tile, two CTAs per SM
        const bool half_mid = il3 && p == 1 && f[p] == 10;
        // lone 2^11-point f32 transform in one CTA: 8x16x16 (3.7 us) beats 4x8x8x8 (4.4 us), profiles/r01_tune30*.txt
        const bool row2048_f32 = kind == KIND_ROW && f[p] == 11 && sizeof(T) == 4;
        // round 2 (profiles/r02_exp_lone_row.txt): f64 2^11 8x16x16 3.3 us (4x8x8x8: 3.7); f32 2^12 16x16x16 3.1 us (8x8x8x8: 4.1);
        // f32 2^13 16x16x32 5.0 us (16x8x8x8: 5.6)
        const bool row_r16 = kind == KIND_ROW && ((f[p] == 11 && sizeof(T) == 8) || (f[p] == 12 && sizeof(T) == 4));
        const bool row8192_f32 = kind == KIND_ROW && f[p] == 13 && sizeof(T) == 4;
        const int pref_c = half_mid ? TileC<T>::CH : 0, pref_v = half_mid ? 62 : (row2048_f32 || row_r16) ? 70 : row8192_f32 ? 91 : 0;
        d.k = pick_kernel<T>(kind, 1 << f[p], max_c, p, /*hbm_strided=*/wide, /*l2_resident=*/!big, /*rows_total=*/n >> f[p], pref_c, pref_v);
        // batched calls are multi-wave streams whatever N is: wide runs only where the rows of a tile are
        // far apart in memory (>= 64 KiB: first-pass loads, last-pass stores of large N), else 64-byte runs
        const size_t far_stride = (kind == KIND_COL ? (size_t(1) << d.log2B) : (n >> f[p])) * sizeof(T);
        const bool wide_b = (p == 0 || last) && far_stride >= (size_t(64) << 10);
        // f32 batches of 2^17..2^20 points: 32-byte-run tiles (more CTAs per SM) 115-122 us per 2^24 points vs 117-140 us with 64-byte
        // runs (profiles/r02_exp_mid_batch.txt); f64 measured the other way round and keeps its 64-byte runs
        // (the opt-in pipelined launch is compiled for the 64-byte-run pairs: whenever PHASTFT_PIPE is set, to 0 or 1, the batch
        // kernels stay those, so that the two settings run the same pass kernels and can be compared bit for bit)
        const bool pipe_on = getenv("PHASTFT_PIPE") != nullptr;
        const int pref_c_b = (sizeof(T) == 4 && pl->num_passes == 2 && ln >= 17 && kind != KIND_ROW && !pipe_on) ? TileC<T>::CH : pref_c;
        d.kb = (kind == KIND_ROW) ? pick_row_batch_kernel<T>(1 << f[p], d.k) : pick_kernel<T>(kind, 1 << f[p], max_c, p, /*hbm_strided=*/wide_b, false, 0, pref_c_b, pref_v);
        if (!d.k) return fail(PHASTFT_ERR_INVALID_ARG, "no kernel for pass size 2^" + std::to_string(f[p]) + " kind " + kind_name(kind));
        if (kind == KIND_ROW) d.kr = find_row_bulk<T>(d.kb);
        if (kind == KIND_ROW) find_real_modes(d);
        if (p == 0 && kind == KIND_COL) {       // the same tile with the c2r pre-processing in its loads, if compiled (c2r_dev uses it)
            d.kc = find_mode(d.k, MODE_C2R_IN);
            // batched c2r: no table of a first COL pass depends on its tile, so any build of the same R serves if kb has none
            d.kcb = find_mode(d.kb, MODE_C2R_IN);
            for (const auto& e : registry<T>())
                if (!d.kcb && e.mode == MODE_C2R_IN && e.kind == kind && e.R == d.k->R && e.C <= max_c) d.kcb = &e;
        }
        if (p > 0) {
            d.has_tw = 1;
            d.log2Rprev = f[p - 1];
            d.tw_shift = ln - (f[p - 1] + f[p] + d.log2B);
        }
        d.tw_stage_off = off; off += (size_t(1) << f[p]) * sizeof(cx<T>);
        if (kind == KIND_ROW) {
            off = (off + 255) & ~size_t(255);
            d.tw_im_off = off; off += std::max<size_t>(1, tw_im_entries<T>(d.k)) * sizeof(cx<T>);
            if (d.kb && d.kb != d.k) {
                off = (off + 255) & ~size_t(255);
                d.tw_im_off_b = off; off += std::max<size_t>(1, tw_im_entries<T>(d.kb)) * sizeof(cx<T>);
            } else {
                d.tw_im_off_b = d.tw_im_off;
            }
        }
        if (kind == KIND_TRANS && pl->num_passes == 2) {
            d.tw_wc_off = off;
            off += (size_t)d.k->C * ((size_t(1) << f[p]) / d.k->first_radix) * sizeof(cx<T>);
            if (d.kb && d.kb != d.k) {
                off = (off + 255) & ~size_t(255);
                d.tw_wc_off_b = off;
                off += (size_t)d.kb->C * ((size_t(1) << f[p]) / d.kb->first_radix) * sizeof(cx<T>);
            } else {
                d.tw_wc_off_b = d.tw_wc_off;
            }
        }
        off = (off + 255) & ~size_t(255);
    }
    // Two-pass plans with both tiles of 256 / 512 / 1024 rows (2^16..2^20 points): a pair of asynchronous-input kernels (TMA boxes
    // of the planar input into the first pass's tile, bulk copies of the interleaved workspace's rows into the second's).
    //   batched calls (batch * N >= 2^21, multi-wave grids): the default -- f64 2^20 x 16 279 -> 199 us, 2^19 250 -> 203, 2^17
    //   208 -> 182, 2^16 188 -> 168; f32 2^18 122 -> 103, 2^17 116 -> 96, 4096 x 2^16 1323 -> 1275 us (profiles/r02_exp_tma_batch.txt);
    //   PHASTFT_TMA_BATCH=0 keeps the register-staged kernels
    //   lone transforms (single-wave grids): equal or slower (profiles/r02_exp_tma1.txt), opt-in with PHASTFT_TMA=1
    // PHASTFT_TMA_VARIANT picks a build (300: 64 KB tiles, 301: 128 KB tiles).
    if (pl->num_passes == 2) {
        int lone = 0, batch = 1, want = 300;
        if (const char* env = getenv("PHASTFT_TMA")) lone = atoi(env);
        if (const char* env = getenv("PHASTFT_TMA_BATCH")) batch = atoi(env);
        else if (getenv("PHASTFT_PIPE")) batch = 0;    // A/B runs of the pipelined launch compare against the kernels it is built from
        if (getenv("PHASTFT_TMA_VARIANT") && !getenv("PHASTFT_TMA")) lone = 1;
        if (const char* env = getenv("PHASTFT_TMA_VARIANT")) want = atoi(env);
        const bool enabled = lone || batch;
        pl->tma_lone = lone != 0; pl->tma_batch = batch != 0;
        const KernelEntry<T>* t0 = nullptr; const KernelEntry<T>* t1 = nullptr;
        if (enabled && tensor_map_encoder())
            for (const auto& e : registry<T>()) {
                if (e.variant != want) continue;
                if (e.mode == MODE_TMA_IN && e.kind == KIND_COL && e.R == (1 << f[0]) && e.C <= (1 << f[1])) t0 = &e;
                if (e.mode == MODE_BULK_IN && e.kind == KIND_TRANS && e.R == (1 << f[1]) && e.C <= (1 << f[0])) t1 = &e;
            }
        if (t0 && t1) {
            pl->pass[0].kt = t0; pl->pass[1].kt = t1;
            PassDesc<T>& d = pl->pass[1];
            d.tw_wc_off_t = off;
            off += (size_t)t1->C * ((size_t(1) << f[1]) / t1->first_radix) * sizeof(cx<T>);
            off = (off + 255) & ~size_t(255);
        }
    }
    // 3-pass plans with interleaved intermediates: the 1024-row middle pass with its tile arriving by TMA (64 KB landing zone =
    // the tile, no register-staged loads: three CTAs per SM each with its whole tile in flight).  PHASTFT_TMA_MID=0|1.
    if (pl->num_passes == 3 && il3) {
        int enabled = 1, ends = 0;
        if (const char* env = getenv("PHASTFT_TMA_MID")) enabled = atoi(env);
        if (const char* env = getenv("PHASTFT_TMA_ENDS")) ends = atoi(env);
        if (tensor_map_encoder())
            for (const auto& e : registry<T>()) {
                if (enabled >= 2 && e.variant == 310 && e.mode == MODE_TMA_IN && e.kind == KIND_COL && e.R == (1 << f[1]) && e.C == TileC<T>::CH) pl->pass[1].kt = &e;
                if (e.variant != 300) continue;
                if (enabled && e.mode == MODE_TMA_IN && e.kind == KIND_COL && e.R == (1 << f[1]) && e.C == TileC<T>::CH) pl->pass[1].kt = &e;
                // the 128-byte-run end passes: planar boxes in (first pass), contiguous rows of the workspace in (last pass)
                if (ends && e.mode == MODE_TMA_IN && e.kind == KIND_COL && e.R == (1 << f[0]) && e.C == TileC<T>::CW) pl->pass[0].kt = &e;
                if (ends && e.mode == MODE_BULK_IN && e.kind == KIND_TRANS && e.R == (1 << f[2]) && e.C == TileC<T>::CW) pl->pass[2].kt = &e;
            }
    }
    // Batches of transforms that one CTA can hold (128 KB tile: 2^13 f64, 2^14 f32) use a one-CTA kernel: one launch,
    // one HBM round trip.  PHASTFT_ONE_CTA_MAX (log2) lowers the limit for re-tuning.
    // 2^13 f64 / 2^13-2^14 f32 in one CTA (64-128 KB tile): slower than two passes of small tiles while the stage twiddles were
    // gathers (205 vs 182 us and 159 vs 97 us per 2^24 points, profiles/r02_exp_cluster1.txt), faster since they are contiguous
    // loads + products (f64 2^13 147 vs 172 us, f32 2^13 61 vs 95, f32 2^14 78 vs 94, profiles/r02_exp_row2.txt).
    int one_cta_max = sizeof(T) == 8 ? 13 : 14;
    if (const char* env = getenv("PHASTFT_ONE_CTA_MAX")) one_cta_max = std::min(atoi(env), sizeof(T) == 8 ? 13 : 14);
    if (pl->num_passes >= 2 && ln <= one_cta_max) {
        PassDesc<T>& d = pl->alt_row;
        d.log2R = ln; d.log2A = 0; d.log2B = 0; d.log2R1 = ln;
        d.k = pick_kernel<T>(KIND_ROW, 1 << ln, 1 << 30, 0, false);
        d.k = pick_row_batch_kernel<T>(1 << ln, d.k);            // alt_row is only ever used for batches
        d.kb = d.k;
        d.kr = find_row_bulk<T>(d.kb);
        find_real_modes(d);
        if (d.k) {
            d.tw_stage_off = off; off += (size_t(1) << ln) * sizeof(cx<T>);
            off = (off + 255) & ~size_t(255);
            d.tw_im_off = d.tw_im_off_b = off; off += std::max<size_t>(1, tw_im_entries<T>(d.k)) * sizeof(cx<T>);
            off = (off + 255) & ~size_t(255);
            pl->alt_row_min_batch = ln <= 12 ? 4 : 32;
        }
    }
    // Larger transforms up to the shared memory of a cluster (2^14..2^16 f64, 2^15..2^16 f32): both passes in one
    // cluster launch.  PHASTFT_CLUSTER=0 disables, PHASTFT_CLUSTER_VARIANT=<id> picks a build, PHASTFT_CLUSTER_MIN_BATCH
    // sets the smallest call that uses it (a lone transform keeps K SMs busy, the two-launch plan the whole chip).
    {
        int want = 0, enabled = 0;        // measured slower than the two-launch plan at every size (profiles/r02_exp_cluster1.txt): opt-in
        if (const char* env = getenv("PHASTFT_CLUSTER")) enabled = atoi(env);
        if (const char* env = getenv("PHASTFT_CLUSTER_VARIANT")) { want = atoi(env); if (!getenv("PHASTFT_CLUSTER")) enabled = 1; }
        if (getenv("PHASTFT_CLUSTER_MIN_BATCH") && !getenv("PHASTFT_CLUSTER")) enabled = 1;
        if (enabled && !pl->alt_row.k)
            for (const auto& ce : cluster_registry<T>())
                if (ce.log2n == ln && ce.variant == want) { pl->cl = &ce; break; }
        if (pl->cl) {
            pl->cl_min_batch = 8;
            if (const char* env = getenv("PHASTFT_CLUSTER_MIN_BATCH")) pl->cl_min_batch = (size_t)std::max(1, atoi(env));
            const int l1 = ilog2((size_t)pl->cl->k1.R), l2 = ilog2((size_t)pl->cl->k2.R);
            PassDesc<T>& a = pl->cl_pass[0];
            a.k = a.kb = &pl->cl->k1;
            a.log2R = l1; a.log2A = 0; a.log2B = l2; a.log2R1 = l1;
            a.tw_stage_off = off; off += (size_t(1) << l1) * sizeof(cx<T>);
            off = (off + 255) & ~size_t(255);
            PassDesc<T>& b = pl->cl_pass[1];
            b.k = b.kb = &pl->cl->k2;
            b.log2R = l2; b.log2A = l1; b.log2B = 0; b.log2R1 = l1;
            b.has_tw = 1; b.log2Rprev = l1; b.tw_shift = 0;
            b.tw_stage_off = off; off += (size_t(1) << l2) * sizeof(cx<T>);
            b.tw_wc_off = b.tw_wc_off_b = off;
            off += (size_t)b.k->C * ((size_t(1) << l2) / b.k->first_radix) * sizeof(cx<T>);
            off = (off + 255) & ~size_t(255);
        }
    }
    // ---- fill the blob ------------------------------------------------------------------------------
    pl->blob_host.assign(off, 0);
    {
        double2* hi = reinterpret_cast<double2*>(pl->blob_host.data() + pl->hi_off);
        double2* lo = reinterpret_cast<double2*>(pl->blob_host.data() + pl->lo_off);
        for (size_t h = 0; h < n_hi; ++h) root_of_unity((uint64_t)h << pl->lo_bits, n, hi[h].x, hi[h].y);
        for (size_t l = 0; l < n_lo; ++l) root_of_unity(l, n, lo[l].x, lo[l].y);
    }
    auto fill_pass_tables = [&](PassDesc<T>& d) {
        const size_t R = size_t(1) << d.log2R;
        cx<T>* tw = reinterpret_cast<cx<T>*>(pl->blob_host.data() + d.tw_stage_off);
        for (size_t e = 0; e < R; ++e) {
            double re, im;
            root_of_unity(e, R, re, im);
            tw[e].x = (T)re; tw[e].y = (T)im;
        }
        for (int which = 0; which < 2; ++which) {      // one-CTA kernels: per-stage [i][m] tables, W_L^(m*i) with L = Ns * rad
            const KernelEntry<T>* kk = which ? d.kb : d.k;
            const size_t ioff = which ? d.tw_im_off_b : d.tw_im_off;
            if (!kk || kk->kind != KIND_ROW || ioff == (size_t)-1 || (which && ioff == d.tw_im_off)) continue;
            cx<T>* t = reinterpret_cast<cx<T>*>(pl->blob_host.data() + ioff);
            size_t ns = (size_t)kk->rads[0];
            for (int q = 1; q < kk->stages; ++q) {
                const size_t rad = (size_t)kk->rads[q], L = ns * rad;
                for (size_t i = 0; i < rad; ++i)
                    for (size_t m = 0; m < ns; ++m) {
                        double re, im;
                        root_of_unity((uint64_t)(m * i), L, re, im);
                        t[i * ns + m].x = (T)re; t[i * ns + m].y = (T)im;
                    }
                t += L; ns = L;
            }
        }
        for (int which = 0; which < 3; ++which) {
            const KernelEntry<T>* kk = which == 2 ? d.kt : which ? d.kb : d.k;
            const size_t woff = which == 2 ? d.tw_wc_off_t : which ? d.tw_wc_off_b : d.tw_wc_off;
            if (!kk || woff == (size_t)-1 || (which == 1 && woff == d.tw_wc_off)) continue;
            // W_L^(c*m), L = N (2-pass plan), [c][m] layout, m < M = R / first_radix
            const size_t M = R / kk->first_radix;
            cx<T>* wc = reinterpret_cast<cx<T>*>(pl->blob_host.data() + woff);
            for (int c = 0; c < kk->C; ++c)
                for (size_t m = 0; m < M; ++m) {
                    double re, im;
                    root_of_unity((uint64_t)c * m, n, re, im);
                    wc[(size_t)c * M + m].x = (T)re; wc[(size_t)c * M + m].y = (T)im;
                }
        }
    };
    for (int p = 0; p < pl->num_passes; ++p) fill_pass_tables(pl->pass[p]);
    if (pl->alt_row.k) fill_pass_tables(pl->alt_row);
    if (pl->cl) { fill_pass_tables(pl->cl_pass[0]); fill_pass_tables(pl->cl_pass[1]); }
    CUDA_TRY(cudaMalloc(&pl->blob_dev, pl->blob_host.size()));
    CUDA_TRY(cudaMemcpy(pl->blob_dev, pl->blob_host.data(), pl->blob_host.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&pl->ws_free, cudaEventDisableTiming));
    for (int p = 0; p < pl->num_passes; ++p) {
        CUDA_TRY(cudaFuncSetAttribute(pl->pass[p].k->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->pass[p].k->smem));
        if (pl->pass[p].kb)
            CUDA_TRY(cudaFuncSetAttribute(pl->pass[p].kb->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->pass[p].kb->smem));
        if (pl->pass[p].kt)
            CUDA_TRY(cudaFuncSetAttribute(pl->pass[p].kt->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->pass[p].kt->smem));
        if (pl->pass[p].kc)
            CUDA_TRY(cudaFuncSetAttribute(pl->pass[p].kc->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->pass[p].kc->smem));
        if (pl->pass[p].kr)
            CUDA_TRY(cudaFuncSetAttribute(pl->pass[p].kr->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->pass[p].kr->smem));
    }
    if (pl->alt_row.k)
        CUDA_TRY(cudaFuncSetAttribute(pl->alt_row.k->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->alt_row.k->smem));
    if (pl->alt_row.kr)
        CUDA_TRY(cudaFuncSetAttribute(pl->alt_row.kr->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->alt_row.kr->smem));
    for (const PassDesc<T>& d : {std::cref(pl->pass[0]), std::cref(pl->alt_row)}) {      // builds for batched real transforms
        const KernelEntry<T>* real_builds[4] = {d.kc, d.kcb, d.kf, d.kfb};
        for (const KernelEntry<T>* e : real_builds)
            if (e) CUDA_TRY(cudaFuncSetAttribute(e->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->smem));
    }
    if (pl->cl) {
        // usable only if the device can co-schedule at least one cluster of this shape
        cudaError_t ce = cudaFuncSetAttribute(pl->cl->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->cl->smem);
        if (ce == cudaSuccess && pl->cl->K > 8) ce = cudaFuncSetAttribute(pl->cl->fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        int nclusters = 0;
        if (ce == cudaSuccess) {
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3((unsigned)pl->cl->K); cfg.blockDim = dim3((unsigned)pl->cl->NT); cfg.dynamicSmemBytes = pl->cl->smem;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = (unsigned)pl->cl->K; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            ce = cudaOccupancyMaxActiveClusters(&nclusters, pl->cl->fn, &cfg);
        }
        if (ce != cudaSuccess || nclusters < 1) { (void)cudaGetLastError(); pl->cl = nullptr; }
        pl->cl_max_active = nclusters;
    }
    if (pl->num_passes >= 2) {
        CUDA_TRY(cudaMalloc(&pl->ws_re, 2 * n * sizeof(T)));
        pl->ws_im = pl->ws_re + n;
        pl->ws_elems = n;
    }
    if (pl->num_passes == 3) {
        // L2 blocking of passes 2+3: group size in bytes from PHASTFT_L2_GROUP_MB (default 32; 0 disables)
        size_t group_mb = 0;   // measured slower than three full-size passes (launch ramp/tail per group), off by default
        if (const char* env = getenv("PHASTFT_L2_GROUP_MB")) group_mb = (size_t)atoi(env);
        const size_t sub_bytes = (n >> f[0]) * 2 * sizeof(T);
        const long long R1 = 1LL << f[0];
        const long long ctrans = pl->pass[2].k->C;
        long long G = ctrans;
        while (G * 2 <= R1 && (size_t)(G * 2) * sub_bytes <= (group_mb << 20)) G *= 2;
        if (group_mb > 0 && (size_t)G * sub_bytes * 2 <= n * 2 * sizeof(T)) {
            pl->l2_group = G;
            CUDA_TRY(cudaMalloc(&pl->ws2_re, (size_t)G * (n >> f[0]) * sizeof(T)));
            CUDA_TRY(cudaMalloc(&pl->ws2_im, (size_t)G * (n >> f[0]) * sizeof(T)));
        }
    }
    if (pl->num_passes == 2) {
        // PHASTFT_PIPE=0 disables the pipelined launch; PHASTFT_PIPE_LONE=1 also sends lone transforms through it
        int enabled = 0, lone = 0;        // opt-in until it beats two launches (profiles/r02_exp_pipe_kernel_v*.txt)
        if (const char* e = getenv("PHASTFT_PIPE")) enabled = atoi(e);
        if (const char* e = getenv("PHASTFT_PIPE_LONE")) lone = atoi(e);
        int want_mode = 0;                 // PHASTFT_PIPE_TMA=1: the pair with asynchronous tile input, where one exists
        if (const char* e = getenv("PHASTFT_PIPE_TMA")) want_mode = atoi(e) != 0;
        auto find = [&](const KernelEntry<T>* a, const KernelEntry<T>* b) -> const PipeEntry<T>* {
            if (!a || !b) return nullptr;
            const PipeEntry<T>* plain = nullptr;
            for (const auto& pe : pipe_registry<T>())
                if (pe.R1 == a->R && pe.C1 == a->C && pe.NT1 == a->NT && pe.rad1 == a->radices && pe.R2 == b->R && pe.C2 == b->C &&
                    pe.NT2 == b->NT && pe.rad2 == b->radices) {
                    if (pe.mode == want_mode && tensor_map_encoder()) return &pe;
                    if (pe.mode == 0) plain = &pe;
                }
            return plain;
        };
        auto resident = [&](const PipeEntry<T>* pe) -> int {
            int occ = 0, sms = 0;
            if (cudaFuncSetAttribute(pe->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pe->smem) != cudaSuccess ||
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pe->fn, pe->NT, pe->smem) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
            return sms * std::max(occ, 0);
        };
        if (enabled) {
            pl->pipe_b = find(pl->pass[0].kb, pl->pass[1].kb);
            if (pl->pipe_b && (pl->pipe_grid_b = resident(pl->pipe_b)) < 2) pl->pipe_b = nullptr;
            if (lone) {
                pl->pipe_1 = find(pl->pass[0].k, pl->pass[1].k);
                if (pl->pipe_1 && (pl->pipe_grid_1 = resident(pl->pipe_1)) < 2) pl->pipe_1 = nullptr;
            }
        }
    }
    // description
    {
        std::string s = "n=2^" + std::to_string(ln) + (sizeof(T) == 8 ? " f64:" : " f32:");
        if (pl->num_passes == 0) s += " identity";
        for (int p = 0; p < pl->num_passes; ++p) {
            const auto* k = pl->pass[p].k;
            s += std::string(p ? " |" : "") + " " + kind_name(k->kind) + " R=" + std::to_string(k->R) + "(" + k->radices + ") C=" +
                 std::to_string(k->C) + " NT=" + std::to_string(k->NT) + " smem=" + std::to_string(k->smem);
        }
        if (pl->num_passes == 2 && pl->pass[0].kt) {
            s += pl->tma_lone && pl->tma_batch ? " || planar input: " : pl->tma_lone ? " || lone planar: " : " || batches, planar input: ";
            for (int p = 0; p < 2; ++p) {
                const auto* k = pl->pass[p].kt;
                s += std::string(p ? " | " : "") + kind_name(k->kind) + " R=" + std::to_string(k->R) + "(" + k->radices + ") C=" + std::to_string(k->C) +
                     " NT=" + std::to_string(k->NT) + " smem=" + std::to_string(k->smem);
            }
        }
        if (pl->num_passes == 3 && pl->pass[1].kt) {
            const auto* k = pl->pass[1].kt;
            s += " [middle pass by TMA: COL R=" + std::to_string(k->R) + "(" + k->radices + ") C=" + std::to_string(k->C) + " NT=" + std::to_string(k->NT) + "]";
        }
        if (pl->num_passes == 3 && pl->pass[0].kt && pl->pass[2].kt) s += " [end passes by TMA / bulk copies, C=" + std::to_string(pl->pass[0].kt->C) + "]";
        if (pl->l2_group) s += " | L2-blocked tail: " + std::to_string(pl->l2_group) + " k1/group";
        bool differs = false;
        for (int p = 0; p < pl->num_passes; ++p) differs |= pl->pass[p].kb && pl->pass[p].kb != pl->pass[p].k;
        if (differs) {
            s += " || batches:";
            for (int p = 0; p < pl->num_passes; ++p) {
                const auto* k = pl->pass[p].kb;
                s += std::string(p ? " |" : "") + " " + kind_name(k->kind) + " R=" + std::to_string(k->R) + "(" + k->radices + ") C=" +
                     std::to_string(k->C) + " NT=" + std::to_string(k->NT);
            }
        }
        if (pl->num_passes >= 2) s += pl->ws_il == 1 ? " [interleaved intermediates]" : pl->ws_il == 0 ? " [planar intermediates]" : "";
        if (pl->pipe_b) s += std::string(" [batches: one pipelined launch, ") + (pl->pipe_b->mode ? "TMA / bulk tile input, " : "") + std::to_string(pl->pipe_grid_b) + " resident CTAs, L2 ring]";
        if (pl->pipe_1) s += " [lone: one pipelined launch, " + std::to_string(pl->pipe_grid_1) + " resident CTAs]";
        if (pl->alt_row.k) s += " || batches: ROW R=" + std::to_string(pl->alt_row.k->R) + "(" + pl->alt_row.k->radices + ")";
        if ((pl->num_passes == 1 && pl->pass[0].kr) || pl->alt_row.kr) s += " [contiguous planar batches: tile in / out by cp.async.bulk]";
        if (pl->cl)
            s += " || batches >= " + std::to_string(pl->cl_min_batch) + ": CLUSTER K=" + std::to_string(pl->cl->K) + " NT=" + std::to_string(pl->cl->NT) +
                 " " + std::to_string(pl->cl->k1.R) + "(" + pl->cl->k1.radices + ") x " + std::to_string(pl->cl->k2.R) + "(" + pl->cl->k2.radices +
                 ") smem=" + std::to_string(pl->cl->smem) + (pl->cl->variant ? ",v" + std::to_string(pl->cl->variant) : std::string()) +
                 " resident clusters=" + std::to_string(pl->cl_max_active);
        pl->description = s;
    }
    {
        BlobHeader h;
        memset(&h, 0, sizeof(h));
        h.magic = BLOB_MAGIC; h.bytes = pl->blob_host.size(); h.n = n;
        h.precision_bits = 8 * sizeof(T); h.num_passes = (uint32_t)pl->num_passes;
        h.layout_sig = fnv1a(pl->description);
        memcpy(pl->blob_host.data(), &h, sizeof(h));
        CUDA_TRY(cudaMemcpy(pl->blob_dev, pl->blob_host.data(), BLOB_HEADER_BYTES, cudaMemcpyHostToDevice));
    }
    *out = pl.release();
    return PHASTFT_OK;
}

// =================================================================================================
// execution
// =================================================================================================

template <typename T>
struct Io {
    const T* in_re; const T* in_im;
    T* out_re; T* out_im;
    long long in_bstride, out_bstride;
    int in_il, out_il;   // 0 planar, 1 interleaved, 2 interleaved with re/im swapped
    // c2r: in_re / in_im are the half-spectrum's N/2 + 1 bins and the first pass builds its input from them while loading
    // (PassDesc::kc / kcb); pre_log2half = log2(N/2), 0 = off
    Tw2 pre_tw2 = {nullptr, nullptr, 0};
    int pre_log2half = 0;
    // batched r2c: the one-CTA kernel untangles its result on store (PassDesc::kf / kfb; W_N in pre_tw2).  Only the one-CTA
    // path of run_c2c takes it (r2c_batch_dev decides).
    int r2c_out = 0;
};

// W_(2 R1)^i, i < R1: the per-launch factors of the c2r pre-processing on load (PassParams::pre_wc), R1 = the kernel's first radix
inline const double2* c2r_pre_wc(int r1) {
    static const std::vector<std::vector<double2>> tabs = [] {
        std::vector<std::vector<double2>> t(6);
        for (int l = 0; l < 6; ++l) {
            t[l].assign(32, make_double2(0.0, 0.0));
            for (uint64_t i = 0; i < (1u << l); ++i) root_of_unity(i, 2u << l, t[l][i].x, t[l][i].y);
        }
        return t;
    }();
    return (r1 >= 1 && r1 <= 32 && is_pow2((size_t)r1)) ? tabs[ilog2((size_t)r1)].data() : nullptr;
}

template <typename T>
bool many_transforms(const Plan<T>& pl, const PassDesc<T>& d, size_t batch) {
    return d.kb != nullptr && batch > 1 && (batch << pl.log2n) >= (size_t(1) << 21);
}
// The MODE_R2C_OUT kernel a one-CTA pass launches for `batch` transforms (NULL: none), and whether that is kb's build.
template <typename T>
const KernelEntry<T>* r2c_out_kernel(const Plan<T>& pl, const PassDesc<T>& d, size_t batch, bool& many) {
    many = many_transforms(pl, d, batch) && d.kfb != nullptr;
    return many ? d.kfb : d.kf;
}

// k1_lo / k1_cnt (multi-pass plans, batch == 1): restrict a pass AFTER the first to the sub-transforms
// whose first-pass output digit k1 lies in [k1_lo, k1_lo + k1_cnt) -- the unit of L2 blocking.
template <typename T>
int32_t prepare_pass(const Plan<T>& pl, int p, const PassParams<T>& base, size_t batch, long long k1_lo, long long k1_cnt,
                     PassParams<T>& prm_out, const KernelEntry<T>*& k_out, unsigned long long& blocks_out, bool use_kt = false);

// use_kt: launch the pass's asynchronous-input kernel (PassDesc::kt); the caller has checked its preconditions
// (pass 0: planar 16-byte-aligned input; last pass: interleaved workspace).
template <typename T>
int32_t launch_pass(const Plan<T>& pl, int p, const PassParams<T>& base, size_t batch, cudaStream_t stream,
                    long long k1_lo = 0, long long k1_cnt = -1, bool use_kt = false) {
    PassParams<T> prm;
    const KernelEntry<T>* k = nullptr;
    unsigned long long blocks = 0;
    int32_t st = prepare_pass(pl, p, base, batch, k1_lo, k1_cnt, prm, k, blocks, use_kt);
    if (st) return st;
    if (k->mode == MODE_TMA_IN) {
        const size_t B = size_t(1) << prm.log2B, A = size_t(1) << prm.log2A;
        const unsigned box_rows = (unsigned)std::min(k->R, 256);
        bool ok;
        if (prm.in_interleaved) {
            // the interleaved workspace as an array of T: rows of 2B values, A * batch blocks of R rows (batch stride = A * R * B pairs)
            if (batch > 1 && (size_t)prm.in_bstride != A * (size_t)k->R * B) return fail(PHASTFT_ERR_INVALID_ARG, "TMA middle pass: the workspace must be dense");
            ok = encode_tile_map<T>(&prm.tmap_re, prm.in_re, 2 * B, (size_t)k->R, 2 * B, A * batch, (size_t)k->R * 2 * B, 2u * (unsigned)k->C, box_rows);
        } else {
            if (A != 1) return fail(PHASTFT_ERR_INVALID_ARG, "TMA planar input: first pass only");
            ok = encode_tile_map<T>(&prm.tmap_re, prm.in_re, B, (size_t)k->R, B, batch, (size_t)prm.in_bstride, (unsigned)k->C, box_rows) &&
                 encode_tile_map<T>(&prm.tmap_im, prm.in_im, B, (size_t)k->R, B, batch, (size_t)prm.in_bstride, (unsigned)k->C, box_rows);
        }
        if (!ok) return fail(PHASTFT_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    }
    void* args[] = {&prm};
    // Programmatic dependent launch: measured no gain with 128 KB tiles (the next grid cannot become resident early), -10%
    // at 2^24+, and slower too with the 64 KB asynchronous-input tiles (profiles/r02_exp_tma1.txt).  PHASTFT_PDL=1 enables it.
    static const int pdl_env = [] { const char* e = getenv("PHASTFT_PDL"); return e ? (atoi(e) != 0 ? 1 : 0) : -1; }();
    const bool use_pdl = pdl_env > 0;     // off by default: measured slower with and without the asynchronous-input kernels
    if (use_pdl) {
        // Programmatic dependent launch: back-to-back passes overlap the next grid's launch and prologue
        // with the previous grid's tail (the kernel waits with griddepcontrol.wait before its first access).
        prm.pdl = 1;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3((unsigned)blocks); cfg.blockDim = dim3(k->NT); cfg.dynamicSmemBytes = k->smem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        CUDA_TRY(cudaLaunchKernelExC(&cfg, k->fn, args));
    } else {
        CUDA_TRY(cudaLaunchKernel(k->fn, dim3((unsigned)blocks), dim3(k->NT), args, k->smem, stream));
    }
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return PHASTFT_OK;
}

template <typename T>
int32_t prepare_pass_desc(const Plan<T>& pl, const PassDesc<T>& d, int p, const PassParams<T>& base, size_t batch, long long k1_lo,
                          long long k1_cnt, PassParams<T>& prm_out, const KernelEntry<T>*& k_out, unsigned long long& blocks_out,
                          bool use_kt = false);

template <typename T>
int32_t prepare_pass(const Plan<T>& pl, int p, const PassParams<T>& base, size_t batch, long long k1_lo, long long k1_cnt,
                     PassParams<T>& prm_out, const KernelEntry<T>*& k_out, unsigned long long& blocks_out, bool use_kt) {
    const PassDesc<T>& d = (p == ALT_ROW_PASS) ? pl.alt_row : pl.pass[p];
    return prepare_pass_desc(pl, d, p, base, batch, k1_lo, k1_cnt, prm_out, k_out, blocks_out, use_kt);
}

template <typename T>
int32_t prepare_pass_desc(const Plan<T>& pl, const PassDesc<T>& d, int p, const PassParams<T>& base, size_t batch, long long k1_lo,
                          long long k1_cnt, PassParams<T>& prm_out, const KernelEntry<T>*& k_out, unsigned long long& blocks_out,
                          bool use_kt) {
    bool many = !use_kt && many_transforms(pl, d, batch);
    const KernelEntry<T>* k_r2c = base.r2c_out ? r2c_out_kernel(pl, d, batch, many) : nullptr;
    const KernelEntry<T>* k = use_kt ? d.kt : many ? d.kb : d.k;
    // one-CTA batch kernel with bulk tile input / output: planar arrays, transforms back to back, 16-byte-aligned planes
    if (many && d.kr && k == d.kb && base.in_interleaved == 0 && base.out_interleaved == 0 && base.in_bstride == (long long)pl.n &&
        base.out_bstride == (long long)pl.n &&
        ((reinterpret_cast<uintptr_t>(base.in_re) | reinterpret_cast<uintptr_t>(base.in_im) | reinterpret_cast<uintptr_t>(base.out_re) |
          reinterpret_cast<uintptr_t>(base.out_im)) & 15) == 0)
        k = d.kr;
    if (base.pre_log2half) {
        const KernelEntry<T>* kc = many ? d.kcb : d.kc;
        if (!kc && k->kind == KIND_COL) kc = d.kcb;    // a first COL pass reads no table that depends on its tile
        if (p > 0 || use_kt || !kc) return fail(PHASTFT_ERR_INVALID_ARG, "c2r pre-processing on load: first pass or one-CTA kernel with a MODE_C2R_IN build only");
        k = kc;
    } else if (base.r2c_out) {
        if (use_kt || !k_r2c) return fail(PHASTFT_ERR_INVALID_ARG, "r2c untangle on store: one-CTA kernel with a MODE_R2C_OUT build only");
        k = k_r2c;
    }
    PassParams<T> prm = base;
    if (base.pre_log2half) {
        const double2* wc = c2r_pre_wc(k->first_radix);
        if (!wc) return fail(PHASTFT_ERR_INVALID_ARG, "c2r pre-processing on load: first radix > 32");
        memcpy(prm.pre_wc, wc, sizeof(prm.pre_wc));
    }
    prm.batch = (int)batch;
    prm.log2A = d.log2A; prm.log2B = d.log2B; prm.log2R1 = d.log2R1; prm.log2Rprev = d.log2Rprev;
    prm.has_tw = d.has_tw; prm.tw_shift = d.tw_shift;
    prm.tw2.hi = reinterpret_cast<const double2*>(pl.blob_dev + pl.hi_off);
    prm.tw2.lo = reinterpret_cast<const double2*>(pl.blob_dev + pl.lo_off);
    prm.tw2.lo_bits = pl.lo_bits;
    prm.tw_stage = reinterpret_cast<const cx<T>*>(pl.blob_dev + d.tw_stage_off);
    const size_t wc_off = use_kt ? d.tw_wc_off_t : many ? d.tw_wc_off_b : d.tw_wc_off;
    const size_t im_off = many ? d.tw_im_off_b : d.tw_im_off;
    prm.tw_stage_im = im_off == (size_t)-1 ? nullptr : reinterpret_cast<const cx<T>*>(pl.blob_dev + im_off);
    prm.tw_wc = wc_off == (size_t)-1 ? nullptr : reinterpret_cast<const cx<T>*>(pl.blob_dev + wc_off);
    unsigned long long blocks;
    prm.blk_offset = 0; prm.kt_base = 0; prm.log2_ktn = d.log2R1 - ilog2(k->C);
    if (k->kind == KIND_ROW) blocks = (batch + k->C - 1) / k->C;
    else blocks = (unsigned long long)batch * (pl.n >> d.log2R) / k->C;
    if (k1_cnt >= 0 && p > 0) {
        const unsigned long long tiles_per_k1 = ((pl.n >> d.log2R) / k->C) >> d.log2R1;   // COL: (A/R1) * B/C
        if (k->kind == KIND_COL) {
            prm.blk_offset = (int)(k1_lo * tiles_per_k1);
            blocks = k1_cnt * tiles_per_k1;
        } else {
            prm.kt_base = (int)(k1_lo / k->C);
            prm.log2_ktn = ilog2((size_t)(k1_cnt / k->C));
            blocks = ((pl.n >> d.log2R) >> d.log2R1) * (k1_cnt / k->C);                     // rest_n * chunk tiles
        }
    }
    if (blocks == 0 || blocks > 0x7fffffffULL) return fail(PHASTFT_ERR_INVALID_ARG, "grid too large");
    prm_out = prm; k_out = k; blocks_out = blocks;
    return PHASTFT_OK;
}

// A batch is processed in chunks so the workspace stays bounded.  Measured on B200 (profiles/r01_tune12*.txt):
// keeping a chunk's intermediate L2-resident (48 MiB chunks) is SLOWER than few large launches --
// 4096 x 2^16 f32: 1.88 ms at 48 MiB, 1.61 ms at 192 MiB, 1.50 ms unchunked -- so the default chunk is
// as large as the workspace cap allows (PHASTFT_L2_CHUNK_MB overrides).
constexpr size_t L2_CHUNK_BYTES_DEFAULT = size_t(4) << 30;
inline size_t l2_chunk_bytes() {
    static const size_t v = [] {
        if (const char* env = getenv("PHASTFT_L2_CHUNK_MB")) { long mb = atol(env); if (mb > 0) return (size_t)mb << 20; }
        return L2_CHUNK_BYTES_DEFAULT;
    }();
    return v;
}

// Ring of workspace slots of the pipelined two-pass launch: the largest power-of-two number of transforms whose
// intermediates fit PHASTFT_PIPE_RING_MB (default 32 MiB: tools/dsmem_bench.cu `ring` keeps 5.4 TB/s up to 32-48 MiB and
// falls to the HBM round trip's 3.4 TB/s at 96 MiB), at least 1.
inline size_t pipe_ring_bytes() {
    static const size_t v = [] {
        long mb = 32;
        if (const char* env = getenv("PHASTFT_PIPE_RING_MB")) mb = atol(env);
        return (size_t)std::max(1L, mb) << 20;
    }();
    return v;
}
template <typename T>
size_t pipe_ring_transforms(const Plan<T>& pl, size_t batch) {
    const size_t bytes_per = pl.n * 2 * sizeof(T);
    size_t ring = 1;
    while (ring * 2 * bytes_per <= pipe_ring_bytes() && ring * 2 <= batch) ring *= 2;
    if (ring < 2 && batch > 1) ring = 2;            // two slots at least: pass 1 of b+1 beside pass 2 of b
    return ring;
}
// caller holds pl.mu
template <typename T>
int32_t grow_workspace(const Plan<T>& pl, size_t transforms, cudaStream_t stream) {
    if (pl.ws_elems >= transforms * pl.n) return PHASTFT_OK;
    if (stream) CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaDeviceSynchronize());
    if (pl.ws_re) cudaFree(pl.ws_re);
    pl.ws_re = pl.ws_im = nullptr; pl.ws_elems = 0;
    CUDA_TRY(cudaMalloc(&pl.ws_re, 2 * transforms * pl.n * sizeof(T)));
    pl.ws_im = pl.ws_re + transforms * pl.n;
    pl.ws_elems = transforms * pl.n;
    return PHASTFT_OK;
}

// `pipe`: calls may take the pipelined launch (a ring of transforms); false sizes the workspace for the chunked path, which
// batched c2r (no pre-processing build of the pipelined pair) always takes
template <typename T>
int32_t plan_reserve(const Plan<T>* pl, size_t batch, bool pipe = true) {
    if (!pl) return fail(PHASTFT_ERR_INVALID_ARG, "plan == NULL");
    if (pl->num_passes < 2 || batch <= 1) return PHASTFT_OK;       // one-CTA plans have no workspace
    DeviceGuard g(pl->device);
    std::lock_guard<std::mutex> lock(pl->mu);
    const size_t bytes_per = pl->n * 2 * sizeof(T);
    size_t chunk = std::max<size_t>(1, l2_chunk_bytes() / bytes_per);
    chunk = std::min(chunk, batch);
    if (pipe && pl->pipe_b && (batch << pl->log2n) >= (size_t(1) << 21)) chunk = pipe_ring_transforms(*pl, batch);
    return grow_workspace(*pl, chunk, nullptr);
}

// `pass_events` (profiling aid, bench.py roofline): if non-NULL, num_passes+1 events are recorded
// around the passes of the FIRST chunk.
template <typename T>
int32_t run_c2c(const Plan<T>& pl, const Io<T>& io, size_t batch, T scale, cudaStream_t stream,
                cudaEvent_t* pass_events = nullptr) {
    if (batch == 0) return PHASTFT_OK;
    PassParams<T> prm;
    memset(&prm, 0, sizeof(prm));
    if (pl.num_passes == 0) {
        // N == 1: the transform is the identity (the reference runs zero stages, dit.rs:44-65).
        if (io.in_re != io.out_re || io.in_il != io.out_il || scale != T(1))
            return fail(PHASTFT_ERR_INVALID_ARG, "N == 1 supports only the in-place unscaled form");
        return PHASTFT_OK;
    }
    const bool use_alt_row = pl.alt_row.k != nullptr && batch >= pl.alt_row_min_batch;
    if (pl.num_passes == 1 || use_alt_row) {
        const int which = use_alt_row ? ALT_ROW_PASS : 0;
        size_t done = 0;
        const size_t max_chunk = (size_t)1 << 24;
        while (done < batch) {
            size_t nb = std::min(batch - done, max_chunk);
            prm.in_re = io.in_re + (io.in_il ? 2 : 1) * done * io.in_bstride;
            prm.in_im = io.in_im ? io.in_im + done * io.in_bstride : nullptr;
            prm.out_re = io.out_re + (io.out_il ? 2 : 1) * done * io.out_bstride;
            prm.out_im = io.out_im ? io.out_im + done * io.out_bstride : nullptr;
            prm.in_bstride = io.in_bstride; prm.out_bstride = io.out_bstride;
            prm.in_interleaved = io.in_il; prm.out_interleaved = io.out_il;
            prm.scale = scale;
            prm.pre_tw2 = io.pre_tw2; prm.pre_log2half = io.pre_log2half; prm.r2c_out = io.r2c_out;
            if (pass_events && done == 0) CUDA_TRY(cudaEventRecord(pass_events[0], stream));
            int32_t st = launch_pass(pl, which, prm, nb, stream);
            if (st) return st;
            if (pass_events && done == 0) {
                CUDA_TRY(cudaEventRecord(pass_events[1], stream));
                for (int q = 2; q <= pl.num_passes; ++q) CUDA_TRY(cudaEventRecord(pass_events[q], stream));
            }
            done += nb;
        }
        return PHASTFT_OK;
    }
    if (io.r2c_out) return fail(PHASTFT_ERR_INVALID_ARG, "r2c untangle on store: one-CTA plans only");
    // ---- both passes in one cluster launch: no workspace, HBM sees the batch once in and once out ----------------
    // (its first pass has no c2r pre-processing build)
    if (pl.cl && batch >= pl.cl_min_batch && !io.pre_log2half) {
        const size_t max_chunk = (size_t(1) << 30) / (size_t)pl.cl->K;        // grid = transforms x K CTAs
        for (size_t done = 0; done < batch; done += max_chunk) {
            const size_t nb = std::min(batch - done, max_chunk);
            PassParams<T> b1, b2, p1, p2;
            memset(&b1, 0, sizeof(b1)); memset(&b2, 0, sizeof(b2));
            b1.scale = T(1);
            b1.in_re = io.in_re + (io.in_il ? 2 : 1) * done * io.in_bstride;
            b1.in_im = io.in_im ? io.in_im + done * io.in_bstride : nullptr;
            b1.in_bstride = io.in_bstride; b1.in_interleaved = io.in_il;
            b1.xch_log2P2 = pl.cl_pass[1].log2R;
            b1.xch_log2CB = ilog2((size_t)pl.cl->k2.C);
            b2.out_re = io.out_re + (io.out_il ? 2 : 1) * done * io.out_bstride;
            b2.out_im = io.out_im ? io.out_im + done * io.out_bstride : nullptr;
            b2.out_bstride = io.out_bstride; b2.out_interleaved = io.out_il;
            b2.scale = scale;
            const KernelEntry<T>* k1 = nullptr; const KernelEntry<T>* k2 = nullptr;
            unsigned long long t1 = 0, t2 = 0;
            int32_t st = prepare_pass_desc(pl, pl.cl_pass[0], 0, b1, nb, 0, -1, p1, k1, t1);
            if (!st) st = prepare_pass_desc(pl, pl.cl_pass[1], 1, b2, nb, 0, -1, p2, k2, t2);
            if (st) return st;
            if (t1 != t2 || t1 != (unsigned long long)nb * pl.cl->K) return fail(PHASTFT_ERR_INVALID_ARG, "cluster plan: tile count mismatch");
            void* args[] = {&p1, &p2};
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3((unsigned)t1); cfg.blockDim = dim3((unsigned)pl.cl->NT); cfg.dynamicSmemBytes = pl.cl->smem; cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = (unsigned)pl.cl->K; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            if (pass_events && done == 0) CUDA_TRY(cudaEventRecord(pass_events[0], stream));
            CUDA_TRY(cudaLaunchKernelExC(&cfg, pl.cl->fn, args));
            g_launches.fetch_add(1, std::memory_order_relaxed);
            if (pass_events && done == 0)
                for (int q = 1; q <= pl.num_passes; ++q) CUDA_TRY(cudaEventRecord(pass_events[q], stream));
        }
        return PHASTFT_OK;
    }
    // multi-pass: in -> ws (COL) [-> ws (COL)] -> out (TRANS), batch processed in L2-sized chunks
    std::lock_guard<std::mutex> lock(pl.mu);
    const size_t bytes_per = pl.n * 2 * sizeof(T);
    size_t chunk = std::max<size_t>(1, l2_chunk_bytes() / bytes_per);
    chunk = std::min(chunk, batch);
    if (pl.num_passes == 3 && pl.ws2_re != nullptr) chunk = 1;
    // pipelined two-pass launch (see fft_pipe2_kernel): the workspace is a ring of transforms instead of the whole chunk
    const PipeEntry<T>* pipe = nullptr;
    if (pl.num_passes == 2 && !pass_events) {
        // (no c2r pre-processing build of its passes; its TMA tile input reads planar data only)
        if (batch > 1 && (batch << pl.log2n) >= (size_t(1) << 21) && !io.pre_log2half && !(pl.pipe_b && pl.pipe_b->mode == 1 && io.in_il != 0))
            pipe = pl.pipe_b;
        else if (batch == 1 && io.in_il == 0 && io.out_il == 0 && !io.pre_log2half) pipe = pl.pipe_1;
    }
    size_t ws_need = chunk;
    const size_t ring = pipe ? pipe_ring_transforms(pl, batch) : 0;
    if (pipe) ws_need = ring;
    // Workspace reuse is ordered by the stream itself when consecutive calls use the same stream;
    // a call on a different stream first waits for the previous user.  While `stream` is being
    // captured into a CUDA graph the cross-stream bookkeeping is skipped (the graph's owner orders
    // replays against other users of the plan).
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    CUDA_TRY(cudaStreamIsCapturing(stream, &cap));
    const bool capturing = cap != cudaStreamCaptureStatusNone;
    if (pl.ws_elems < ws_need * pl.n || (pipe && pl.pipe_state_batch < batch)) {
        // The plan is created with room for one transform; the first batched call grows it (synchronising).
        // phastft_plan_dit_*_reserve(batch) does this ahead of time; inside a graph capture growing is an error.
        if (capturing)
            return fail(PHASTFT_ERR_INVALID_ARG, "the plan's workspace is too small for this batch and the stream is being captured: "
                                                 "call phastft_plan_dit_*_reserve(batch) before capturing");
        int32_t st = grow_workspace(pl, ws_need, stream);
        if (st) return st;
        if (pipe && pl.pipe_state_batch < batch) {
            CUDA_TRY(cudaStreamSynchronize(stream));
            if (pl.pipe_state) cudaFree(pl.pipe_state);
            pl.pipe_state = nullptr; pl.pipe_state_batch = 0;
            const size_t cap = std::max<size_t>(batch, 4096);
            CUDA_TRY(cudaMalloc(&pl.pipe_state, 64 + 2 * cap * sizeof(unsigned)));
            pl.pipe_state_batch = cap;
        }
    }
    if (!capturing && pl.ws_last_stream != stream && pl.ws_used) CUDA_TRY(cudaStreamWaitEvent(stream, pl.ws_free, 0));
    const int P = pl.num_passes;
    if (pipe) {
        const bool lone = batch == 1;
        const int il_p = lone ? (pl.ws_il >= 0 ? pl.ws_il : 0) : (pl.ws_il >= 0 ? pl.ws_il : 1);
        PassParams<T> b1, b2, p1, p2;
        memset(&b1, 0, sizeof(b1)); memset(&b2, 0, sizeof(b2));
        b1.scale = T(1);
        b1.in_re = io.in_re; b1.in_im = io.in_im; b1.in_bstride = io.in_bstride; b1.in_interleaved = io.in_il;
        b1.out_re = pl.ws_re; b1.out_im = pl.ws_re + ring * pl.n; b1.out_bstride = (long long)pl.n; b1.out_interleaved = il_p;
        b1.out_ring = (int)ring;
        b2.in_re = pl.ws_re; b2.in_im = pl.ws_re + ring * pl.n; b2.in_bstride = (long long)pl.n; b2.in_interleaved = il_p;
        b2.in_ring = (int)ring;
        b2.out_re = io.out_re; b2.out_im = io.out_im; b2.out_bstride = io.out_bstride; b2.out_interleaved = io.out_il;
        b2.scale = scale;
        const KernelEntry<T>* k1 = nullptr; const KernelEntry<T>* k2 = nullptr;
        unsigned long long t1 = 0, t2 = 0;
        // descriptors with the batch flavour of each pass's kernel (prepare_pass picks kb for many-transform calls)
        int32_t st = prepare_pass(pl, 0, b1, batch, 0, -1, p1, k1, t1);
        if (!st) st = prepare_pass(pl, 1, b2, batch, 0, -1, p2, k2, t2);
        if (st) return st;
        if (k1->R != pipe->R1 || k1->C != pipe->C1 || k2->R != pipe->R2 || k2->C != pipe->C2)
            return fail(PHASTFT_ERR_INVALID_ARG, "pipelined launch: kernel pair does not match the plan");
        if (pipe->mode == 1) {
            const size_t B = size_t(1) << p1.log2B;
            const bool ok_align = io.in_il == 0 && il_p == 1 && ((reinterpret_cast<uintptr_t>(io.in_re) | reinterpret_cast<uintptr_t>(io.in_im)) & 15) == 0 &&
                                  ((size_t)io.in_bstride * sizeof(T)) % 16 == 0;
            if (!ok_align) return fail(PHASTFT_ERR_INVALID_ARG, "pipelined launch with TMA input needs planar 16-byte-aligned input (unset PHASTFT_PIPE_TMA)");
            const unsigned box_rows = (unsigned)std::min(k1->R, 256);
            if (!encode_tile_map<T>(&p1.tmap_re, p1.in_re, B, (size_t)k1->R, B, batch, (size_t)p1.in_bstride, (unsigned)k1->C, box_rows) ||
                !encode_tile_map<T>(&p1.tmap_im, p1.in_im, B, (size_t)k1->R, B, batch, (size_t)p1.in_bstride, (unsigned)k1->C, box_rows))
                return fail(PHASTFT_ERR_CUDA, "cuTensorMapEncodeTiled failed");
        }
        PipeCtl ctl;
        ctl.ticket = reinterpret_cast<unsigned*>(pl.pipe_state);
        ctl.done1 = reinterpret_cast<unsigned*>(pl.pipe_state + 64);
        ctl.done2 = ctl.done1 + pl.pipe_state_batch;
        ctl.tiles1 = (unsigned)(t1 / batch); ctl.tiles2 = (unsigned)(t2 / batch);
        ctl.batch = (unsigned)batch; ctl.ring = (unsigned)ring;
        ctl.delay = lone ? 1u : (unsigned)std::max<size_t>(1, ring / 2);
        static const int discard_env = [] { const char* e = getenv("PHASTFT_PIPE_DISCARD"); return e ? atoi(e) : 1; }();
        ctl.discard = (discard_env && il_p == 1 && !lone) ? 1 : 0;
        CUDA_TRY(cudaMemsetAsync(pl.pipe_state, 0, 64 + 2 * pl.pipe_state_batch * sizeof(unsigned), stream));
        const unsigned long long items = (unsigned long long)(batch + ctl.delay) * (ctl.tiles1 + ctl.tiles2);
        if (items > 0x7fffffffULL) return fail(PHASTFT_ERR_INVALID_ARG, "grid too large");
        const unsigned grid = (unsigned)items;                               // one CTA per work item (a ticket decides which)
        void* args[] = {&p1, &p2, &ctl};
        CUDA_TRY(cudaLaunchKernel(pipe->fn, dim3(grid), dim3(pipe->NT), args, pipe->smem, stream));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (!capturing) {
            CUDA_TRY(cudaEventRecord(pl.ws_free, stream));
            pl.ws_last_stream = stream;
            pl.ws_used = true;
        }
        return PHASTFT_OK;
    }
    // ---- 3-pass plans: pass 1 streams the whole signal HBM -> HBM; passes 2+3 then run per group of
    // G consecutive k1 values (G * N/R1 elements ~ tens of MiB): pass 2 writes its result into a small
    // reused scratch that stays L2-resident and pass 3 reads it back from L2, so the tail costs one
    // HBM read + one HBM write instead of two of each.
    if (P == 3 && pl.ws2_re != nullptr) {
        const long long R1 = 1LL << pl.pass[0].log2R;
        const long long sub = (long long)(pl.n >> pl.pass[0].log2R);    // elements per k1
        const long long G = pl.l2_group;
        for (size_t b = 0; b < batch; ++b) {
            memset(&prm, 0, sizeof(prm));
            prm.scale = T(1);
            prm.in_re = io.in_re + (io.in_il ? 2 : 1) * b * io.in_bstride;
            prm.in_im = io.in_im ? io.in_im + b * io.in_bstride : nullptr;
            prm.in_bstride = io.in_bstride; prm.in_interleaved = io.in_il;
            prm.pre_tw2 = io.pre_tw2; prm.pre_log2half = io.pre_log2half;
            prm.out_re = pl.ws_re; prm.out_im = pl.ws_im; prm.out_bstride = (long long)pl.n;
            if (pass_events && b == 0) CUDA_TRY(cudaEventRecord(pass_events[0], stream));
            int32_t st = launch_pass(pl, 0, prm, 1, stream);
            if (st) return st;
            if (pass_events && b == 0) CUDA_TRY(cudaEventRecord(pass_events[1], stream));
            for (long long k1 = 0; k1 < R1; k1 += G) {
                memset(&prm, 0, sizeof(prm));
                prm.scale = T(1);
                prm.in_re = pl.ws_re; prm.in_im = pl.ws_im; prm.in_bstride = (long long)pl.n;
                prm.out_re = pl.ws2_re - k1 * sub; prm.out_im = pl.ws2_im - k1 * sub; prm.out_bstride = (long long)pl.n;
                st = launch_pass(pl, 1, prm, 1, stream, k1, G);
                if (st) return st;
                memset(&prm, 0, sizeof(prm));
                prm.in_re = pl.ws2_re - k1 * sub; prm.in_im = pl.ws2_im - k1 * sub; prm.in_bstride = (long long)pl.n;
                prm.out_re = io.out_re + (io.out_il ? 2 : 1) * b * io.out_bstride;
                prm.out_im = io.out_im ? io.out_im + b * io.out_bstride : nullptr;
                prm.out_bstride = io.out_bstride; prm.out_interleaved = io.out_il;
                prm.scale = scale;
                st = launch_pass(pl, 2, prm, 1, stream, k1, G);
                if (st) return st;
            }
            if (pass_events && b == 0) { CUDA_TRY(cudaEventRecord(pass_events[2], stream)); CUDA_TRY(cudaEventRecord(pass_events[3], stream)); }
        }
        if (!capturing) {
            CUDA_TRY(cudaEventRecord(pl.ws_free, stream));
            pl.ws_last_stream = stream;
            pl.ws_used = true;
        }
        return PHASTFT_OK;
    }
    const bool many_call = batch > 1 && (batch << pl.log2n) >= (size_t(1) << 21);
    // asynchronous-input kernels: planar 16-byte-aligned input whose batch stride keeps the alignment, interleaved intermediates
    // batches: from 32 MiB of signal per array (2^22 f64 / 2^23 f32 points) -- below that the grid is about one wave and the pair
    // measures equal or up to 5 % slower (profiles/r02_exp_tma_batch.txt, last block)
    const bool tma_many = many_call && pl.tma_batch && (batch << pl.log2n) * sizeof(T) >= (size_t(32) << 20);
    const bool tma = P == 2 && pl.pass[0].kt && pl.pass[1].kt && (many_call ? tma_many : pl.tma_lone) && io.in_il == 0 && pl.ws_il != 0 && !io.pre_log2half &&
                     ((reinterpret_cast<uintptr_t>(io.in_re) | reinterpret_cast<uintptr_t>(io.in_im)) & 15) == 0 &&
                     (batch == 1 || ((size_t)io.in_bstride * sizeof(T)) % 16 == 0);
    const int il = tma ? 1 : pl.ws_il >= 0 ? pl.ws_il : ((P == 3 || many_call) ? 1 : 0);
    for (size_t done = 0; done < batch; done += chunk) {
        const size_t nb = std::min(chunk, batch - done);
        for (int p = 0; p < P; ++p) {
            memset(&prm, 0, sizeof(prm));
            prm.scale = T(1);
            if (p == 0) {
                prm.in_re = io.in_re + (io.in_il ? 2 : 1) * done * io.in_bstride;
                prm.in_im = io.in_im ? io.in_im + done * io.in_bstride : nullptr;
                prm.in_bstride = io.in_bstride;
                prm.in_interleaved = io.in_il;
                prm.pre_tw2 = io.pre_tw2; prm.pre_log2half = io.pre_log2half;
            } else {
                prm.in_re = pl.ws_re; prm.in_im = pl.ws_im; prm.in_bstride = (long long)pl.n;
                prm.in_interleaved = il;
            }
            if (p == P - 1) {
                prm.out_re = io.out_re + (io.out_il ? 2 : 1) * done * io.out_bstride;
                prm.out_im = io.out_im ? io.out_im + done * io.out_bstride : nullptr;
                prm.out_bstride = io.out_bstride;
                prm.out_interleaved = io.out_il;
                prm.scale = scale;
            } else {
                prm.out_re = pl.ws_re; prm.out_im = pl.ws_im; prm.out_bstride = (long long)pl.n;
                prm.out_interleaved = il;
            }
            if (pass_events && done == 0 && p == 0) CUDA_TRY(cudaEventRecord(pass_events[0], stream));
            bool tma3 = false;
            if (P == 3 && pl.pass[p].kt != nullptr && il == 1 && nb == 1) {
                if (p == 0) tma3 = io.in_il == 0 && !io.pre_log2half && ((reinterpret_cast<uintptr_t>(prm.in_re) | reinterpret_cast<uintptr_t>(prm.in_im)) & 15) == 0;
                else tma3 = true;
            }
            int32_t st = launch_pass(pl, p, prm, nb, stream, 0, -1, tma || tma3);
            if (st) return st;
            if (pass_events && done == 0) CUDA_TRY(cudaEventRecord(pass_events[p + 1], stream));
        }
    }
    if (!capturing) {
        CUDA_TRY(cudaEventRecord(pl.ws_free, stream));
        pl.ws_last_stream = stream;
        pl.ws_used = true;
    }
    return PHASTFT_OK;
}

template <typename T>
int32_t check_c2c_args(const Plan<T>* pl, size_t len_re, size_t len_im, int direction) {
    if (!pl) return fail(PHASTFT_ERR_INVALID_ARG, "plan == NULL");
    if (len_re != len_im) return fail(PHASTFT_ERR_LEN_MISMATCH);                      // dit.rs:284
    if (!is_pow2(len_re)) return fail(PHASTFT_ERR_NOT_POW2);                          // dit.rs:285
    if (ilog2(len_re) != pl->log2n) return fail(PHASTFT_ERR_PLAN_MISMATCH);           // dit.rs:289
    if (direction != PHASTFT_FORWARD && direction != PHASTFT_REVERSE) return fail(PHASTFT_ERR_INVALID_ARG, "direction must be 1 or -1");
    return PHASTFT_OK;
}

// planar, in place, device pointers ------------------------------------------------------------------
template <typename T>
int32_t fft_dev(const Plan<T>* pl, T* d_re, T* d_im, int direction, size_t batch, size_t bstride, cudaStream_t stream,
                cudaEvent_t* pass_events = nullptr) {
    if (!pl || !d_re || !d_im) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    if (direction != PHASTFT_FORWARD && direction != PHASTFT_REVERSE) return fail(PHASTFT_ERR_INVALID_ARG, "direction must be 1 or -1");
    if (batch > 1 && bstride < pl->n) return fail(PHASTFT_ERR_INVALID_ARG, "batch_stride < N");
    DeviceGuard g(pl->device);
    Io<T> io;
    // inverse via the swap trick (algorithms/dit.rs:297-300): forward transform of (imags, reals), then 1/N
    if (direction == PHASTFT_FORWARD) { io.in_re = d_re; io.in_im = d_im; io.out_re = d_re; io.out_im = d_im; }
    else { io.in_re = d_im; io.in_im = d_re; io.out_re = d_im; io.out_im = d_re; }
    io.in_bstride = io.out_bstride = (long long)bstride;
    io.in_il = io.out_il = 0;
    const T scale = direction == PHASTFT_REVERSE ? T(1) / (T)pl->n : T(1);   // dit.rs:326
    if (pl->num_passes == 0) return PHASTFT_OK;
    return run_c2c(*pl, io, batch, scale, stream, pass_events);
}

// One profiled call: per-pass device time from CUDA events on the launching stream (synchronises).
template <typename T>
int32_t fft_dev_profile(const Plan<T>* pl, T* d_re, T* d_im, int direction, size_t batch, size_t bstride,
                        cudaStream_t stream, float* pass_ms, int* num_passes) {
    if (!pl || !pass_ms || !num_passes) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    DeviceGuard g(pl->device);
    *num_passes = pl->num_passes;
    cudaEvent_t ev[MAX_PASSES + 1];
    for (int i = 0; i <= pl->num_passes; ++i) CUDA_TRY(cudaEventCreate(&ev[i]));
    int32_t st = fft_dev(pl, d_re, d_im, direction, batch, bstride, stream, ev);
    if (st == PHASTFT_OK && pl->num_passes > 0) {
        cudaError_t e = cudaEventSynchronize(ev[pl->num_passes]);
        if (e != cudaSuccess) st = fail(PHASTFT_ERR_CUDA, cudaGetErrorString(e));
        for (int i = 0; i < pl->num_passes && st == PHASTFT_OK; ++i) cudaEventElapsedTime(&pass_ms[i], ev[i], ev[i + 1]);
    }
    for (int i = 0; i <= pl->num_passes; ++i) cudaEventDestroy(ev[i]);
    return st;
}

template <typename T>
int32_t fft_interleaved_dev(const Plan<T>* pl, T* d_sig, int direction, size_t batch, size_t bstride, cudaStream_t stream) {
    if (!pl || !d_sig) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    if (direction != PHASTFT_FORWARD && direction != PHASTFT_REVERSE) return fail(PHASTFT_ERR_INVALID_ARG, "direction must be 1 or -1");
    if (batch > 1 && bstride < pl->n) return fail(PHASTFT_ERR_INVALID_ARG, "batch_stride < N");
    DeviceGuard g(pl->device);
    if (pl->num_passes == 0) return PHASTFT_OK;
    Io<T> io;
    io.in_re = d_sig; io.in_im = nullptr; io.out_re = d_sig; io.out_im = nullptr;
    io.in_bstride = io.out_bstride = (long long)bstride;
    io.in_il = io.out_il = direction == PHASTFT_FORWARD ? 1 : 2;
    const T scale = direction == PHASTFT_REVERSE ? T(1) / (T)pl->n : T(1);
    return run_c2c(*pl, io, batch, scale, stream);
}

template <typename T>
int32_t ensure_staging(const Plan<T>* pl, size_t elems) {
    if (pl->stage_elems >= elems) return PHASTFT_OK;
    if (pl->stage_re) cudaFree(pl->stage_re);
    if (pl->stage_im) cudaFree(pl->stage_im);
    pl->stage_re = pl->stage_im = nullptr; pl->stage_elems = 0;
    CUDA_TRY(cudaMalloc(&pl->stage_re, elems * sizeof(T)));
    CUDA_TRY(cudaMalloc(&pl->stage_im, elems * sizeof(T)));
    pl->stage_elems = elems;
    return PHASTFT_OK;
}

// host slices: H2D, run, D2H, synchronous (lib.rs:143-150 semantics) ----------------------------------
template <typename T>
int32_t fft_host(const Plan<T>* pl, T* re, size_t len_re, T* im, size_t len_im, int direction) {
    int32_t st = check_c2c_args(pl, len_re, len_im, direction);
    if (st) return st;
    if (!re || !im) return fail(PHASTFT_ERR_INVALID_ARG, "NULL slice");
    DeviceGuard g(pl->device);
    std::lock_guard<std::mutex> host_lock(pl->host_mu);   // planners are shared by reference between threads
    {
        std::lock_guard<std::mutex> lock(pl->mu);
        st = ensure_staging(pl, pl->n);
        if (st) return st;
    }
    const size_t bytes = pl->n * sizeof(T);
    CUDA_TRY(cudaMemcpyAsync(pl->stage_re, re, bytes, cudaMemcpyHostToDevice, pl->stream));
    CUDA_TRY(cudaMemcpyAsync(pl->stage_im, im, bytes, cudaMemcpyHostToDevice, pl->stream));
    st = fft_dev(pl, pl->stage_re, pl->stage_im, direction, 1, pl->n, pl->stream);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(re, pl->stage_re, bytes, cudaMemcpyDeviceToHost, pl->stream));
    CUDA_TRY(cudaMemcpyAsync(im, pl->stage_im, bytes, cudaMemcpyDeviceToHost, pl->stream));
    CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return PHASTFT_OK;
}

template <typename T>
int32_t fft_interleaved_host(const Plan<T>* pl, T* sig, size_t len_complex, int direction) {
    int32_t st = check_c2c_args(pl, len_complex, len_complex, direction);
    if (st) return st;
    if (!sig) return fail(PHASTFT_ERR_INVALID_ARG, "NULL slice");
    DeviceGuard g(pl->device);
    std::lock_guard<std::mutex> host_lock(pl->host_mu);
    {
        std::lock_guard<std::mutex> lock(pl->mu);
        st = ensure_staging(pl, 2 * pl->n);
        if (st) return st;
    }
    const size_t bytes = 2 * pl->n * sizeof(T);
    CUDA_TRY(cudaMemcpyAsync(pl->stage_re, sig, bytes, cudaMemcpyHostToDevice, pl->stream));
    st = fft_interleaved_dev(pl, pl->stage_re, direction, 1, pl->n, pl->stream);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(sig, pl->stage_re, bytes, cudaMemcpyDeviceToHost, pl->stream));
    CUDA_TRY(cudaStreamSynchronize(pl->stream));
    return PHASTFT_OK;
}

// One-shot calls build their planner per call, like the reference (lib.rs:180-183).  Building is cheap, but
// allocating and releasing the workspace and staging buffers is not (130 ms per 2^24 f64 call), so the most
// recent one-shot plan per precision is kept and reused when the next call has the same size and device;
// phastft_oneshot_cache_clear() releases it.  The cache entry is held under its lock for the whole call.
template <class P>
struct OneShotCache {
    std::mutex mu;
    P* plan = nullptr;          // intentionally not freed at process exit (the CUDA context may be gone by then)
    size_t n = 0;
    int device = -1;
    void clear() {
        std::lock_guard<std::mutex> lock(mu);
        delete plan;
        plan = nullptr; n = 0; device = -1;
    }
};
template <typename T> OneShotCache<Plan<T>>& oneshot_c2c_cache() { static auto* c = new OneShotCache<Plan<T>>(); return *c; }

template <typename T>
int32_t fft_oneshot(T* re, size_t len_re, T* im, size_t len_im, int direction, int device) {
    if (!is_pow2(len_re)) return fail(PHASTFT_ERR_NOT_POW2);
    auto& c = oneshot_c2c_cache<T>();
    std::lock_guard<std::mutex> lock(c.mu);
    if (!c.plan || c.n != len_re || c.device != device) {
        delete c.plan;
        c.plan = nullptr; c.n = 0; c.device = -1;
        int32_t st = build_plan<T>(len_re, device, &c.plan);
        if (st) return st;
        c.n = len_re; c.device = device;
    }
    return fft_host(c.plan, re, len_re, im, len_im, direction);
}

// Host-resident batch, sharded over the plans' devices (contiguous ranges, SURVEY.md 8e; no collective on
// the data path).  Per device the shard moves through a three-slot pipeline -- H2D of chunk j+1, the FFTs of
// chunk j and D2H of chunk j-1 run on three streams -- so both PCIe directions are busy at once; a chunk is
// ~16 MiB per array (PHASTFT_HOST_CHUNK_MB).  Overlap needs page-locked host memory; pageable memory is
// still correct, the copies just serialise.
template <typename T>
int32_t batch_sharded_host(Plan<T>* const* plans, int num_plans, T* re, T* im, size_t batch, size_t bstride, int direction) {
    if (!plans || num_plans <= 0 || !re || !im) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    if (direction != PHASTFT_FORWARD && direction != PHASTFT_REVERSE) return fail(PHASTFT_ERR_INVALID_ARG, "direction must be 1 or -1");
    for (int g = 0; g < num_plans; ++g)
        if (!plans[g]) return fail(PHASTFT_ERR_INVALID_ARG, "NULL plan in the plan list");
    const size_t n = plans[0]->n;
    for (int g = 0; g < num_plans; ++g)
        if (plans[g]->n != n) return fail(PHASTFT_ERR_PLAN_MISMATCH);
    if (bstride < n) return fail(PHASTFT_ERR_INVALID_ARG, "batch_stride < N");
    if (batch == 0) return PHASTFT_OK;
    std::vector<std::mutex*> locks;
    for (int g = 0; g < num_plans; ++g) locks.push_back(&plans[g]->host_mu);
    std::sort(locks.begin(), locks.end(), std::less<std::mutex*>());
    locks.erase(std::unique(locks.begin(), locks.end()), locks.end());
    if (locks.size() != (size_t)num_plans) return fail(PHASTFT_ERR_INVALID_ARG, "the same plan passed twice");
    struct Unlock { std::vector<std::mutex*>& l; ~Unlock() { for (auto* m : l) m->unlock(); } };
    for (auto* m : locks) m->lock();                         // address order: no deadlock between overlapping calls
    Unlock unlock_all{locks};
    constexpr int NSLOT = 3;
    size_t chunk_mb = 16;
    if (const char* e = getenv("PHASTFT_HOST_CHUNK_MB")) { long v = atol(e); if (v > 0) chunk_mb = (size_t)v; }
    const size_t per_chunk = std::max<size_t>(1, (chunk_mb << 20) / (n * sizeof(T)));   // transforms per chunk
    struct Shard {
        const Plan<T>* pl; size_t lo, nb, chunks; size_t slot_elems;
        cudaEvent_t h2d_done[NSLOT], fft_done[NSLOT], d2h_done[NSLOT];
        bool ev = false;
    };
    std::vector<Shard> sh(num_plans);
    auto cleanup = [&]() {
        for (auto& s : sh)
            if (s.ev) {
                DeviceGuard guard(s.pl->device);
                for (int k = 0; k < NSLOT; ++k)
                    for (cudaEvent_t e : {s.h2d_done[k], s.fft_done[k], s.d2h_done[k]}) if (e) cudaEventDestroy(e);
                s.ev = false;
            }
    };
    size_t max_chunks = 0;
    for (int g = 0; g < num_plans; ++g) {
        Shard& s = sh[g];
        s.pl = plans[g];
        s.lo = batch * g / num_plans;
        s.nb = batch * (g + 1) / num_plans - s.lo;
        const size_t pc = std::min(per_chunk, std::max<size_t>(1, s.nb));
        s.chunks = (s.nb + pc - 1) / pc;
        s.slot_elems = pc * n;
        max_chunks = std::max(max_chunks, s.chunks);
        if (!s.nb) continue;
        DeviceGuard guard(s.pl->device);
        {
            std::lock_guard<std::mutex> lock(s.pl->mu);
            int32_t st = ensure_staging(s.pl, std::min<size_t>(NSLOT, s.chunks) * s.slot_elems);
            if (st) { cleanup(); return st; }
            if (!s.pl->stream_h2d) {
                if (cudaStreamCreateWithFlags(&s.pl->stream_h2d, cudaStreamNonBlocking) != cudaSuccess ||
                    cudaStreamCreateWithFlags(&s.pl->stream_d2h, cudaStreamNonBlocking) != cudaSuccess) { cleanup(); return fail(PHASTFT_ERR_CUDA, "stream create"); }
            }
        }
        bool ev_ok = true;
        for (int k = 0; k < NSLOT; ++k) { s.h2d_done[k] = s.fft_done[k] = s.d2h_done[k] = nullptr; }
        for (int k = 0; k < NSLOT; ++k) {
            ev_ok &= cudaEventCreateWithFlags(&s.h2d_done[k], cudaEventDisableTiming) == cudaSuccess;
            ev_ok &= cudaEventCreateWithFlags(&s.fft_done[k], cudaEventDisableTiming) == cudaSuccess;
            ev_ok &= cudaEventCreateWithFlags(&s.d2h_done[k], cudaEventDisableTiming) == cudaSuccess;
        }
        s.ev = true;
        if (!ev_ok) { (void)cudaGetLastError(); cleanup(); return fail(PHASTFT_ERR_CUDA, "cudaEventCreate"); }
    }
    // issue chunk j of every device before chunk j+1 of any, so all devices stream concurrently
    int32_t st = PHASTFT_OK;
    for (size_t j = 0; j < max_chunks && !st; ++j) {
        for (int g = 0; g < num_plans && !st; ++g) {
            Shard& s = sh[g];
            if (j >= s.chunks) continue;
            const Plan<T>* pl = s.pl;
            DeviceGuard guard(pl->device);
            const size_t pc = s.slot_elems / n;
            const size_t first = s.lo + j * pc;
            const size_t cnt = std::min(pc, s.lo + s.nb - first);
            const int slot = (int)(j % NSLOT);
            T* d_re = pl->stage_re + (size_t)slot * s.slot_elems;
            T* d_im = pl->stage_im + (size_t)slot * s.slot_elems;
            T* h_re = re + first * bstride;
            T* h_im = im + first * bstride;
            auto ok = [&](cudaError_t e) { if (e != cudaSuccess && !st) st = fail(PHASTFT_ERR_CUDA, cudaGetErrorString(e)); return e == cudaSuccess; };
            if (j >= NSLOT) ok(cudaStreamWaitEvent(pl->stream_h2d, s.d2h_done[slot], 0));     // the slot's previous result has left
            ok(cudaMemcpy2DAsync(d_re, n * sizeof(T), h_re, bstride * sizeof(T), n * sizeof(T), cnt, cudaMemcpyHostToDevice, pl->stream_h2d));
            ok(cudaMemcpy2DAsync(d_im, n * sizeof(T), h_im, bstride * sizeof(T), n * sizeof(T), cnt, cudaMemcpyHostToDevice, pl->stream_h2d));
            ok(cudaEventRecord(s.h2d_done[slot], pl->stream_h2d));
            ok(cudaStreamWaitEvent(pl->stream, s.h2d_done[slot], 0));
            if (!st) st = fft_dev(pl, d_re, d_im, direction, cnt, n, pl->stream);
            ok(cudaEventRecord(s.fft_done[slot], pl->stream));
            ok(cudaStreamWaitEvent(pl->stream_d2h, s.fft_done[slot], 0));
            ok(cudaMemcpy2DAsync(h_re, bstride * sizeof(T), d_re, n * sizeof(T), n * sizeof(T), cnt, cudaMemcpyDeviceToHost, pl->stream_d2h));
            ok(cudaMemcpy2DAsync(h_im, bstride * sizeof(T), d_im, n * sizeof(T), n * sizeof(T), cnt, cudaMemcpyDeviceToHost, pl->stream_d2h));
            ok(cudaEventRecord(s.d2h_done[slot], pl->stream_d2h));
        }
    }
    for (int g = 0; g < num_plans; ++g) {
        if (!sh[g].nb) continue;
        DeviceGuard guard(plans[g]->device);
        cudaError_t e1 = cudaStreamSynchronize(plans[g]->stream_h2d);
        cudaError_t e2 = cudaStreamSynchronize(plans[g]->stream);
        cudaError_t e3 = cudaStreamSynchronize(plans[g]->stream_d2h);
        for (cudaError_t e : {e1, e2, e3})
            if (e != cudaSuccess && !st) st = fail(PHASTFT_ERR_CUDA, cudaGetErrorString(e));
    }
    cleanup();
    return st;
}

// ---- PlannerMode::Tune (planner.rs:25-32: "benchmarks both paths at plan time, picks whichever is faster";
// the reference accepts the mode and ignores it, planner.rs:65).  Here it is real: a handful of pass
// decompositions / tile widths around the heuristic choice are built, timed on a scratch signal with CUDA
// events, and the fastest is kept.
template <typename T>
int32_t build_plan_tuned(size_t n, int device, Plan<T>** out) {
    if (!out) return fail(PHASTFT_ERR_INVALID_ARG, "out == NULL");
    *out = nullptr;
    int32_t st = build_plan<T>(n, device, out);             // the heuristic plan (also validates n / device)
    if (st) return st;
    Plan<T>* best = *out;
    const int ln = best->log2n;
    if (best->num_passes < 2) return PHASTFT_OK;            // one-CTA sizes: nothing to choose
    DeviceGuard guard(device);
    const int CH = TileC<T>::CH, CN = TileC<T>::CN, CW = TileC<T>::CW;
    std::vector<PlanChoice> cands;
    auto add = [&](std::vector<int> f, std::vector<int> c) { PlanChoice pc; pc.factors = std::move(f); pc.pass_c = std::move(c); cands.push_back(std::move(pc)); };
    if (ln <= 20) {
        for (int a : {ln / 2, (ln + 1) / 2})
            for (int c : {CH, CN, CW}) {
                if (a > 10 || ln - a > 10 || a < 5 || ln - a < 5) continue;
                add({a, ln - a}, {c, c});
            }
        if (ln >= 18) { add({6, ln - 12, 6}, {CN, CN, CN}); add({7, ln - 14, 7}, {CN, CN, CN}); }
    } else {
        for (int e : {7, 8, 9}) {
            const int m = ln - 2 * e;
            if (m < 5 || m > 10) continue;
            add({e, m, e}, {CW, CN, CW});
            add({e, m, e}, {CN, CN, CN});
        }
        if (ln - 18 >= 5 && ln - 18 <= 10) { add({10, ln - 18, 8}, {CN, CN, CW}); add({8, ln - 18, 10}, {CW, CN, CN}); }
    }
    T *re = nullptr, *im = nullptr;
    if (cudaMalloc(&re, n * sizeof(T)) != cudaSuccess || cudaMalloc(&im, n * sizeof(T)) != cudaSuccess) {
        cudaGetLastError();
        if (re) cudaFree(re);
        return PHASTFT_OK;                                   // no room to tune: keep the heuristic plan
    }
    cudaMemset(re, 0, n * sizeof(T)); cudaMemset(im, 0, n * sizeof(T));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    auto time_plan = [&](Plan<T>* pl) -> float {
        const int reps = ln <= 20 ? 20 : (ln <= 24 ? 5 : 2);
        for (int w = 0; w < 2; ++w) if (fft_dev(pl, re, im, PHASTFT_FORWARD, 1, n, pl->stream) != PHASTFT_OK) return 1e30f;
        cudaEventRecord(e0, pl->stream);
        for (int r = 0; r < reps; ++r) fft_dev(pl, re, im, PHASTFT_FORWARD, 1, n, pl->stream);
        cudaEventRecord(e1, pl->stream);
        if (cudaEventSynchronize(e1) != cudaSuccess) return 1e30f;
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        return ms / reps;
    };
    float best_ms = time_plan(best);
    for (const PlanChoice& pc : cands) {
        Plan<T>* cand = nullptr;
        g_choice = &pc;
        int32_t cst = build_plan<T>(n, device, &cand);
        g_choice = nullptr;
        if (cst != PHASTFT_OK || !cand) { delete cand; continue; }
        if (cand->description == best->description) { delete cand; continue; }
        const float ms = time_plan(cand);
        if (ms < best_ms * 0.98f) { delete best; best = cand; best_ms = ms; } else delete cand;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(re); cudaFree(im);
    best->description += " [tuned]";
    g_last_error.clear();
    *out = best;
    return PHASTFT_OK;
}

// ---- table blob export / import / broadcast ------------------------------------------------------------
template <typename T>
int32_t tables_export(const Plan<T>* pl, void* dst, cudaStream_t s) {
    if (!pl || !dst) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    DeviceGuard g(pl->device);
    CUDA_TRY(cudaMemcpyAsync(dst, pl->blob_dev, pl->blob_host.size(), cudaMemcpyDeviceToDevice, s));
    return PHASTFT_OK;
}
// Compares a blob header (already on the host) with the plan's own.
template <typename T>
int32_t check_blob_header(const Plan<T>* pl, const BlobHeader& h) {
    BlobHeader mine;
    memcpy(&mine, pl->blob_host.data(), sizeof(mine));
    if (h.magic != BLOB_MAGIC) return fail(PHASTFT_ERR_PLAN_MISMATCH, "table blob: bad magic (not a phastft table blob)");
    if (h.n != mine.n || h.precision_bits != mine.precision_bits) return fail(PHASTFT_ERR_PLAN_MISMATCH, "table blob is for another size / precision");
    if (h.bytes != mine.bytes || h.num_passes != mine.num_passes || h.layout_sig != mine.layout_sig)
        return fail(PHASTFT_ERR_PLAN_MISMATCH, "table blob was laid out for a different pass decomposition / kernel choice "
                                               "(PlannerMode::Tune or a PHASTFT_* override on one rank only?)");
    return PHASTFT_OK;
}

template <typename T>
int32_t tables_import(Plan<T>* pl, const void* src, cudaStream_t s) {
    if (!pl || !src) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    DeviceGuard g(pl->device);
    BlobHeader h;
    CUDA_TRY(cudaMemcpyAsync(&h, src, sizeof(h), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    int32_t st = check_blob_header(pl, h);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(pl->blob_dev, src, pl->blob_host.size(), cudaMemcpyDeviceToDevice, s));
    return PHASTFT_OK;
}

typedef int (*nccl_bcast_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
// Two collectives, both joined by every rank whatever it finds (so a mismatching rank cannot leave the others hanging):
// the root's 256-byte header first, then the root's blob at the size the header states -- into the plan's tables when the
// layouts agree, into a throw-away buffer (and PHASTFT_ERR_PLAN_MISMATCH) when they do not.
template <typename T>
int32_t tables_broadcast(Plan<T>* pl, void* comm, int root, cudaStream_t s) {
    if (!pl || !comm) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    static nccl_bcast_fn bcast = [] {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        return h ? reinterpret_cast<nccl_bcast_fn>(dlsym(h, "ncclBroadcast")) : nullptr;
    }();
    if (!bcast) return fail(PHASTFT_ERR_NCCL, "libnccl.so.2 / ncclBroadcast not found");
    DeviceGuard g(pl->device);
    unsigned char* d_hdr = nullptr;
    CUDA_TRY(cudaMalloc(&d_hdr, BLOB_HEADER_BYTES));
    int rc = bcast(pl->blob_dev, d_hdr, BLOB_HEADER_BYTES, /*ncclChar*/ 0, root, comm, s);
    BlobHeader h;
    memset(&h, 0, sizeof(h));
    cudaError_t ce = rc == 0 ? cudaMemcpyAsync(&h, d_hdr, sizeof(h), cudaMemcpyDeviceToHost, s) : cudaSuccess;
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
    cudaFree(d_hdr);
    if (rc != 0) return fail(PHASTFT_ERR_NCCL, "ncclBroadcast (header) returned " + std::to_string(rc));
    if (ce != cudaSuccess) return fail(PHASTFT_ERR_CUDA, cudaGetErrorString(ce));
    const int32_t st = check_blob_header(pl, h);
    if (h.magic != BLOB_MAGIC || h.bytes == 0 || h.bytes > (uint64_t(1) << 34)) return st ? st : fail(PHASTFT_ERR_PLAN_MISMATCH, "bad header from root");
    unsigned char* target = pl->blob_dev;
    unsigned char* scratch = nullptr;
    if (st) {   // join the second collective anyway, at the root's size
        if (cudaMalloc(&scratch, h.bytes) != cudaSuccess) { (void)cudaGetLastError(); return st; }
        target = scratch;
    }
    rc = bcast(pl->blob_dev, target, h.bytes, /*ncclChar*/ 0, root, comm, s);
    if (scratch) { cudaStreamSynchronize(s); cudaFree(scratch); }
    if (st) { const std::string keep = g_last_error; (void)keep; return check_blob_header(pl, h); }
    if (rc != 0) return fail(PHASTFT_ERR_NCCL, "ncclBroadcast returned " + std::to_string(rc));
    return PHASTFT_OK;
}

// =================================================================================================
// r2c / c2r
// =================================================================================================
template <typename T>
struct PlanR2c {
    size_t n = 0;
    int device = 0;
    Plan<T>* inner = nullptr;          // half-length c2c (planner.rs:203)
    unsigned char* tw_dev = nullptr;   // two-level W_n table for the untangle / preprocess twiddles
    size_t hi_elems = 0, lo_elems = 0;
    int lo_bits = 0;
    mutable std::mutex mu;
    mutable std::mutex host_mu;        // held for a whole *_host call (lock order: host_mu, then mu)
    mutable T* d_real = nullptr;       // host-API staging: N reals
    mutable T* d_spec_re = nullptr;    // N/2+1
    mutable T* d_spec_im = nullptr;
    mutable T* d_scr_re = nullptr;     // N/2 (c2r scratch when the caller passes none)
    mutable T* d_scr_im = nullptr;
    mutable cudaEvent_t scr_free = nullptr;        // orders reuse of the plan-owned scratch across streams (like Plan::ws_free)
    mutable cudaStream_t scr_last_stream = nullptr;
    mutable bool scr_used = false;
    ~PlanR2c() {
        DeviceGuard g(device);
        if (scr_free) cudaEventDestroy(scr_free);
        for (void* p : {(void*)tw_dev, (void*)d_real, (void*)d_spec_re, (void*)d_spec_im, (void*)d_scr_re, (void*)d_scr_im})
            if (p) cudaFree(p);
        delete inner;
    }
};

template <typename T>
int32_t build_plan_r2c(size_t n, int device, PlanR2c<T>** out) {
    if (!out) return fail(PHASTFT_ERR_INVALID_ARG, "out == NULL");
    *out = nullptr;
    if (!(n >= 4 && is_pow2(n))) return fail(PHASTFT_ERR_R2C_N);   // planner.rs:195
    if (n > (size_t(1) << 31)) return fail(PHASTFT_ERR_INVALID_ARG, "n > 2^31 not supported");
    std::unique_ptr<PlanR2c<T>> pl(new PlanR2c<T>());
    pl->n = n; pl->device = device;
    int32_t st = build_plan<T>(n / 2, device, &pl->inner);
    if (st) return st;
    DeviceGuard g(device);
    const int ln = ilog2(n);
    pl->lo_bits = (ln + 1) / 2;
    pl->lo_elems = size_t(1) << pl->lo_bits;
    pl->hi_elems = size_t(1) << (ln - pl->lo_bits);
    std::vector<double2> tab(pl->hi_elems + pl->lo_elems);
    for (size_t h = 0; h < pl->hi_elems; ++h) root_of_unity((uint64_t)h << pl->lo_bits, n, tab[h].x, tab[h].y);
    for (size_t l = 0; l < pl->lo_elems; ++l) root_of_unity(l, n, tab[pl->hi_elems + l].x, tab[pl->hi_elems + l].y);
    CUDA_TRY(cudaMalloc(&pl->tw_dev, tab.size() * sizeof(double2)));
    CUDA_TRY(cudaMemcpy(pl->tw_dev, tab.data(), tab.size() * sizeof(double2), cudaMemcpyHostToDevice));
    // c2r scratch for the allocating variants lives in the plan (r2c.rs:716-718 allocates per call)
    CUDA_TRY(cudaMalloc(&pl->d_scr_re, (n / 2) * sizeof(T)));
    CUDA_TRY(cudaMalloc(&pl->d_scr_im, (n / 2) * sizeof(T)));
    CUDA_TRY(cudaEventCreateWithFlags(&pl->scr_free, cudaEventDisableTiming));
    *out = pl.release();
    return PHASTFT_OK;
}

template <typename T>
Tw2 r2c_tw2(const PlanR2c<T>* pl) {
    Tw2 t;
    t.hi = reinterpret_cast<const double2*>(pl->tw_dev);
    t.lo = t.hi + pl->hi_elems;
    t.lo_bits = pl->lo_bits;
    return t;
}

template <typename T>
int32_t r2c_dev(const PlanR2c<T>* pl, const T* d_in, T* d_ore, T* d_oim, cudaStream_t stream) {
    if (!pl || !d_in || !d_ore || !d_oim) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    DeviceGuard g(pl->device);
    const size_t half = pl->n / 2;
    // (1)+(2) deinterleave fused into the first pass load: z[k] = x[2k] + i x[2k+1] (r2c.rs:557-569),
    //         half-length forward c2c into output[..half] (r2c.rs:575)
    Io<T> io;
    io.in_re = d_in; io.in_im = nullptr; io.in_il = 1; io.in_bstride = (long long)half;
    io.out_re = d_ore; io.out_im = d_oim; io.out_il = 0; io.out_bstride = (long long)half;
    int32_t st;
    if (pl->inner->num_passes == 0) return fail(PHASTFT_ERR_INVALID_ARG, "unreachable: half >= 2");
    st = run_c2c(*pl->inner, io, 1, T(1), stream);
    if (st) return st;
    // (3) untangle in place over all half+1 slots (r2c.rs:584-592)
    RealParams<T> rp;
    memset(&rp, 0, sizeof(rp));
    rp.re = d_ore; rp.im = d_oim; rp.log2half = ilog2(half); rp.tw2 = r2c_tw2(pl);
    const size_t q = half / 2;
    dim3 grid((unsigned)((q + 1 + 255) / 256), 1);
    r2c_untangle_kernel<T><<<grid, 256, 0, stream>>>(rp);
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return PHASTFT_OK;
}

template <typename T>
int32_t c2r_dev(const PlanR2c<T>* pl, const T* d_ire, const T* d_iim, T* d_out, T* d_sre, T* d_sim, cudaStream_t stream) {
    if (!pl || !d_ire || !d_iim || !d_out) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    if ((d_sre == nullptr) != (d_sim == nullptr)) return fail(PHASTFT_ERR_INVALID_ARG, "pass both scratch arrays or neither");
    DeviceGuard g(pl->device);
    const size_t half = pl->n / 2;
    // Pre-processing (r2c.rs:764-780) folded into the loads of the inverse transform's first pass when the plan has that
    // kernel: no scratch, one HBM round trip of N/2 complex values less.  PHASTFT_C2R_FUSE=0 keeps the separate sweep.
    const char* fuse_e = getenv("PHASTFT_C2R_FUSE");
    const bool fuse_env = fuse_e ? atoi(fuse_e) != 0 : true;
    const Plan<T>& in = *pl->inner;
    // Measured (profiles/r02_exp_c2r_fuse2.txt): 1.03-1.26x for f64 up to N = 2^20 and from 2^24, 1.04-1.23x for every f32 size;
    // f64 2^21..2^23 (whole signal in L2, so the sweep's scratch round trip is cheap, and the 1024-row tile of 2^21 keeps only 8
    // of its 32 loads per thread in flight) 0.96-0.99x: those keep the separate sweep unless PHASTFT_C2R_FUSE=1 is set.
    const bool fuse_size = sizeof(T) == 4 || in.log2n < 20 || in.log2n > 22 || fuse_e != nullptr;
    if (fuse_env && fuse_size && in.num_passes >= 2 && in.pass[0].kc && !(in.cl && in.cl_min_batch <= 1) && !in.pipe_1) {
        Io<T> io;
        io.in_re = d_ire; io.in_im = d_iim; io.in_il = 0; io.in_bstride = (long long)half;
        io.pre_tw2 = r2c_tw2(pl); io.pre_log2half = ilog2(half);
        io.out_re = d_out; io.out_im = nullptr; io.out_il = 2; io.out_bstride = (long long)half;
        return run_c2c(in, io, 1, T(1) / (T)half, stream);
    }
    std::unique_lock<std::mutex> lock(pl->mu, std::defer_lock);
    bool own_scratch = false, capturing = false;
    if (!d_sre) {
        // The plan-owned scratch is used by kernels that run after this call returns: a caller on another stream
        // first waits for the previous user (the same protocol as the c2c workspace, run_c2c).
        lock.lock();
        d_sre = pl->d_scr_re; d_sim = pl->d_scr_im;
        own_scratch = true;
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        CUDA_TRY(cudaStreamIsCapturing(stream, &cap));
        capturing = cap != cudaStreamCaptureStatusNone;
        if (!capturing && pl->scr_used && pl->scr_last_stream != stream) CUDA_TRY(cudaStreamWaitEvent(stream, pl->scr_free, 0));
    }
    // (1) pre-process into scratch (r2c.rs:764-780)
    RealParams<T> rp;
    memset(&rp, 0, sizeof(rp));
    rp.re = d_sre; rp.im = d_sim; rp.in_re = d_ire; rp.in_im = d_iim; rp.log2half = ilog2(half); rp.tw2 = r2c_tw2(pl);
    dim3 grid((unsigned)((half + 255) / 256), 1);
    c2r_preprocess_kernel<T><<<grid, 256, 0, stream>>>(rp);
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1, std::memory_order_relaxed);
    // (2) inverse half-length c2c on the scratch (swap trick + 1/half, r2c.rs:782) with
    // (3) the re-interleave into the real output (r2c.rs:790-798) fused into the last store
    Io<T> io;
    io.in_re = d_sim; io.in_im = d_sre; io.in_il = 0; io.in_bstride = (long long)half;
    io.out_re = d_out; io.out_im = nullptr; io.out_il = 2; io.out_bstride = (long long)half;
    int32_t st = run_c2c(*pl->inner, io, 1, T(1) / (T)half, stream);
    if (st == PHASTFT_OK && own_scratch && !capturing) {
        CUDA_TRY(cudaEventRecord(pl->scr_free, stream));
        pl->scr_last_stream = stream;
        pl->scr_used = true;
    }
    return st;
}

// Batched device-resident r2c / c2r (strides in elements of T).  The real side is read or written as complex pairs, so its
// stride must be even and its base aligned to 2 * sizeof(T).  Checked before anything is launched.
template <typename T>
int32_t check_real_batch(const PlanR2c<T>* pl, const void* p0, const void* p1, const void* p2, const T* real, size_t real_stride,
                         size_t spec_stride, size_t batch) {
    if (!pl || !p0 || !p1 || !p2) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    const size_t n = pl->n, half = n / 2;
    if (real_stride < n) return fail(PHASTFT_ERR_INVALID_ARG, "real-side stride < N");
    if (spec_stride < half + 1) return fail(PHASTFT_ERR_INVALID_ARG, "spectrum stride < N/2 + 1");
    if (real_stride & 1) return fail(PHASTFT_ERR_INVALID_ARG, "real-side stride must be even (the reals are read as complex pairs)");
    if (reinterpret_cast<uintptr_t>(real) % (2 * sizeof(T))) return fail(PHASTFT_ERR_INVALID_ARG, "real-side base not aligned to 2 * sizeof(T)");
    const size_t lim = (size_t(1) << 62) / sizeof(T);
    if (batch > 1 && (batch - 1) > (lim - n) / std::max(real_stride, spec_stride)) return fail(PHASTFT_ERR_INVALID_ARG, "batch * stride too large");
    return PHASTFT_OK;
}

// r2c of the inner plan's one-CTA kernel with the untangle in its store (MODE_R2C_OUT), or NULL: the half-length c2c and the
// separate untangle sweep.  PHASTFT_R2C_FUSE=0 forces the latter (equivalence tests, measurement).
template <typename T>
const KernelEntry<T>* r2c_fused_kernel(const Plan<T>& in, size_t batch) {
    const char* e = getenv("PHASTFT_R2C_FUSE");
    if (e && atoi(e) == 0) return nullptr;
    const bool one_cta = in.num_passes == 1 || (in.alt_row.k && batch >= in.alt_row_min_batch);     // as run_c2c decides
    if (!one_cta) return nullptr;
    bool many = false;
    return r2c_out_kernel(in, in.num_passes == 1 ? in.pass[0] : in.alt_row, batch, many);
}

template <typename T>
int32_t r2c_batch_dev(const PlanR2c<T>* pl, const T* d_in, T* d_ore, T* d_oim, size_t batch, size_t in_stride, size_t out_stride,
                      cudaStream_t stream) {
    int32_t st = check_real_batch(pl, d_in, d_ore, d_oim, d_in, in_stride, out_stride, batch);
    if (st || batch == 0) return st;
    if (batch == 1) return r2c_dev(pl, d_in, d_ore, d_oim, stream);          // bit-identical to the single call by construction
    DeviceGuard g(pl->device);
    const size_t half = pl->n / 2;
    const Plan<T>& in = *pl->inner;
    Io<T> io;
    io.in_re = d_in; io.in_im = nullptr; io.in_il = 1; io.in_bstride = (long long)(in_stride / 2);
    io.out_re = d_ore; io.out_im = d_oim; io.out_il = 0; io.out_bstride = (long long)out_stride;
    if (r2c_fused_kernel(in, batch)) {
        io.r2c_out = 1; io.pre_tw2 = r2c_tw2(pl);
        return run_c2c(in, io, batch, T(1), stream);
    }
    st = run_c2c(in, io, batch, T(1), stream);
    if (st) return st;
    // untangle sweep over every member: (member, pair) flattened into grid.x, launches of at most 2^30 blocks
    RealParams<T> rp;
    memset(&rp, 0, sizeof(rp));
    rp.bstride = (long long)out_stride; rp.log2half = ilog2(half); rp.tw2 = r2c_tw2(pl);
    const size_t q1 = half / 2 + 1;
    const size_t max_members = (size_t(256) << 30) / q1;
    for (size_t done = 0; done < batch; done += max_members) {
        const size_t nb = std::min(max_members, batch - done);
        rp.re = d_ore + done * out_stride; rp.im = d_oim + done * out_stride;
        r2c_untangle_batch_kernel<T><<<(unsigned)((nb * q1 + 255) / 256), 256, 0, stream>>>(rp, (long long)nb);
        CUDA_TRY(cudaGetLastError());
        g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    return PHASTFT_OK;
}

// Every batched c2r path pre-processes on load (first pass, or the one-CTA kernel): no scratch that would grow with the batch.
template <typename T>
int32_t c2r_batch_dev(const PlanR2c<T>* pl, const T* d_ire, const T* d_iim, T* d_out, size_t batch, size_t in_stride, size_t out_stride,
                      cudaStream_t stream) {
    int32_t st = check_real_batch(pl, d_ire, d_iim, d_out, d_out, out_stride, in_stride, batch);
    if (st || batch == 0) return st;
    if (batch == 1) return c2r_dev<T>(pl, d_ire, d_iim, d_out, nullptr, nullptr, stream);
    DeviceGuard g(pl->device);
    const size_t half = pl->n / 2;
    Io<T> io;
    io.in_re = d_ire; io.in_im = d_iim; io.in_il = 0; io.in_bstride = (long long)in_stride;
    io.pre_tw2 = r2c_tw2(pl); io.pre_log2half = ilog2(half);
    io.out_re = d_out; io.out_im = nullptr; io.out_il = 2; io.out_bstride = (long long)(out_stride / 2);
    return run_c2c(*pl->inner, io, batch, T(1) / (T)half, stream);
}

template <typename T>
int32_t ensure_r2c_staging(const PlanR2c<T>* pl) {
    const size_t half = pl->n / 2;
    if (!pl->d_real) CUDA_TRY(cudaMalloc(&pl->d_real, pl->n * sizeof(T)));
    if (!pl->d_spec_re) CUDA_TRY(cudaMalloc(&pl->d_spec_re, (half + 1) * sizeof(T)));
    if (!pl->d_spec_im) CUDA_TRY(cudaMalloc(&pl->d_spec_im, (half + 1) * sizeof(T)));
    return PHASTFT_OK;
}

template <typename T>
int32_t r2c_host(const PlanR2c<T>* pl, const T* in, size_t len_in, T* ore, size_t len_ore, T* oim, size_t len_oim) {
    if (!pl) return fail(PHASTFT_ERR_INVALID_ARG, "plan == NULL");
    const size_t n = pl->n, half = n / 2;
    if (len_in != n) return fail(PHASTFT_ERR_INPUT_LEN);              // r2c.rs:543
    if (len_ore != half + 1) return fail(PHASTFT_ERR_OUTPUT_RE_LEN);  // r2c.rs:544
    if (len_oim != half + 1) return fail(PHASTFT_ERR_OUTPUT_IM_LEN);  // r2c.rs:549
    if (!in || !ore || !oim) return fail(PHASTFT_ERR_INVALID_ARG, "NULL slice");
    DeviceGuard g(pl->device);
    std::lock_guard<std::mutex> host_lock(pl->host_mu);     // same lock as c2r_host: both use the plan's staging buffers
    std::lock_guard<std::mutex> lock(pl->mu);
    int32_t st = ensure_r2c_staging(pl);
    if (st) return st;
    cudaStream_t s = pl->inner->stream;
    CUDA_TRY(cudaMemcpyAsync(pl->d_real, in, n * sizeof(T), cudaMemcpyHostToDevice, s));
    st = r2c_dev(pl, pl->d_real, pl->d_spec_re, pl->d_spec_im, s);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(ore, pl->d_spec_re, (half + 1) * sizeof(T), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaMemcpyAsync(oim, pl->d_spec_im, (half + 1) * sizeof(T), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return PHASTFT_OK;
}

template <typename T>
int32_t c2r_host(const PlanR2c<T>* pl, const T* ire, size_t len_ire, const T* iim, size_t len_iim, T* out, size_t len_out,
                 T* sre, size_t len_sre, T* sim, size_t len_sim) {
    if (!pl) return fail(PHASTFT_ERR_INVALID_ARG, "plan == NULL");
    const size_t n = pl->n, half = n / 2;
    if (len_out != n) return fail(PHASTFT_ERR_OUTPUT_LEN);            // r2c.rs:750
    if (len_ire != half + 1) return fail(PHASTFT_ERR_INPUT_RE_LEN);   // r2c.rs:751
    if (len_iim != half + 1) return fail(PHASTFT_ERR_INPUT_IM_LEN);   // r2c.rs:756
    const bool has_scratch = sre || sim || len_sre || len_sim;
    if (has_scratch) {
        if (len_sre != half) return fail(PHASTFT_ERR_SCRATCH_RE_LEN);  // r2c.rs:761
        if (len_sim != half) return fail(PHASTFT_ERR_SCRATCH_IM_LEN);  // r2c.rs:762
    }
    if (!ire || !iim || !out) return fail(PHASTFT_ERR_INVALID_ARG, "NULL slice");
    DeviceGuard g(pl->device);
    cudaStream_t s = pl->inner->stream;
    std::lock_guard<std::mutex> host_lock(pl->host_mu);     // whole call: the staging buffers and the stream are per plan
    {
        std::lock_guard<std::mutex> lock(pl->mu);           // released before c2r_dev, which takes it for the plan-owned scratch
        int32_t st = ensure_r2c_staging(pl);
        if (st) return st;
    }
    CUDA_TRY(cudaMemcpyAsync(pl->d_spec_re, ire, (half + 1) * sizeof(T), cudaMemcpyHostToDevice, s));
    CUDA_TRY(cudaMemcpyAsync(pl->d_spec_im, iim, (half + 1) * sizeof(T), cudaMemcpyHostToDevice, s));
    int32_t st = c2r_dev<T>(pl, pl->d_spec_re, pl->d_spec_im, pl->d_real, nullptr, nullptr, s);
    if (st) return st;
    CUDA_TRY(cudaMemcpyAsync(out, pl->d_real, n * sizeof(T), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(cudaStreamSynchronize(s));
    return PHASTFT_OK;
}

template <typename T> OneShotCache<PlanR2c<T>>& oneshot_r2c_cache() { static auto* c = new OneShotCache<PlanR2c<T>>(); return *c; }
// caller holds c.mu
template <typename T>
int32_t oneshot_r2c_plan(OneShotCache<PlanR2c<T>>& c, size_t n, int device, PlanR2c<T>** out) {
    if (!c.plan || c.n != n || c.device != device) {
        delete c.plan;
        c.plan = nullptr; c.n = 0; c.device = -1;
        int32_t st = build_plan_r2c<T>(n, device, &c.plan);
        if (st) return st;
        c.n = n; c.device = device;
    }
    *out = c.plan;
    return PHASTFT_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
#define AS_PLAN(T, p) reinterpret_cast<Plan<T>*>(p)
#define AS_CPLAN(T, p) reinterpret_cast<const Plan<T>*>(p)
#define AS_R2C(T, p) reinterpret_cast<PlanR2c<T>*>(p)
#define AS_CR2C(T, p) reinterpret_cast<const PlanR2c<T>*>(p)

extern "C" {

const char* phastft_last_error(void) { return g_last_error.c_str(); }
const char* phastft_version(void) { return "phastft_cuda 0.2.0 (sm_100a)"; }
int32_t phastft_host_register(void* host_ptr, size_t bytes) {
    if (!host_ptr || !bytes) return fail(PHASTFT_ERR_INVALID_ARG, "NULL or empty range");
    CUDA_TRY(cudaHostRegister(host_ptr, bytes, cudaHostRegisterPortable));
    return PHASTFT_OK;
}
int32_t phastft_host_unregister(void* host_ptr) {
    if (!host_ptr) return fail(PHASTFT_ERR_INVALID_ARG, "NULL pointer");
    CUDA_TRY(cudaHostUnregister(host_ptr));
    return PHASTFT_OK;
}
void phastft_oneshot_cache_clear(void) {
    oneshot_c2c_cache<double>().clear();
    oneshot_c2c_cache<float>().clear();
    oneshot_r2c_cache<double>().clear();
    oneshot_r2c_cache<float>().clear();
}

uint64_t phastft_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
int32_t phastft_device_count(int* count) {
    if (!count) return fail(PHASTFT_ERR_INVALID_ARG, "count == NULL");
    *count = 0;
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess || *count == 0) { *count = 0; return fail(PHASTFT_ERR_NO_DEVICE, e != cudaSuccess ? cudaGetErrorString(e) : ""); }
    return PHASTFT_OK;
}

int32_t phastft_plan_factorization(size_t n, int precision_bits, int* log2_factors, int* num_passes) {
    if (!log2_factors || !num_passes) return fail(PHASTFT_ERR_INVALID_ARG, "NULL argument");
    if (!is_pow2(n)) return fail(PHASTFT_ERR_NOT_POW2);
    if (precision_bits != 32 && precision_bits != 64) return fail(PHASTFT_ERR_INVALID_ARG, "precision_bits must be 32 or 64");
    const int ln = ilog2(n);
    std::vector<int> f = ln == 0 ? std::vector<int>{} : (precision_bits == 64 ? choose_factors<double>(ln) : choose_factors<float>(ln));
    *num_passes = (int)f.size();
    for (size_t i = 0; i < f.size(); ++i) log2_factors[i] = f[i];
    return PHASTFT_OK;
}

void phastft_options_default(phastft_options* out) {
    if (!out) return;
    out->multithreaded_bit_reversal = 0;
    out->smallest_parallel_chunk_size = 16384;
}
void phastft_options_guess(size_t input_size, phastft_options* out) {
    if (!out) return;
    phastft_options_default(out);
    out->multithreaded_bit_reversal = input_size ? (ilog2(input_size) >= 16) : 0;
}

#define DEFINE_DIT_API(T, SFX)                                                                                          \
    int32_t phastft_plan_dit_##SFX##_create(size_t n, int device, int mode, phastft_plan_dit_##SFX** out) {             \
        Plan<T>* pl = nullptr;                                                                                          \
        int32_t st = (mode == PHASTFT_MODE_TUNE) ? build_plan_tuned<T>(n, device, &pl) : build_plan<T>(n, device, &pl); \
        if (out) *out = reinterpret_cast<phastft_plan_dit_##SFX*>(pl);                                                  \
        else if (pl) delete pl;                                                                                         \
        return st;                                                                                                      \
    }                                                                                                                   \
    void phastft_plan_dit_##SFX##_destroy(phastft_plan_dit_##SFX* p) { delete AS_PLAN(T, p); }                          \
    size_t phastft_plan_dit_##SFX##_size(const phastft_plan_dit_##SFX* p) { return p ? AS_CPLAN(T, p)->n : 0; }         \
    const char* phastft_plan_dit_##SFX##_describe(const phastft_plan_dit_##SFX* p) {                                    \
        return p ? AS_CPLAN(T, p)->description.c_str() : "";                                                            \
    }                                                                                                                   \
    int32_t phastft_plan_dit_##SFX##_reserve(const phastft_plan_dit_##SFX* p, size_t batch) {                           \
        return plan_reserve<T>(AS_CPLAN(T, p), batch);                                                                  \
    }                                                                                                                   \
    size_t phastft_plan_dit_##SFX##_tables_bytes(const phastft_plan_dit_##SFX* p) {                                     \
        return p ? AS_CPLAN(T, p)->blob_host.size() : 0;                                                                \
    }                                                                                                                   \
    int32_t phastft_plan_dit_##SFX##_tables_export(const phastft_plan_dit_##SFX* p, void* dst, void* s) {               \
        return tables_export<T>(AS_CPLAN(T, p), dst, (cudaStream_t)s);                                                  \
    }                                                                                                                   \
    int32_t phastft_plan_dit_##SFX##_tables_import(phastft_plan_dit_##SFX* p, const void* src, void* s) {               \
        return tables_import<T>(AS_PLAN(T, p), src, (cudaStream_t)s);                                                   \
    }                                                                                                                   \
    int32_t phastft_plan_dit_##SFX##_tables_broadcast(phastft_plan_dit_##SFX* p, void* comm, int root, void* s) {       \
        return tables_broadcast<T>(AS_PLAN(T, p), comm, root, (cudaStream_t)s);                                         \
    }                                                                                                                   \
    int32_t phastft_fft_dit_##SFX##_host(const phastft_plan_dit_##SFX* p, T* re, size_t lre, T* im, size_t lim,        \
                                         int dir, const phastft_options* opts) {                                        \
        (void)opts;                                                                                                     \
        return fft_host<T>(AS_CPLAN(T, p), re, lre, im, lim, dir);                                                      \
    }                                                                                                                   \
    int32_t phastft_fft_dit_##SFX##_oneshot(T* re, size_t lre, T* im, size_t lim, int dir, int device) {                \
        return fft_oneshot<T>(re, lre, im, lim, dir, device);                                                           \
    }                                                                                                                   \
    int32_t phastft_fft_dit_##SFX##_dev(const phastft_plan_dit_##SFX* p, T* re, T* im, int dir, size_t batch,          \
                                        size_t bstride, void* s) {                                                      \
        return fft_dev<T>(AS_CPLAN(T, p), re, im, dir, batch, bstride, (cudaStream_t)s);                                \
    }                                                                                                                   \
    int32_t phastft_fft_dit_##SFX##_dev_profile(const phastft_plan_dit_##SFX* p, T* re, T* im, int dir, size_t batch,  \
                                                size_t bstride, void* s, float* pass_ms, int* num_passes) {             \
        return fft_dev_profile<T>(AS_CPLAN(T, p), re, im, dir, batch, bstride, (cudaStream_t)s, pass_ms, num_passes);   \
    }                                                                                                                   \
    int32_t phastft_fft_dit_##SFX##_batch_sharded_host(phastft_plan_dit_##SFX* const* plans, int np, T* re, T* im,     \
                                                       size_t batch, size_t bstride, int dir) {                         \
        return batch_sharded_host<T>(reinterpret_cast<Plan<T>* const*>(plans), np, re, im, batch, bstride, dir);        \
    }                                                                                                                   \
    int32_t phastft_fft_interleaved_##SFX##_host(const phastft_plan_dit_##SFX* p, T* sig, size_t len, int dir) {        \
        return fft_interleaved_host<T>(AS_CPLAN(T, p), sig, len, dir);                                                  \
    }                                                                                                                   \
    int32_t phastft_fft_interleaved_##SFX##_dev(const phastft_plan_dit_##SFX* p, T* sig, int dir, size_t batch,        \
                                                size_t bstride, void* s) {                                              \
        return fft_interleaved_dev<T>(AS_CPLAN(T, p), sig, dir, batch, bstride, (cudaStream_t)s);                       \
    }                                                                                                                   \
    int32_t phastft_plan_r2c_##SFX##_create(size_t n, int device, phastft_plan_r2c_##SFX** out) {                       \
        PlanR2c<T>* pl = nullptr;                                                                                       \
        int32_t st = build_plan_r2c<T>(n, device, &pl);                                                                 \
        if (out) *out = reinterpret_cast<phastft_plan_r2c_##SFX*>(pl);                                                  \
        else if (pl) delete pl;                                                                                         \
        return st;                                                                                                      \
    }                                                                                                                   \
    void phastft_plan_r2c_##SFX##_destroy(phastft_plan_r2c_##SFX* p) { delete AS_R2C(T, p); }                           \
    size_t phastft_plan_r2c_##SFX##_size(const phastft_plan_r2c_##SFX* p) { return p ? AS_CR2C(T, p)->n : 0; }          \
    int32_t phastft_r2c_##SFX##_host(const phastft_plan_r2c_##SFX* p, const T* in, size_t lin, T* ore, size_t lore,    \
                                     T* oim, size_t loim) {                                                             \
        return r2c_host<T>(AS_CR2C(T, p), in, lin, ore, lore, oim, loim);                                               \
    }                                                                                                                   \
    int32_t phastft_r2c_##SFX##_oneshot(const T* in, size_t lin, T* ore, size_t lore, T* oim, size_t loim, int dev) {   \
        PlanR2c<T>* pl = nullptr; /* r2c.rs:522: PlannerR2c::new(input_re.len()), kept for the next same-size call */  \
        auto& c = oneshot_r2c_cache<T>();                                                                               \
        std::lock_guard<std::mutex> lock(c.mu);                                                                         \
        int32_t st = oneshot_r2c_plan<T>(c, lin, dev, &pl);                                                             \
        if (st) return st;                                                                                              \
        return r2c_host<T>(pl, in, lin, ore, lore, oim, loim);                                                          \
    }                                                                                                                   \
    int32_t phastft_r2c_##SFX##_dev(const phastft_plan_r2c_##SFX* p, const T* in, T* ore, T* oim, void* s) {            \
        return r2c_dev<T>(AS_CR2C(T, p), in, ore, oim, (cudaStream_t)s);                                                \
    }                                                                                                                   \
    int32_t phastft_c2r_##SFX##_host(const phastft_plan_r2c_##SFX* p, const T* ire, size_t lire, const T* iim,          \
                                     size_t liim, T* out, size_t lout, T* sre, size_t lsre, T* sim, size_t lsim) {      \
        return c2r_host<T>(AS_CR2C(T, p), ire, lire, iim, liim, out, lout, sre, lsre, sim, lsim);                       \
    }                                                                                                                   \
    int32_t phastft_c2r_##SFX##_oneshot(const T* ire, size_t lire, const T* iim, size_t liim, T* out, size_t lout,     \
                                        int dev) {                                                                      \
        PlanR2c<T>* pl = nullptr; /* r2c.rs:696: PlannerR2c::new(output.len()), kept for the next same-size call */    \
        auto& c = oneshot_r2c_cache<T>();                                                                               \
        std::lock_guard<std::mutex> lock(c.mu);                                                                         \
        int32_t st = oneshot_r2c_plan<T>(c, lout, dev, &pl);                                                            \
        if (st) return st;                                                                                              \
        return c2r_host<T>(pl, ire, lire, iim, liim, out, lout, nullptr, 0, nullptr, 0);                                \
    }                                                                                                                   \
    int32_t phastft_c2r_##SFX##_dev(const phastft_plan_r2c_##SFX* p, const T* ire, const T* iim, T* out, T* sre,        \
                                    T* sim, void* s) {                                                                  \
        return c2r_dev<T>(AS_CR2C(T, p), ire, iim, out, sre, sim, (cudaStream_t)s);                                     \
    }                                                                                                                   \
    int32_t phastft_r2c_##SFX##_dev_batch(const phastft_plan_r2c_##SFX* p, const T* in, T* ore, T* oim, size_t batch,  \
                                          size_t in_stride, size_t out_stride, void* s) {                               \
        return r2c_batch_dev<T>(AS_CR2C(T, p), in, ore, oim, batch, in_stride, out_stride, (cudaStream_t)s);            \
    }                                                                                                                   \
    int32_t phastft_c2r_##SFX##_dev_batch(const phastft_plan_r2c_##SFX* p, const T* ire, const T* iim, T* out,         \
                                          size_t batch, size_t in_stride, size_t out_stride, void* s) {                 \
        return c2r_batch_dev<T>(AS_CR2C(T, p), ire, iim, out, batch, in_stride, out_stride, (cudaStream_t)s);           \
    }                                                                                                                   \
    int32_t phastft_plan_r2c_##SFX##_reserve(const phastft_plan_r2c_##SFX* p, size_t batch) {                           \
        if (!p) return fail(PHASTFT_ERR_INVALID_ARG, "plan == NULL");                                                   \
        return plan_reserve<T>(AS_CR2C(T, p)->inner, batch, false);                                                     \
    }

DEFINE_DIT_API(double, f64)
DEFINE_DIT_API(float, f32)

}  // extern "C"
