/*
 * phastft_cuda.h -- C ABI of libphastft_cuda.so, the B200 (sm_100a) drop-in for PhastFT's
 * 1-D power-of-two FFT path.
 *
 * The reference (QuState/PhastFT @ 8cd3a39) has no FFI boundary: the path sits behind its
 * public Rust API.  Each entry point below names the reference item it stands in for; the
 * thin Rust wrappers that keep the reference's names and panics are in rust/src/lib.rs, the
 * C++ and Python mirrors in cpp/phastft.hpp and phastft_b200/api.py (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns a phastft_status (int32_t), never
 *     aborts, never throws; phastft_last_error() gives a thread-local detail string.
 *   - planar data: separate re[] and im[] arrays of T, natural order in and out
 *     (README.md:174-178 of the reference); forward unscaled, reverse scaled by 1/N
 *     (algorithms/dit.rs:297-331).
 *   - `*_host` entry points take HOST pointers and are synchronous and in place from the
 *     caller's view (API parity with the Rust slices).  `*_dev` entry points take DEVICE
 *     pointers, enqueue on the given cudaStream_t (passed as void*), allocate nothing and do
 *     not synchronise: these are what bench.py's device-resident number measures.
 *   - plans are immutable after creation and may be shared between host threads (the Rust
 *     planners are Send + Sync); calls on one plan serialise on the plan's internal workspace.
 *   - there is NO CPU fallback: without a CUDA device every call returns PHASTFT_ERR_NO_DEVICE.
 */
#ifndef PHASTFT_CUDA_H
#define PHASTFT_CUDA_H

#include <stddef.h>
#include <stdint.h>

#include "phastft_status.h"

#ifdef __cplusplus
extern "C" {
#endif

#define PHASTFT_API __attribute__((visibility("default")))

/* ---- library -------------------------------------------------------------------------- */
PHASTFT_API const char* phastft_last_error(void);            /* thread-local, never NULL */
PHASTFT_API const char* phastft_version(void);
PHASTFT_API int32_t phastft_device_count(int* count);
/* number of CUDA kernels this library has launched in this process (bench.py "gpu_launches") */
PHASTFT_API uint64_t phastft_launch_count(void);
/* The *_oneshot entry points (a planner per call, lib.rs:180 / r2c.rs:522,696) keep their most recent plan per
 * precision and reuse it when the next call has the same size and device; this releases those plans and their
 * device buffers. */
PHASTFT_API void phastft_oneshot_cache_clear(void);
/* Page-lock / release a caller-owned host range (cudaHostRegister / cudaHostUnregister).  The *_host entry points
 * accept any host memory, but copies from ordinary pageable memory run at ~13 GB/s against ~52 GB/s from page-locked
 * memory (profiles/r01_host_call_cost.txt), and the batched host pipeline only overlaps with page-locked memory.
 * Register long-lived buffers once; registration itself costs about as much as several copies. */
PHASTFT_API int32_t phastft_host_register(void* host_ptr, size_t bytes);
PHASTFT_API int32_t phastft_host_unregister(void* host_ptr);

/* ---- options.rs:10-43 : Options / guess_options ------------------------------------------
 * Kept for source compatibility.  On the GPU both fields are hints with no effect: there is
 * no separate bit-reversal step to thread and the grid is always full-chip parallel. */
typedef struct phastft_options {
    int32_t multithreaded_bit_reversal;     /* options.rs:16 */
    size_t smallest_parallel_chunk_size;    /* options.rs:23, default 16384 */
} phastft_options;
PHASTFT_API void phastft_options_default(phastft_options* out);            /* options.rs:26-33 */
PHASTFT_API void phastft_options_guess(size_t input_size, phastft_options* out); /* options.rs:38-43 */

/* ---- planner.rs:25-32 PlannerMode ------------------------------------------------------ */
#define PHASTFT_MODE_HEURISTIC 0
#define PHASTFT_MODE_TUNE 1   /* times a few pass decompositions / tile widths at plan time and keeps the fastest
                                 (the reference accepts the mode and ignores it, planner.rs:65) */

/* ---- planner.rs:34-114 : PlannerDit64 / PlannerDit32 -------------------------------------
 * num_points must be a non-zero power of two (planner.rs:66) else PHASTFT_ERR_NOT_POW2.
 * The plan owns the device twiddle tables (two-level W_N table + per-pass W_R tables) and,
 * lazily, a device workspace of N complex elements (multi-pass sizes only). */
typedef struct phastft_plan_dit_f64 phastft_plan_dit_f64;
typedef struct phastft_plan_dit_f32 phastft_plan_dit_f32;
PHASTFT_API int32_t phastft_plan_dit_f64_create(size_t num_points, int device, int mode, phastft_plan_dit_f64** out);
PHASTFT_API int32_t phastft_plan_dit_f32_create(size_t num_points, int device, int mode, phastft_plan_dit_f32** out);
PHASTFT_API void phastft_plan_dit_f64_destroy(phastft_plan_dit_f64* plan);
PHASTFT_API void phastft_plan_dit_f32_destroy(phastft_plan_dit_f32* plan);
PHASTFT_API size_t phastft_plan_dit_f64_size(const phastft_plan_dit_f64* plan);
PHASTFT_API size_t phastft_plan_dit_f32_size(const phastft_plan_dit_f32* plan);
/* Human-readable pass decomposition, e.g. "n=2^20 f64: COL R=1024 C=8 | TRANS R=1024 C=8". */
PHASTFT_API const char* phastft_plan_dit_f64_describe(const phastft_plan_dit_f64* plan);
PHASTFT_API const char* phastft_plan_dit_f32_describe(const phastft_plan_dit_f32* plan);

/* Sizes the plan's device workspace for calls of up to `batch` transforms now (the *_dev entry points otherwise
 * grow it on the first larger call, which synchronises the device and is an error inside a CUDA-graph capture). */
PHASTFT_API int32_t phastft_plan_dit_f64_reserve(const phastft_plan_dit_f64* plan, size_t batch);
PHASTFT_API int32_t phastft_plan_dit_f32_reserve(const phastft_plan_dit_f32* plan, size_t batch);

/* Host-only planning logic (no device needed): the pass decomposition N = 2^f0 * 2^f1 [* 2^f2] the
 * planner uses for `num_points` (one CTA per transform when *num_passes == 1; 0 passes for N == 1).
 * log2_factors must hold 3 ints. */
PHASTFT_API int32_t phastft_plan_factorization(size_t num_points, int precision_bits, int* log2_factors, int* num_passes);

/* Planner-table blob (multi-GPU init, SURVEY.md section 8e): rank 0 exports its tables into a
 * device buffer, the host framework broadcasts that buffer once (ncclBroadcast /
 * torch.distributed.broadcast), every other rank imports it.  No per-call collectives.
 * The blob starts with a 256-byte layout header (size, precision, pass sizes, each pass's tile width and first
 * radix): import / broadcast return PHASTFT_ERR_PLAN_MISMATCH when the receiving plan was built with a different
 * decomposition (PlannerMode::Tune or a PHASTFT_* override on one rank only) instead of installing foreign tables. */
PHASTFT_API size_t phastft_plan_dit_f64_tables_bytes(const phastft_plan_dit_f64* plan);
PHASTFT_API size_t phastft_plan_dit_f32_tables_bytes(const phastft_plan_dit_f32* plan);
PHASTFT_API int32_t phastft_plan_dit_f64_tables_export(const phastft_plan_dit_f64* plan, void* dst_dev, void* stream);
PHASTFT_API int32_t phastft_plan_dit_f32_tables_export(const phastft_plan_dit_f32* plan, void* dst_dev, void* stream);
PHASTFT_API int32_t phastft_plan_dit_f64_tables_import(phastft_plan_dit_f64* plan, const void* src_dev, void* stream);
PHASTFT_API int32_t phastft_plan_dit_f32_tables_import(phastft_plan_dit_f32* plan, const void* src_dev, void* stream);
/* Native NCCL path for the same broadcast: `comm` is an ncclComm_t created by the caller;
 * libnccl.so.2 is dlopen()ed on first use (PHASTFT_ERR_NCCL if absent). */
PHASTFT_API int32_t phastft_plan_dit_f64_tables_broadcast(phastft_plan_dit_f64* plan, void* nccl_comm, int root, void* stream);
PHASTFT_API int32_t phastft_plan_dit_f32_tables_broadcast(phastft_plan_dit_f32* plan, void* nccl_comm, int root, void* stream);

/* ---- lib.rs:143-226, algorithms/dit.rs:263-401 : fft_64_dit* / fft_32_dit* ----------------
 * Host-slice execution: fft_{64,32}_dit_with_planner[_and_opts](reals, imags, direction, planner[, opts]).
 * len_re / len_im are the slice lengths; the reference's asserts map to
 *   len_re != len_im -> PHASTFT_ERR_LEN_MISMATCH, not a power of two -> PHASTFT_ERR_NOT_POW2,
 *   log2(len) != plan -> PHASTFT_ERR_PLAN_MISMATCH.
 * `opts` may be NULL (= guess_options(len), lib.rs:149). */
PHASTFT_API int32_t phastft_fft_dit_f64_host(const phastft_plan_dit_f64* plan, double* reals, size_t len_re,
                                             double* imags, size_t len_im, int direction, const phastft_options* opts);
PHASTFT_API int32_t phastft_fft_dit_f32_host(const phastft_plan_dit_f32* plan, float* reals, size_t len_re,
                                             float* imags, size_t len_im, int direction, const phastft_options* opts);
/* fft_64_dit / fft_32_dit (lib.rs:180, 223): plans per call on `device`, like the reference. */
PHASTFT_API int32_t phastft_fft_dit_f64_oneshot(double* reals, size_t len_re, double* imags, size_t len_im,
                                                int direction, int device);
PHASTFT_API int32_t phastft_fft_dit_f32_oneshot(float* reals, size_t len_re, float* imags, size_t len_im,
                                                int direction, int device);

/* Device-resident execution (batched): `batch` transforms, transform b at d_re + b*batch_stride
 * (batch_stride >= N elements; the reference has no batch API -- a batch is a caller loop over
 * fft_32_dit_with_planner sharing one planner, examples/benchmark.rs:24-36).  In place. */
PHASTFT_API int32_t phastft_fft_dit_f64_dev(const phastft_plan_dit_f64* plan, double* d_reals, double* d_imags,
                                            int direction, size_t batch, size_t batch_stride, void* stream);
PHASTFT_API int32_t phastft_fft_dit_f32_dev(const phastft_plan_dit_f32* plan, float* d_reals, float* d_imags,
                                            int direction, size_t batch, size_t batch_stride, void* stream);
/* Profiling aid (bench.py's roofline): same as *_dev, but records CUDA events on `stream` around
 * every pass (kernel launch) of the first L2 chunk, synchronises, and returns the per-pass device
 * times in milliseconds (pass_ms must hold 3 floats). */
PHASTFT_API int32_t phastft_fft_dit_f64_dev_profile(const phastft_plan_dit_f64* plan, double* d_reals, double* d_imags,
                                                    int direction, size_t batch, size_t batch_stride, void* stream,
                                                    float* pass_ms, int* num_passes);
PHASTFT_API int32_t phastft_fft_dit_f32_dev_profile(const phastft_plan_dit_f32* plan, float* d_reals, float* d_imags,
                                                    int direction, size_t batch, size_t batch_stride, void* stream,
                                                    float* pass_ms, int* num_passes);
/* Host-slice batched execution sharded over devices (SURVEY.md section 8e): transforms
 * [g*batch/G, (g+1)*batch/G) run on plans[g] (one plan per device, tables made identical by the
 * init-time broadcast).  Synchronous. */
PHASTFT_API int32_t phastft_fft_dit_f32_batch_sharded_host(phastft_plan_dit_f32* const* plans, int num_plans,
                                                           float* reals, float* imags, size_t batch,
                                                           size_t batch_stride, int direction);
PHASTFT_API int32_t phastft_fft_dit_f64_batch_sharded_host(phastft_plan_dit_f64* const* plans, int num_plans,
                                                           double* reals, double* imags, size_t batch,
                                                           size_t batch_stride, int direction);

/* ---- planner.rs:164-212 : PlannerR2c64 / PlannerR2c32 -------------------------------------
 * n must be a power of two >= 4 else PHASTFT_ERR_R2C_N ("n must be a power of 2 >= 4"). */
typedef struct phastft_plan_r2c_f64 phastft_plan_r2c_f64;
typedef struct phastft_plan_r2c_f32 phastft_plan_r2c_f32;
PHASTFT_API int32_t phastft_plan_r2c_f64_create(size_t n, int device, phastft_plan_r2c_f64** out);
PHASTFT_API int32_t phastft_plan_r2c_f32_create(size_t n, int device, phastft_plan_r2c_f32** out);
PHASTFT_API void phastft_plan_r2c_f64_destroy(phastft_plan_r2c_f64* plan);
PHASTFT_API void phastft_plan_r2c_f32_destroy(phastft_plan_r2c_f32* plan);
PHASTFT_API size_t phastft_plan_r2c_f64_size(const phastft_plan_r2c_f64* plan);
PHASTFT_API size_t phastft_plan_r2c_f32_size(const phastft_plan_r2c_f32* plan);

/* ---- algorithms/r2c.rs:521-662 : r2c_fft_{f64,f32}[_with_planner] --------------------------
 * input (length N, not modified) -> output_re/output_im (length N/2+1 each).  Length checks in
 * the reference's order (r2c.rs:543-553). */
PHASTFT_API int32_t phastft_r2c_f64_host(const phastft_plan_r2c_f64* plan, const double* input, size_t len_in,
                                         double* output_re, size_t len_ore, double* output_im, size_t len_oim);
PHASTFT_API int32_t phastft_r2c_f32_host(const phastft_plan_r2c_f32* plan, const float* input, size_t len_in,
                                         float* output_re, size_t len_ore, float* output_im, size_t len_oim);
/* r2c_fft_f64 / r2c_fft_f32 (r2c.rs:521, 598): plans per call. */
PHASTFT_API int32_t phastft_r2c_f64_oneshot(const double* input, size_t len_in, double* output_re, size_t len_ore,
                                            double* output_im, size_t len_oim, int device);
PHASTFT_API int32_t phastft_r2c_f32_oneshot(const float* input, size_t len_in, float* output_re, size_t len_ore,
                                            float* output_im, size_t len_oim, int device);
/* Device-resident: d_input N reals, d_out_re/d_out_im N/2+1 each; asynchronous on `stream`. */
PHASTFT_API int32_t phastft_r2c_f64_dev(const phastft_plan_r2c_f64* plan, const double* d_input, double* d_out_re,
                                        double* d_out_im, void* stream);
PHASTFT_API int32_t phastft_r2c_f32_dev(const phastft_plan_r2c_f32* plan, const float* d_input, float* d_out_re,
                                        float* d_out_im, void* stream);

/* ---- algorithms/r2c.rs:695-895 : c2r_fft_{f64,f32}[_with_planner[_and_scratch]] -------------
 * input_re/input_im (N/2+1 each, not modified) -> output (N reals), fully normalised so that
 * c2r(r2c(x)) == x.  scratch_re/scratch_im: caller scratch of N/2 each, or both NULL with
 * len 0 to let the plan use its own device workspace (the reference's allocating variants,
 * r2c.rs:716-718).  Host scratch is only length-checked (r2c.rs:761-762): the work happens in
 * device memory. */
PHASTFT_API int32_t phastft_c2r_f64_host(const phastft_plan_r2c_f64* plan, const double* input_re, size_t len_ire,
                                         const double* input_im, size_t len_iim, double* output, size_t len_out,
                                         double* scratch_re, size_t len_sre, double* scratch_im, size_t len_sim);
PHASTFT_API int32_t phastft_c2r_f32_host(const phastft_plan_r2c_f32* plan, const float* input_re, size_t len_ire,
                                         const float* input_im, size_t len_iim, float* output, size_t len_out,
                                         float* scratch_re, size_t len_sre, float* scratch_im, size_t len_sim);
PHASTFT_API int32_t phastft_c2r_f64_oneshot(const double* input_re, size_t len_ire, const double* input_im,
                                            size_t len_iim, double* output, size_t len_out, int device);
PHASTFT_API int32_t phastft_c2r_f32_oneshot(const float* input_re, size_t len_ire, const float* input_im,
                                            size_t len_iim, float* output, size_t len_out, int device);
/* Device-resident: d_scratch_re/d_scratch_im N/2 each or both NULL (plan workspace). */
PHASTFT_API int32_t phastft_c2r_f64_dev(const phastft_plan_r2c_f64* plan, const double* d_in_re, const double* d_in_im,
                                        double* d_output, double* d_scratch_re, double* d_scratch_im, void* stream);
PHASTFT_API int32_t phastft_c2r_f32_dev(const phastft_plan_r2c_f32* plan, const float* d_in_re, const float* d_in_im,
                                        float* d_output, float* d_scratch_re, float* d_scratch_im, void* stream);

/* ---- batched device-resident r2c / c2r (the reference has no batch API: a caller loop sharing one planner) --------
 * Strides are in elements of T.
 *   r2c: member b reads d_input[b*in_stride ..][..N] and writes bins [b*out_stride ..][..N/2+1] of both output planes
 *        (in_stride >= N, out_stride >= N/2+1).
 *   c2r: member b reads bins [b*in_stride ..][..N/2+1] of both input planes and writes d_output[b*out_stride ..][..N]
 *        (in_stride >= N/2+1, out_stride >= N), normalised as phastft_c2r_*_dev.
 * The real side is read or written as complex pairs: its stride must be even and its base pointer aligned to
 * 2*sizeof(T), else PHASTFT_ERR_INVALID_ARG before anything is launched.  Padding between members and the spectrum input
 * of c2r are never written.  Stream-ordered and asynchronous like the single-call entries, which batch == 1 runs.  No
 * scratch: every batched c2r pre-processes the spectrum while its first kernel loads it.  Any batch count. */
PHASTFT_API int32_t phastft_r2c_f64_dev_batch(const phastft_plan_r2c_f64* plan, const double* d_input, double* d_out_re,
                                              double* d_out_im, size_t batch, size_t in_stride, size_t out_stride, void* stream);
PHASTFT_API int32_t phastft_r2c_f32_dev_batch(const phastft_plan_r2c_f32* plan, const float* d_input, float* d_out_re,
                                              float* d_out_im, size_t batch, size_t in_stride, size_t out_stride, void* stream);
PHASTFT_API int32_t phastft_c2r_f64_dev_batch(const phastft_plan_r2c_f64* plan, const double* d_in_re, const double* d_in_im,
                                              double* d_output, size_t batch, size_t in_stride, size_t out_stride, void* stream);
PHASTFT_API int32_t phastft_c2r_f32_dev_batch(const phastft_plan_r2c_f32* plan, const float* d_in_re, const float* d_in_im,
                                              float* d_output, size_t batch, size_t in_stride, size_t out_stride, void* stream);
/* Sizes the workspace of the plan's half-length transform for batches of up to `batch` members now, as
 * phastft_plan_dit_*_reserve does: a batched r2c / c2r can then be captured into a CUDA graph.  (With the opt-in
 * pipelined two-pass launch, PHASTFT_PIPE=1, that launch's per-call counters are still allocated by the first
 * uncaptured call, for c2c and r2c alike.) */
PHASTFT_API int32_t phastft_plan_r2c_f64_reserve(const phastft_plan_r2c_f64* plan, size_t batch);
PHASTFT_API int32_t phastft_plan_r2c_f32_reserve(const phastft_plan_r2c_f32* plan, size_t batch);

/* ---- lib.rs:41-140 (feature complex-nums): fft_{64,32}_interleaved* --------------------------
 * signal = N interleaved (re, im) pairs (num_complex::Complex<T> layout), in place.  The
 * reference deinterleaves into two fresh Vecs, runs the planar FFT and re-interleaves
 * (complex_nums.rs:11-55); here the AoS<->planar conversion is fused into the first pass's
 * load and the last pass's store. */
PHASTFT_API int32_t phastft_fft_interleaved_f64_host(const phastft_plan_dit_f64* plan, double* signal, size_t len_complex,
                                                     int direction);
PHASTFT_API int32_t phastft_fft_interleaved_f32_host(const phastft_plan_dit_f32* plan, float* signal, size_t len_complex,
                                                     int direction);
PHASTFT_API int32_t phastft_fft_interleaved_f64_dev(const phastft_plan_dit_f64* plan, double* d_signal, int direction,
                                                    size_t batch, size_t batch_stride_complex, void* stream);
PHASTFT_API int32_t phastft_fft_interleaved_f32_dev(const phastft_plan_dit_f32* plan, float* d_signal, int direction,
                                                    size_t batch, size_t batch_stride_complex, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PHASTFT_CUDA_H */
