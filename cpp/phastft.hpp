// phastft.hpp -- C++ host-side mirror of PhastFT's public API over the C ABI (include/phastft_cuda.h).
//
// The reference is compiled code (Rust) and there is no Rust toolchain in the build image, so the
// host side above the C ABI is also provided in C++: same names, argument meaning and error
// behaviour as the reference crate (src/lib.rs:143-226, src/planner.rs, src/options.rs,
// src/algorithms/r2c.rs:521-895).  Where the reference panics these throw phastft::Panic whose
// what() is the reference's panic message.  Header-only; link with -lphastft_cuda.
#pragma once

#include <cstddef>
#include <stdexcept>
#include <string>
#include <vector>

#include "../include/phastft_cuda.h"

namespace phastft {

struct Panic : std::runtime_error {
    int code;
    Panic(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

inline void check(int32_t code) {
    if (code == PHASTFT_OK) return;
    std::string msg = phastft_status_message(code);
    if (code >= PHASTFT_ERR_INVALID_ARG) { msg += ": "; msg += phastft_last_error(); }
    throw Panic(code, msg);
}

/// planner.rs:10-16
enum class Direction : int { Forward = 1, Reverse = -1 };
/// planner.rs:25-32
enum class PlannerMode : int { Heuristic = 0, Tune = 1 };   // Tune is real here (times candidate plans); the reference ignores it, planner.rs:65

/// options.rs:10-43
struct Options {
    bool multithreaded_bit_reversal = false;
    std::size_t smallest_parallel_chunk_size = 16384;
    static Options guess_options(std::size_t input_size) {
        phastft_options o;
        phastft_options_guess(input_size, &o);
        Options r;
        r.multithreaded_bit_reversal = o.multithreaded_bit_reversal != 0;
        r.smallest_parallel_chunk_size = o.smallest_parallel_chunk_size;
        return r;
    }
};

namespace detail {
template <typename T> struct Api;
template <> struct Api<double> {
    using Dit = phastft_plan_dit_f64; using R2c = phastft_plan_r2c_f64;
    static int32_t dit_create(std::size_t n, int dev, int mode, Dit** o) { return phastft_plan_dit_f64_create(n, dev, mode, o); }
    static void dit_destroy(Dit* p) { phastft_plan_dit_f64_destroy(p); }
    static std::size_t dit_size(const Dit* p) { return phastft_plan_dit_f64_size(p); }
    static const char* dit_describe(const Dit* p) { return phastft_plan_dit_f64_describe(p); }
    static int32_t dit_reserve(const Dit* p, std::size_t b) { return phastft_plan_dit_f64_reserve(p, b); }
    static int32_t fft_dev(const Dit* p, double* re, double* im, int d, std::size_t b, std::size_t st, void* s) { return phastft_fft_dit_f64_dev(p, re, im, d, b, st, s); }
    static int32_t fft_batch_host(Dit* const* ps, int np, double* re, double* im, std::size_t b, std::size_t st, int d) { return phastft_fft_dit_f64_batch_sharded_host(ps, np, re, im, b, st, d); }
    static int32_t r2c_oneshot(const double* in, std::size_t li, double* ore, std::size_t lre, double* oim, std::size_t lim) { return phastft_r2c_f64_oneshot(in, li, ore, lre, oim, lim, 0); }
    static int32_t c2r_oneshot(const double* ire, std::size_t lre, const double* iim, std::size_t lim, double* out, std::size_t lo) { return phastft_c2r_f64_oneshot(ire, lre, iim, lim, out, lo, 0); }
    static int32_t fft_host(const Dit* p, double* re, std::size_t lr, double* im, std::size_t li, int d) { return phastft_fft_dit_f64_host(p, re, lr, im, li, d, nullptr); }
    static int32_t r2c_create(std::size_t n, int dev, R2c** o) { return phastft_plan_r2c_f64_create(n, dev, o); }
    static void r2c_destroy(R2c* p) { phastft_plan_r2c_f64_destroy(p); }
    static int32_t r2c_host(const R2c* p, const double* in, std::size_t li, double* ore, std::size_t lre, double* oim, std::size_t lim) { return phastft_r2c_f64_host(p, in, li, ore, lre, oim, lim); }
    static int32_t c2r_host(const R2c* p, const double* ire, std::size_t lre, const double* iim, std::size_t lim, double* out, std::size_t lo, double* sre, std::size_t lsr, double* sim, std::size_t lsi) { return phastft_c2r_f64_host(p, ire, lre, iim, lim, out, lo, sre, lsr, sim, lsi); }
    static int32_t r2c_reserve(const R2c* p, std::size_t b) { return phastft_plan_r2c_f64_reserve(p, b); }
    static int32_t r2c_dev_batch(const R2c* p, const double* in, double* ore, double* oim, std::size_t b, std::size_t is, std::size_t os, void* s) { return phastft_r2c_f64_dev_batch(p, in, ore, oim, b, is, os, s); }
    static int32_t c2r_dev_batch(const R2c* p, const double* ire, const double* iim, double* out, std::size_t b, std::size_t is, std::size_t os, void* s) { return phastft_c2r_f64_dev_batch(p, ire, iim, out, b, is, os, s); }
};
template <> struct Api<float> {
    using Dit = phastft_plan_dit_f32; using R2c = phastft_plan_r2c_f32;
    static int32_t dit_create(std::size_t n, int dev, int mode, Dit** o) { return phastft_plan_dit_f32_create(n, dev, mode, o); }
    static void dit_destroy(Dit* p) { phastft_plan_dit_f32_destroy(p); }
    static std::size_t dit_size(const Dit* p) { return phastft_plan_dit_f32_size(p); }
    static const char* dit_describe(const Dit* p) { return phastft_plan_dit_f32_describe(p); }
    static int32_t dit_reserve(const Dit* p, std::size_t b) { return phastft_plan_dit_f32_reserve(p, b); }
    static int32_t fft_dev(const Dit* p, float* re, float* im, int d, std::size_t b, std::size_t st, void* s) { return phastft_fft_dit_f32_dev(p, re, im, d, b, st, s); }
    static int32_t fft_batch_host(Dit* const* ps, int np, float* re, float* im, std::size_t b, std::size_t st, int d) { return phastft_fft_dit_f32_batch_sharded_host(ps, np, re, im, b, st, d); }
    static int32_t r2c_oneshot(const float* in, std::size_t li, float* ore, std::size_t lre, float* oim, std::size_t lim) { return phastft_r2c_f32_oneshot(in, li, ore, lre, oim, lim, 0); }
    static int32_t c2r_oneshot(const float* ire, std::size_t lre, const float* iim, std::size_t lim, float* out, std::size_t lo) { return phastft_c2r_f32_oneshot(ire, lre, iim, lim, out, lo, 0); }
    static int32_t fft_host(const Dit* p, float* re, std::size_t lr, float* im, std::size_t li, int d) { return phastft_fft_dit_f32_host(p, re, lr, im, li, d, nullptr); }
    static int32_t r2c_create(std::size_t n, int dev, R2c** o) { return phastft_plan_r2c_f32_create(n, dev, o); }
    static void r2c_destroy(R2c* p) { phastft_plan_r2c_f32_destroy(p); }
    static int32_t r2c_host(const R2c* p, const float* in, std::size_t li, float* ore, std::size_t lre, float* oim, std::size_t lim) { return phastft_r2c_f32_host(p, in, li, ore, lre, oim, lim); }
    static int32_t c2r_host(const R2c* p, const float* ire, std::size_t lre, const float* iim, std::size_t lim, float* out, std::size_t lo, float* sre, std::size_t lsr, float* sim, std::size_t lsi) { return phastft_c2r_f32_host(p, ire, lre, iim, lim, out, lo, sre, lsr, sim, lsi); }
    static int32_t r2c_reserve(const R2c* p, std::size_t b) { return phastft_plan_r2c_f32_reserve(p, b); }
    static int32_t r2c_dev_batch(const R2c* p, const float* in, float* ore, float* oim, std::size_t b, std::size_t is, std::size_t os, void* s) { return phastft_r2c_f32_dev_batch(p, in, ore, oim, b, is, os, s); }
    static int32_t c2r_dev_batch(const R2c* p, const float* ire, const float* iim, float* out, std::size_t b, std::size_t is, std::size_t os, void* s) { return phastft_c2r_f32_dev_batch(p, ire, iim, out, b, is, os, s); }
};

/// planner.rs:34-114
template <typename T>
class PlannerDit {
  public:
    explicit PlannerDit(std::size_t num_points, int device = 0) : PlannerDit(num_points, PlannerMode::Heuristic, device) {}
    PlannerDit(std::size_t num_points, PlannerMode mode, int device = 0) { check(Api<T>::dit_create(num_points, device, (int)mode, &raw_)); }
    static PlannerDit with_mode(std::size_t num_points, PlannerMode mode) { return PlannerDit(num_points, mode); }
    ~PlannerDit() { if (raw_) Api<T>::dit_destroy(raw_); }
    PlannerDit(PlannerDit&& o) noexcept : raw_(o.raw_) { o.raw_ = nullptr; }
    PlannerDit(const PlannerDit&) = delete;
    PlannerDit& operator=(const PlannerDit&) = delete;
    const typename Api<T>::Dit* raw() const { return raw_; }
    typename Api<T>::Dit* raw_mut() const { return raw_; }
    std::size_t num_points() const { return Api<T>::dit_size(raw_); }
    /// additive: the pass decomposition and kernels the planner chose
    std::string describe() const { return Api<T>::dit_describe(raw_); }
    /// additive: size the device workspace for calls of up to `batch` transforms now
    void reserve(std::size_t batch) const { check(Api<T>::dit_reserve(raw_, batch)); }
  private:
    typename Api<T>::Dit* raw_ = nullptr;
};

/// planner.rs:164-212
template <typename T>
class PlannerR2c {
  public:
    explicit PlannerR2c(std::size_t n, int device = 0) { check(Api<T>::r2c_create(n, device, &raw_)); }
    ~PlannerR2c() { if (raw_) Api<T>::r2c_destroy(raw_); }
    PlannerR2c(PlannerR2c&& o) noexcept : raw_(o.raw_) { o.raw_ = nullptr; }
    PlannerR2c(const PlannerR2c&) = delete;
    PlannerR2c& operator=(const PlannerR2c&) = delete;
    const typename Api<T>::R2c* raw() const { return raw_; }
    /// additive: size the half-length transform's workspace for batched calls of up to `batch` members now
    void reserve(std::size_t batch) const { check(Api<T>::r2c_reserve(raw_, batch)); }
  private:
    typename Api<T>::R2c* raw_ = nullptr;
};
}  // namespace detail

using PlannerDit64 = detail::PlannerDit<double>;
using PlannerDit32 = detail::PlannerDit<float>;
using PlannerR2c64 = detail::PlannerR2c<double>;
using PlannerR2c32 = detail::PlannerR2c<float>;

// ---- c2c (lib.rs:143-226, algorithms/dit.rs:263,338): in place on planar vectors -----------------------
inline void fft_64_dit_with_planner_and_opts(std::vector<double>& reals, std::vector<double>& imags, Direction d, const PlannerDit64& p, const Options&) {
    check(detail::Api<double>::fft_host(p.raw(), reals.data(), reals.size(), imags.data(), imags.size(), (int)d));
}
inline void fft_64_dit_with_planner(std::vector<double>& reals, std::vector<double>& imags, Direction d, const PlannerDit64& p) {
    fft_64_dit_with_planner_and_opts(reals, imags, d, p, Options::guess_options(reals.size()));
}
inline void fft_64_dit(std::vector<double>& reals, std::vector<double>& imags, Direction d) {
    // lib.rs:181: a planner per call; the library keeps the latest one for the next same-size call
    check(phastft_fft_dit_f64_oneshot(reals.data(), reals.size(), imags.data(), imags.size(), (int)d, 0));
}
inline void fft_32_dit_with_planner_and_opts(std::vector<float>& reals, std::vector<float>& imags, Direction d, const PlannerDit32& p, const Options&) {
    check(detail::Api<float>::fft_host(p.raw(), reals.data(), reals.size(), imags.data(), imags.size(), (int)d));
}
inline void fft_32_dit_with_planner(std::vector<float>& reals, std::vector<float>& imags, Direction d, const PlannerDit32& p) {
    fft_32_dit_with_planner_and_opts(reals, imags, d, p, Options::guess_options(reals.size()));
}
inline void fft_32_dit(std::vector<float>& reals, std::vector<float>& imags, Direction d) {
    check(phastft_fft_dit_f32_oneshot(reals.data(), reals.size(), imags.data(), imags.size(), (int)d, 0));
}

// ---- additive: batches and device-resident data (the reference's batch is a caller loop sharing one planner,
// examples/benchmark.rs:24-36; here it is one call) -------------------------------------------------------------
template <typename T>
inline void fft_dit_batch(std::vector<T>& reals, std::vector<T>& imags, Direction d, const detail::PlannerDit<T>& p, std::size_t batch, std::size_t batch_stride) {
    if (reals.size() != imags.size()) check(1);
    const std::size_t n = p.num_points();
    if (batch_stride < n || (batch && reals.size() < (batch - 1) * batch_stride + n)) check(13);
    typename detail::Api<T>::Dit* one[1] = {p.raw_mut()};
    check(detail::Api<T>::fft_batch_host(one, 1, reals.data(), imags.data(), batch, batch_stride, (int)d));
}
inline void fft_64_dit_batch(std::vector<double>& re, std::vector<double>& im, Direction d, const PlannerDit64& p, std::size_t batch, std::size_t stride) { fft_dit_batch<double>(re, im, d, p, batch, stride); }
inline void fft_32_dit_batch(std::vector<float>& re, std::vector<float>& im, Direction d, const PlannerDit32& p, std::size_t batch, std::size_t stride) { fft_dit_batch<float>(re, im, d, p, batch, stride); }
/// Device pointers on the planner's device; stream-ordered on `stream` (cudaStream_t, nullptr = default stream), no allocation, no host sync.
inline void fft_64_dit_device(double* d_reals, double* d_imags, Direction d, const PlannerDit64& p, std::size_t batch, std::size_t batch_stride, void* stream) {
    check(detail::Api<double>::fft_dev(p.raw(), d_reals, d_imags, (int)d, batch, batch_stride, stream));
}
inline void fft_32_dit_device(float* d_reals, float* d_imags, Direction d, const PlannerDit32& p, std::size_t batch, std::size_t batch_stride, void* stream) {
    check(detail::Api<float>::fft_dev(p.raw(), d_reals, d_imags, (int)d, batch, batch_stride, stream));
}
/// Batched device-resident r2c / c2r (phastft_{r2c,c2r}_*_dev_batch): strides in elements; the real-side stride even and
/// its base aligned to two elements.
inline void r2c_fft_f64_device_batch(const double* d_in, double* d_out_re, double* d_out_im, const PlannerR2c64& p, std::size_t batch, std::size_t in_stride, std::size_t out_stride, void* stream) {
    check(detail::Api<double>::r2c_dev_batch(p.raw(), d_in, d_out_re, d_out_im, batch, in_stride, out_stride, stream));
}
inline void r2c_fft_f32_device_batch(const float* d_in, float* d_out_re, float* d_out_im, const PlannerR2c32& p, std::size_t batch, std::size_t in_stride, std::size_t out_stride, void* stream) {
    check(detail::Api<float>::r2c_dev_batch(p.raw(), d_in, d_out_re, d_out_im, batch, in_stride, out_stride, stream));
}
inline void c2r_fft_f64_device_batch(const double* d_in_re, const double* d_in_im, double* d_out, const PlannerR2c64& p, std::size_t batch, std::size_t in_stride, std::size_t out_stride, void* stream) {
    check(detail::Api<double>::c2r_dev_batch(p.raw(), d_in_re, d_in_im, d_out, batch, in_stride, out_stride, stream));
}
inline void c2r_fft_f32_device_batch(const float* d_in_re, const float* d_in_im, float* d_out, const PlannerR2c32& p, std::size_t batch, std::size_t in_stride, std::size_t out_stride, void* stream) {
    check(detail::Api<float>::c2r_dev_batch(p.raw(), d_in_re, d_in_im, d_out, batch, in_stride, out_stride, stream));
}

// ---- r2c / c2r (algorithms/r2c.rs:521-895) --------------------------------------------------------------
inline void r2c_fft_f64_with_planner(const std::vector<double>& in, std::vector<double>& ore, std::vector<double>& oim, const PlannerR2c64& p) {
    check(detail::Api<double>::r2c_host(p.raw(), in.data(), in.size(), ore.data(), ore.size(), oim.data(), oim.size()));
}
inline void r2c_fft_f64(const std::vector<double>& in, std::vector<double>& ore, std::vector<double>& oim) {
    // r2c.rs:522: a planner per call; the library keeps the latest one for the next same-size call
    check(detail::Api<double>::r2c_oneshot(in.data(), in.size(), ore.data(), ore.size(), oim.data(), oim.size()));
}
inline void c2r_fft_f64_with_planner_and_scratch(const std::vector<double>& ire, const std::vector<double>& iim, std::vector<double>& out,
                                                 const PlannerR2c64& p, std::vector<double>& sre, std::vector<double>& sim) {
    check(detail::Api<double>::c2r_host(p.raw(), ire.data(), ire.size(), iim.data(), iim.size(), out.data(), out.size(), sre.data(), sre.size(), sim.data(), sim.size()));
}
inline void c2r_fft_f64_with_planner(const std::vector<double>& ire, const std::vector<double>& iim, std::vector<double>& out, const PlannerR2c64& p) {
    check(detail::Api<double>::c2r_host(p.raw(), ire.data(), ire.size(), iim.data(), iim.size(), out.data(), out.size(), nullptr, 0, nullptr, 0));
}
inline void c2r_fft_f64(const std::vector<double>& ire, const std::vector<double>& iim, std::vector<double>& out) {
    check(detail::Api<double>::c2r_oneshot(ire.data(), ire.size(), iim.data(), iim.size(), out.data(), out.size()));
}
inline void r2c_fft_f32_with_planner(const std::vector<float>& in, std::vector<float>& ore, std::vector<float>& oim, const PlannerR2c32& p) {
    check(detail::Api<float>::r2c_host(p.raw(), in.data(), in.size(), ore.data(), ore.size(), oim.data(), oim.size()));
}
inline void r2c_fft_f32(const std::vector<float>& in, std::vector<float>& ore, std::vector<float>& oim) {
    check(detail::Api<float>::r2c_oneshot(in.data(), in.size(), ore.data(), ore.size(), oim.data(), oim.size()));
}
inline void c2r_fft_f32_with_planner_and_scratch(const std::vector<float>& ire, const std::vector<float>& iim, std::vector<float>& out,
                                                 const PlannerR2c32& p, std::vector<float>& sre, std::vector<float>& sim) {
    check(detail::Api<float>::c2r_host(p.raw(), ire.data(), ire.size(), iim.data(), iim.size(), out.data(), out.size(), sre.data(), sre.size(), sim.data(), sim.size()));
}
inline void c2r_fft_f32_with_planner(const std::vector<float>& ire, const std::vector<float>& iim, std::vector<float>& out, const PlannerR2c32& p) {
    check(detail::Api<float>::c2r_host(p.raw(), ire.data(), ire.size(), iim.data(), iim.size(), out.data(), out.size(), nullptr, 0, nullptr, 0));
}
inline void c2r_fft_f32(const std::vector<float>& ire, const std::vector<float>& iim, std::vector<float>& out) {
    check(detail::Api<float>::c2r_oneshot(ire.data(), ire.size(), iim.data(), iim.size(), out.data(), out.size()));
}

}  // namespace phastft
