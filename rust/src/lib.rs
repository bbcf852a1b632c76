//! PhastFT's public API, unchanged, over `libphastft_cuda.so` (B200 / sm_100a).
//!
//! Every item below keeps the name, signature and panic behaviour of the reference crate
//! (QuState/PhastFT @ 8cd3a39; the `file:line` in each doc comment is the item it replaces), so a user
//! switches by changing the dependency, not the call sites:
//!
//! ```ignore
//! use phastft::{fft_64_dit, planner::Direction};
//! let mut reals = vec![1.0, 0.0, 0.0, 0.0];
//! let mut imags = vec![0.0; 4];
//! fft_64_dit(&mut reals, &mut imags, Direction::Forward);   // runs on cuda:0
//! ```
//!
//! The wrappers are deliberately thin: length checks that the reference performs with `assert!` happen
//! inside the C ABI, which returns a status code; `check()` turns a non-zero code back into a `panic!`
//! carrying the reference's message, so `#[should_panic(expected = "...")]` tests carry over.
//! The device is chosen with the `PHASTFT_DEVICE` environment variable (default 0).
pub mod ffi;
pub mod options;
pub mod planner;

use options::Options;
use planner::{Direction, PlannerDit32, PlannerDit64, PlannerR2c32, PlannerR2c64};

/// Reference panic texts by status code (include/phastft_status.h).
#[track_caller]
pub(crate) fn check(code: i32) {
    let msg = match code {
        0 => return,
        1 => "assertion `left == right` failed: reals.len() == imags.len()",
        2 => "assertion failed: length must be a non-zero power of two",
        3 => "assertion `left == right` failed: log_n == planner.log_n",
        4 => "n must be a power of 2 >= 4",
        5 => "input length must match planner size",
        6 => "output_re must have length N/2 + 1",
        7 => "output_im must have length N/2 + 1",
        8 => "output length must match planner size",
        9 => "input_re must have length N/2 + 1",
        10 => "input_im must have length N/2 + 1",
        11 => "scratch_re must have length N/2",
        12 => "scratch_im must have length N/2",
        _ => {
            let detail = unsafe { std::ffi::CStr::from_ptr(ffi::phastft_last_error()) }.to_string_lossy().into_owned();
            panic!("phastft_cuda error {code}: {detail}");
        }
    };
    panic!("{msg}");
}

/// Page-lock a long-lived buffer so the host-slice calls copy at full PCIe speed (~52 GB/s instead of ~13 GB/s
/// from pageable memory). Additive: the reference has no analogue. Undo with [`host_unregister`] before the
/// buffer is freed.
pub fn host_register<T>(buf: &mut [T]) {
    check(unsafe { ffi::phastft_host_register(buf.as_mut_ptr() as *mut std::os::raw::c_void, std::mem::size_of_val(buf)) });
}
pub fn host_unregister<T>(buf: &mut [T]) {
    check(unsafe { ffi::phastft_host_unregister(buf.as_mut_ptr() as *mut std::os::raw::c_void) });
}

pub(crate) fn device() -> i32 {
    std::env::var("PHASTFT_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0)
}

fn c_opts(o: &Options) -> ffi::phastft_options {
    ffi::phastft_options {
        multithreaded_bit_reversal: o.multithreaded_bit_reversal as i32,
        smallest_parallel_chunk_size: o.smallest_parallel_chunk_size,
    }
}

// ------------------------------------------------------------------------------------------------
// c2c, planar
// ------------------------------------------------------------------------------------------------

/// `algorithms/dit.rs:263` -- in place on planar slices; panics like the reference on length
/// mismatch, non-power-of-two length, or a planner built for another size.
pub fn fft_64_dit_with_planner_and_opts(reals: &mut [f64], imags: &mut [f64], direction: Direction, planner: &PlannerDit64, opts: &Options) {
    let o = c_opts(opts);
    check(unsafe {
        ffi::phastft_fft_dit_f64_host(planner.raw, reals.as_mut_ptr(), reals.len(), imags.as_mut_ptr(), imags.len(), direction as i32, &o)
    });
}

/// `algorithms/dit.rs:338`
pub fn fft_32_dit_with_planner_and_opts(reals: &mut [f32], imags: &mut [f32], direction: Direction, planner: &PlannerDit32, opts: &Options) {
    let o = c_opts(opts);
    check(unsafe {
        ffi::phastft_fft_dit_f32_host(planner.raw, reals.as_mut_ptr(), reals.len(), imags.as_mut_ptr(), imags.len(), direction as i32, &o)
    });
}

/// `lib.rs:143`
pub fn fft_64_dit_with_planner(reals: &mut [f64], imags: &mut [f64], direction: Direction, planner: &PlannerDit64) {
    let opts = Options::guess_options(reals.len());
    fft_64_dit_with_planner_and_opts(reals, imags, direction, planner, &opts);
}

/// `lib.rs:180` -- plans per call, like the reference.
pub fn fft_64_dit(reals: &mut [f64], imags: &mut [f64], direction: Direction) {
    // a planner per call, as in the reference; the library keeps the latest one for the next same-size call
    check(unsafe {
        ffi::phastft_fft_dit_f64_oneshot(reals.as_mut_ptr(), reals.len(), imags.as_mut_ptr(), imags.len(), direction as i32, device())
    });
}

/// `lib.rs:186`
pub fn fft_32_dit_with_planner(reals: &mut [f32], imags: &mut [f32], direction: Direction, planner: &PlannerDit32) {
    let opts = Options::guess_options(reals.len());
    fft_32_dit_with_planner_and_opts(reals, imags, direction, planner, &opts);
}

/// `lib.rs:223`
pub fn fft_32_dit(reals: &mut [f32], imags: &mut [f32], direction: Direction) {
    check(unsafe {
        ffi::phastft_fft_dit_f32_oneshot(reals.as_mut_ptr(), reals.len(), imags.as_mut_ptr(), imags.len(), direction as i32, device())
    });
}

// ------------------------------------------------------------------------------------------------
// Additive: batches and device-resident data.  The reference has no batch API -- a batch is a caller loop sharing one
// planner (examples/benchmark.rs:24-36); on a GPU the loop is one call, and the data can stay in device memory.
// ------------------------------------------------------------------------------------------------

macro_rules! impl_batch {
    ($batch:ident, $sharded:ident, $device:ident, $t:ty, $planner:ident, $ffi_sharded:ident, $ffi_dev:ident) => {
        /// `batch` transforms of `planner.num_points()` points, transform `b` at `[b * batch_stride ..][.. n]` of the planar
        /// host slices, in place; equivalent to calling the `_with_planner` function on every transform.  Host memory is
        /// streamed through a three-slot H2D / FFT / D2H pipeline (page-lock it with [`host_register`] for full PCIe speed).
        pub fn $batch(reals: &mut [$t], imags: &mut [$t], direction: Direction, planner: &$planner, batch: usize, batch_stride: usize) {
            $sharded(reals, imags, direction, &[planner], batch, batch_stride);
        }
        /// The same batch sharded over several devices from one process: transforms `[g*batch/G, (g+1)*batch/G)` run on
        /// `planners[g]` (one planner per device).  No data-path collective.
        pub fn $sharded(reals: &mut [$t], imags: &mut [$t], direction: Direction, planners: &[&$planner], batch: usize, batch_stride: usize) {
            assert!(!planners.is_empty(), "at least one planner");
            let n = planners[0].num_points();
            assert_eq!(reals.len(), imags.len(), "reals.len() == imags.len()");
            assert!(batch_stride >= n && (batch == 0 || reals.len() >= (batch - 1) * batch_stride + n), "slices shorter than batch * batch_stride");
            let raw: Vec<*mut _> = planners.iter().map(|p| p.raw).collect();
            check(unsafe { ffi::$ffi_sharded(raw.as_ptr(), raw.len() as i32, reals.as_mut_ptr(), imags.as_mut_ptr(), batch, batch_stride, direction as i32) });
        }
        /// Device-resident planar data: stream-ordered on `stream` (a `cudaStream_t`, null = the default stream), no
        /// allocation, no host synchronisation.
        ///
        /// # Safety
        /// `d_reals` / `d_imags` must be device pointers valid for `(batch - 1) * batch_stride + n` elements on the
        /// planner's device, and must not be used by other work on other streams until this call's work has completed.
        pub unsafe fn $device(d_reals: *mut $t, d_imags: *mut $t, direction: Direction, planner: &$planner, batch: usize, batch_stride: usize,
                              stream: *mut std::os::raw::c_void) {
            check(ffi::$ffi_dev(planner.raw, d_reals, d_imags, direction as i32, batch, batch_stride, stream));
        }
    };
}
impl_batch!(fft_64_dit_batch, fft_64_dit_batch_sharded, fft_64_dit_device, f64, PlannerDit64, phastft_fft_dit_f64_batch_sharded_host, phastft_fft_dit_f64_dev);
impl_batch!(fft_32_dit_batch, fft_32_dit_batch_sharded, fft_32_dit_device, f32, PlannerDit32, phastft_fft_dit_f32_batch_sharded_host, phastft_fft_dit_f32_dev);

/// Number of CUDA devices the library sees (0 without a driver; every transform then panics with the NO_DEVICE message).
pub fn device_count() -> usize {
    let mut n: std::os::raw::c_int = 0;
    unsafe { ffi::phastft_device_count(&mut n) };
    n.max(0) as usize
}

/// Device-resident real transforms (`r2c.rs:535`, `:740` on device pointers).
///
/// # Safety
/// Device pointers on the planner's device: `d_input` N reals, `d_out_*` N/2 + 1 each.
pub unsafe fn r2c_fft_f64_device(d_input: *const f64, d_out_re: *mut f64, d_out_im: *mut f64, planner: &PlannerR2c64, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_r2c_f64_dev(planner.raw, d_input, d_out_re, d_out_im, stream));
}
/// # Safety
/// As [`r2c_fft_f64_device`]; `d_scratch_*` are N/2 each or both null (the plan's own scratch is then used).
pub unsafe fn c2r_fft_f64_device(d_in_re: *const f64, d_in_im: *const f64, d_output: *mut f64, planner: &PlannerR2c64,
                                 d_scratch_re: *mut f64, d_scratch_im: *mut f64, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_c2r_f64_dev(planner.raw, d_in_re, d_in_im, d_output, d_scratch_re, d_scratch_im, stream));
}
/// # Safety
/// As [`r2c_fft_f64_device`].
pub unsafe fn r2c_fft_f32_device(d_input: *const f32, d_out_re: *mut f32, d_out_im: *mut f32, planner: &PlannerR2c32, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_r2c_f32_dev(planner.raw, d_input, d_out_re, d_out_im, stream));
}
/// # Safety
/// As [`c2r_fft_f64_device`].
pub unsafe fn c2r_fft_f32_device(d_in_re: *const f32, d_in_im: *const f32, d_output: *mut f32, planner: &PlannerR2c32,
                                 d_scratch_re: *mut f32, d_scratch_im: *mut f32, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_c2r_f32_dev(planner.raw, d_in_re, d_in_im, d_output, d_scratch_re, d_scratch_im, stream));
}

/// Batched device-resident real transforms (`phastft_{r2c,c2r}_*_dev_batch`): member `b` of the real side at
/// `b * real_stride`, of the spectrum at `b * spectrum_stride` (elements).  Panics with code 13 on a bad stride or alignment.
///
/// # Safety
/// Device pointers on the planner's device, `batch` members long at the given strides; the real-side stride even and its
/// base aligned to two elements.
pub unsafe fn r2c_fft_f64_device_batch(d_input: *const f64, d_out_re: *mut f64, d_out_im: *mut f64, planner: &PlannerR2c64, batch: usize,
                                       in_stride: usize, out_stride: usize, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_r2c_f64_dev_batch(planner.raw, d_input, d_out_re, d_out_im, batch, in_stride, out_stride, stream));
}
/// # Safety
/// As [`r2c_fft_f64_device_batch`].
pub unsafe fn c2r_fft_f64_device_batch(d_in_re: *const f64, d_in_im: *const f64, d_output: *mut f64, planner: &PlannerR2c64, batch: usize,
                                       in_stride: usize, out_stride: usize, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_c2r_f64_dev_batch(planner.raw, d_in_re, d_in_im, d_output, batch, in_stride, out_stride, stream));
}
/// # Safety
/// As [`r2c_fft_f64_device_batch`].
pub unsafe fn r2c_fft_f32_device_batch(d_input: *const f32, d_out_re: *mut f32, d_out_im: *mut f32, planner: &PlannerR2c32, batch: usize,
                                       in_stride: usize, out_stride: usize, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_r2c_f32_dev_batch(planner.raw, d_input, d_out_re, d_out_im, batch, in_stride, out_stride, stream));
}
/// # Safety
/// As [`r2c_fft_f64_device_batch`].
pub unsafe fn c2r_fft_f32_device_batch(d_in_re: *const f32, d_in_im: *const f32, d_output: *mut f32, planner: &PlannerR2c32, batch: usize,
                                       in_stride: usize, out_stride: usize, stream: *mut std::os::raw::c_void) {
    check(ffi::phastft_c2r_f32_dev_batch(planner.raw, d_in_re, d_in_im, d_output, batch, in_stride, out_stride, stream));
}

// ------------------------------------------------------------------------------------------------
// r2c / c2r  (algorithms/r2c.rs:521-895)
// ------------------------------------------------------------------------------------------------

/// `r2c.rs:535`
pub fn r2c_fft_f64_with_planner(input_re: &[f64], output_re: &mut [f64], output_im: &mut [f64], planner: &PlannerR2c64) {
    check(unsafe {
        ffi::phastft_r2c_f64_host(planner.raw, input_re.as_ptr(), input_re.len(), output_re.as_mut_ptr(), output_re.len(),
                                  output_im.as_mut_ptr(), output_im.len())
    });
}

/// `r2c.rs:521`
pub fn r2c_fft_f64(input_re: &[f64], output_re: &mut [f64], output_im: &mut [f64]) {
    // a planner per call, as in the reference; the library keeps the latest one for the next same-size call
    check(unsafe {
        ffi::phastft_r2c_f64_oneshot(input_re.as_ptr(), input_re.len(), output_re.as_mut_ptr(), output_re.len(),
                                     output_im.as_mut_ptr(), output_im.len(), device())
    });
}

/// `r2c.rs:607`
pub fn r2c_fft_f32_with_planner(input_re: &[f32], output_re: &mut [f32], output_im: &mut [f32], planner: &PlannerR2c32) {
    check(unsafe {
        ffi::phastft_r2c_f32_host(planner.raw, input_re.as_ptr(), input_re.len(), output_re.as_mut_ptr(), output_re.len(),
                                  output_im.as_mut_ptr(), output_im.len())
    });
}

/// `r2c.rs:598`
pub fn r2c_fft_f32(input_re: &[f32], output_re: &mut [f32], output_im: &mut [f32]) {
    check(unsafe {
        ffi::phastft_r2c_f32_oneshot(input_re.as_ptr(), input_re.len(), output_re.as_mut_ptr(), output_re.len(),
                                     output_im.as_mut_ptr(), output_im.len(), device())
    });
}

/// `r2c.rs:740` -- caller scratch is length-checked like the reference; the work happens in device memory.
pub fn c2r_fft_f64_with_planner_and_scratch(input_re: &[f64], input_im: &[f64], output: &mut [f64], planner: &PlannerR2c64,
                                            scratch_re: &mut [f64], scratch_im: &mut [f64]) {
    check(unsafe {
        ffi::phastft_c2r_f64_host(planner.raw, input_re.as_ptr(), input_re.len(), input_im.as_ptr(), input_im.len(),
                                  output.as_mut_ptr(), output.len(), scratch_re.as_mut_ptr(), scratch_re.len(),
                                  scratch_im.as_mut_ptr(), scratch_im.len())
    });
}

/// `r2c.rs:708` -- the reference allocates two N/2 Vecs here; the CUDA plan owns device scratch instead.
pub fn c2r_fft_f64_with_planner(input_re: &[f64], input_im: &[f64], output: &mut [f64], planner: &PlannerR2c64) {
    check(unsafe {
        ffi::phastft_c2r_f64_host(planner.raw, input_re.as_ptr(), input_re.len(), input_im.as_ptr(), input_im.len(),
                                  output.as_mut_ptr(), output.len(), std::ptr::null_mut(), 0, std::ptr::null_mut(), 0)
    });
}

/// `r2c.rs:695`
pub fn c2r_fft_f64(input_re: &[f64], input_im: &[f64], output: &mut [f64]) {
    check(unsafe {
        ffi::phastft_c2r_f64_oneshot(input_re.as_ptr(), input_re.len(), input_im.as_ptr(), input_im.len(), output.as_mut_ptr(), output.len(), device())
    });
}

/// `r2c.rs:835`
pub fn c2r_fft_f32_with_planner_and_scratch(input_re: &[f32], input_im: &[f32], output: &mut [f32], planner: &PlannerR2c32,
                                            scratch_re: &mut [f32], scratch_im: &mut [f32]) {
    check(unsafe {
        ffi::phastft_c2r_f32_host(planner.raw, input_re.as_ptr(), input_re.len(), input_im.as_ptr(), input_im.len(),
                                  output.as_mut_ptr(), output.len(), scratch_re.as_mut_ptr(), scratch_re.len(),
                                  scratch_im.as_mut_ptr(), scratch_im.len())
    });
}

/// `r2c.rs:813`
pub fn c2r_fft_f32_with_planner(input_re: &[f32], input_im: &[f32], output: &mut [f32], planner: &PlannerR2c32) {
    check(unsafe {
        ffi::phastft_c2r_f32_host(planner.raw, input_re.as_ptr(), input_re.len(), input_im.as_ptr(), input_im.len(),
                                  output.as_mut_ptr(), output.len(), std::ptr::null_mut(), 0, std::ptr::null_mut(), 0)
    });
}

/// `r2c.rs:804`
pub fn c2r_fft_f32(input_re: &[f32], input_im: &[f32], output: &mut [f32]) {
    check(unsafe {
        ffi::phastft_c2r_f32_oneshot(input_re.as_ptr(), input_re.len(), input_im.as_ptr(), input_im.len(), output.as_mut_ptr(), output.len(), device())
    });
}

// ------------------------------------------------------------------------------------------------
// interleaved Complex<T> API (lib.rs:41-140, feature `complex-nums`)
// ------------------------------------------------------------------------------------------------
#[cfg(feature = "complex-nums")]
mod interleaved {
    use super::*;
    use num_complex::Complex;

    /// `lib.rs:41-60`: the reference deinterleaves into two Vecs, transforms, re-interleaves; here the
    /// AoS <-> planar conversion is fused into the first pass's load and the last pass's store.
    pub fn fft_64_interleaved_with_planner_and_opts(signal: &mut [Complex<f64>], direction: Direction, planner: &PlannerDit64, _opts: &Options) {
        check(unsafe { ffi::phastft_fft_interleaved_f64_host(planner.raw, signal.as_mut_ptr() as *mut f64, signal.len(), direction as i32) });
    }
    pub fn fft_32_interleaved_with_planner_and_opts(signal: &mut [Complex<f32>], direction: Direction, planner: &PlannerDit32, _opts: &Options) {
        check(unsafe { ffi::phastft_fft_interleaved_f32_host(planner.raw, signal.as_mut_ptr() as *mut f32, signal.len(), direction as i32) });
    }
    /// `lib.rs:77-97`
    pub fn fft_64_interleaved_with_planner(signal: &mut [Complex<f64>], direction: Direction, planner: &PlannerDit64) {
        let opts = Options::guess_options(signal.len());
        fft_64_interleaved_with_planner_and_opts(signal, direction, planner, &opts);
    }
    pub fn fft_32_interleaved_with_planner(signal: &mut [Complex<f32>], direction: Direction, planner: &PlannerDit32) {
        let opts = Options::guess_options(signal.len());
        fft_32_interleaved_with_planner_and_opts(signal, direction, planner, &opts);
    }
    /// `lib.rs:113-140`
    pub fn fft_64_interleaved(signal: &mut [Complex<f64>], direction: Direction) {
        let planner = PlannerDit64::new(signal.len());
        fft_64_interleaved_with_planner(signal, direction, &planner);
    }
    pub fn fft_32_interleaved(signal: &mut [Complex<f32>], direction: Direction) {
        let planner = PlannerDit32::new(signal.len());
        fft_32_interleaved_with_planner(signal, direction, &planner);
    }
}
#[cfg(feature = "complex-nums")]
pub use interleaved::*;
