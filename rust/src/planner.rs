//! `planner.rs` of the reference: `Direction`, `PlannerMode`, `PlannerDit{64,32}`, `PlannerR2c{64,32}`.
//! The planners own an opaque handle to the CUDA plan (device twiddle tables, workspace, stream) and free
//! it on drop.  They stay `Send + Sync` like the reference's (plain `Vec` fields there): the C library
//! serialises workspace use inside the plan.
use crate::{check, device, ffi};

/// `planner.rs:10-16`
#[derive(Copy, Clone)]
pub enum Direction {
    Forward = 1,
    Reverse = -1,
}

/// `planner.rs:25-32`.  The reference accepts the mode and ignores it (`planner.rs:65`); here `Tune` is real: the
/// planner builds a handful of pass decompositions / tile widths around the heuristic one, times them on the device
/// and keeps the fastest.
#[derive(Copy, Clone, Debug, Default)]
pub enum PlannerMode {
    #[default]
    Heuristic,
    Tune,
}

macro_rules! impl_planner_dit {
    ($name:ident, $raw:ty, $create:ident, $destroy:ident, $size:ident, $describe:ident, $reserve:ident) => {
        pub struct $name {
            pub(crate) raw: *mut $raw,
        }
        unsafe impl Send for $name {}
        unsafe impl Sync for $name {}
        impl $name {
            /// `planner.rs:55`: panics unless `num_points` is a non-zero power of two.
            pub fn new(num_points: usize) -> Self {
                Self::with_mode(num_points, PlannerMode::Heuristic)
            }
            /// `planner.rs:65`
            pub fn with_mode(num_points: usize, mode: PlannerMode) -> Self {
                let mut raw = std::ptr::null_mut();
                check(unsafe { ffi::$create(num_points, device(), mode as i32, &mut raw) });
                Self { raw }
            }
            /// Number of points the planner was built for.
            pub fn num_points(&self) -> usize {
                unsafe { ffi::$size(self.raw) }
            }
            /// Additive: the pass decomposition and kernels the planner chose, e.g.
            /// `"n=2^20 f64: COL R=1024(32x32) C=8 NT=256 | TRANS R=1024(32x32) C=8 NT=256"`.
            pub fn describe(&self) -> String {
                unsafe { std::ffi::CStr::from_ptr(ffi::$describe(self.raw)) }.to_string_lossy().into_owned()
            }
            /// Additive: size the device workspace for calls of up to `batch` transforms now (otherwise the first larger
            /// batched call grows it, synchronising the device).
            pub fn reserve(&self, batch: usize) {
                check(unsafe { ffi::$reserve(self.raw, batch) });
            }
        }
        impl Drop for $name {
            fn drop(&mut self) {
                unsafe { ffi::$destroy(self.raw) }
            }
        }
    };
}
impl_planner_dit!(PlannerDit64, ffi::phastft_plan_dit_f64, phastft_plan_dit_f64_create, phastft_plan_dit_f64_destroy,
                  phastft_plan_dit_f64_size, phastft_plan_dit_f64_describe, phastft_plan_dit_f64_reserve);
impl_planner_dit!(PlannerDit32, ffi::phastft_plan_dit_f32, phastft_plan_dit_f32_create, phastft_plan_dit_f32_destroy,
                  phastft_plan_dit_f32_size, phastft_plan_dit_f32_describe, phastft_plan_dit_f32_reserve);

macro_rules! impl_planner_r2c {
    ($name:ident, $raw:ty, $create:ident, $destroy:ident, $reserve:ident) => {
        pub struct $name {
            pub(crate) raw: *mut $raw,
        }
        unsafe impl Send for $name {}
        unsafe impl Sync for $name {}
        impl $name {
            /// `planner.rs:194`: panics with "n must be a power of 2 >= 4".
            pub fn new(n: usize) -> Self {
                let mut raw = std::ptr::null_mut();
                check(unsafe { ffi::$create(n, device(), &mut raw) });
                Self { raw }
            }
            /// Additive: size the half-length transform's workspace for batched calls of up to `batch` members now.
            pub fn reserve(&self, batch: usize) {
                check(unsafe { ffi::$reserve(self.raw, batch) });
            }
        }
        impl Drop for $name {
            fn drop(&mut self) {
                unsafe { ffi::$destroy(self.raw) }
            }
        }
    };
}
impl_planner_r2c!(PlannerR2c64, ffi::phastft_plan_r2c_f64, phastft_plan_r2c_f64_create, phastft_plan_r2c_f64_destroy,
                  phastft_plan_r2c_f64_reserve);
impl_planner_r2c!(PlannerR2c32, ffi::phastft_plan_r2c_f32, phastft_plan_r2c_f32_create, phastft_plan_r2c_f32_destroy,
                  phastft_plan_r2c_f32_reserve);
