//! `extern "C"` declarations of include/rimphony_b200.h (ABI version 2), one to one.
use std::os::raw::{c_char, c_double, c_float, c_int, c_void};

/// struct rimphony_b200_options
#[repr(C)]
#[derive(Default)]
pub struct Options {
    pub struct_size: u32,
    pub mode: i32,
    pub coeff_mask: u32,           // 0 = all eight
    pub param_broadcast_mask: u32,
    pub device_plus_one: i32,      // 0 = the calling thread's current device
    pub reserved0: i32,
    pub epsrel_gamma: f64,
    pub epsrel_n: f64,
    pub epsrel_heyvaerts_inner: f64,
    pub epsrel_heyvaerts_outer: f64,
}

/// struct rimphony_b200_extras
#[repr(C)]
pub struct Extras {
    pub lobes4: *mut c_double,
    pub counters: *mut u32,
    pub norm: *mut c_double,
}

extern "C" {
    pub fn rimphony_b200_compute_all_dimensionless(
        kind: c_int, n_points: i64, s: *const c_double, theta: *const c_double, params: *const *const c_double,
        n_params: c_int, opts: *const Options, out8: *mut c_double, status: *mut i32) -> c_int;
    pub fn rimphony_b200_compute_all_dimensionless_ex(
        kind: c_int, n_points: i64, s: *const c_double, theta: *const c_double, params: *const *const c_double,
        n_params: c_int, opts: *const Options, out8: *mut c_double, status: *mut i32, extras: *const Extras) -> c_int;
    pub fn rimphony_b200_compute_all_dimensionless_device(
        kind: c_int, n_points: i64, s: *const c_double, theta: *const c_double, params: *const *const c_double,
        n_params: c_int, opts: *const Options, out8: *mut c_double, status: *mut i32, extras: *const Extras,
        stream: *mut c_void, synchronize: c_int) -> c_int;
    pub fn rimphony_b200_compute_all_dimensionless_multi(
        kind: c_int, n_points: i64, s: *const c_double, theta: *const c_double, params: *const *const c_double,
        n_params: c_int, opts: *const Options, out8: *mut c_double, status: *mut i32, n_devices: c_int) -> c_int;
    pub fn rimphony_b200_compute_dimensionless(
        kind: c_int, params: *const c_double, n_params: c_int, coeff: c_int, stokes: c_int, s: c_double,
        theta: c_double, out: *mut c_double) -> c_int;
    pub fn rimphony_b200_compute_cgs(
        kind: c_int, params: *const c_double, n_params: c_int, coeff: c_int, stokes: c_int, nu: c_double,
        b: c_double, n_e: c_double, theta: c_double, out: *mut c_double) -> c_int;
    pub fn rimphony_b200_diagnostic_symphony(
        kind: c_int, params: *const c_double, n_params: c_int, coeff: c_int, stokes: c_int, s: c_double,
        theta: c_double, what: c_int, count: i64, a: *const c_double, b: *const c_double, out: *mut c_double,
        status: *mut i32) -> c_int;
    pub fn rimphony_b200_bessel_jn(count: i64, n: *const c_double, x: *const c_double, j: *mut c_double,
                                   dj: *mut c_double) -> c_int;
    pub fn rimphony_b200_dist_eval(kind: c_int, params: *const c_double, n_params: c_int, count: i64,
                                   gamma: *const c_double, cos_xi: *const c_double, out3: *mut c_double) -> c_int;
    pub fn rimphony_b200_transfer(
        n_rays: i64, n_cells: i64, coeffs8: *const c_double, psi: *const c_double, ds: *const c_double,
        stokes0: *const c_double, stokes4: *mut c_double, status: *mut i32) -> c_int;
    pub fn rimphony_b200_transfer_device(
        n_rays: i64, n_cells: i64, coeffs8: *const c_double, psi: *const c_double, ds: *const c_double,
        stokes0: *const c_double, stokes4: *mut c_double, status: *mut i32, stream: *mut c_void,
        synchronize: c_int) -> c_int;
    pub fn rimphony_b200_compute_stokes_cgs(
        kind: c_int, n_rays: i64, n_cells: i64, nu: *const c_double, b: *const c_double, n_e: *const c_double,
        theta: *const c_double, psi: *const c_double, ds: *const c_double, params: *const *const c_double,
        n_params: c_int, opts: *const Options, stokes4: *mut c_double, coeffs8_cgs: *mut c_double,
        status: *mut i32) -> c_int;
    pub fn rimphony_b200_last_kernel_ms(device: c_int, out_ms: *mut c_float) -> c_int;
    pub fn rimphony_b200_fp64_peak_tflops(device: c_int, out_tflops: *mut c_double) -> c_int;
    pub fn rimphony_b200_kernel_launch_count() -> u64;
    pub fn rimphony_b200_device_count() -> c_int;
    pub fn rimphony_b200_abi_version() -> c_int;
    pub fn rimphony_b200_last_error() -> *const c_char;
    pub fn rimphony_b200_shutdown();
}
