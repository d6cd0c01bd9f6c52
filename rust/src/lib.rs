//! Rust facade over `include/rimphony_b200.h`.
//!
//! Keeps the reference's public surface for the hot path -- `Coefficient`, `Stokes`, the
//! distribution types with their builders, `full_calculation()`, and the
//! `SynchrotronCalculator` trait (reference `src/lib.rs:75-107, 150-210, 231-247`) -- and adds the
//! batched call the GPU path is built for.  Numerical failure is `NaN`, never a panic or an
//! `Err` (reference `src/lib.rs:239-240`, `symphony.rs:115-146`, `heyvaerts.rs:98-177`);
//! `Err(String)` is reserved for infrastructure errors (no CUDA device, bad arguments).
//!
//! NOT COMPILED IN THIS IMAGE (no rustc); the same ABI is exercised through ctypes in `tests/`.

use std::ffi::CStr;
use std::os::raw::{c_char, c_double, c_int, c_void};

pub mod ffi;

pub const PI: f64 = std::f64::consts::PI;
pub const TWO_PI: f64 = 2. * PI;
/// src/lib.rs:58-67 (cgs)
pub const MASS_ELECTRON: f64 = 9.1093826e-28;
pub const SPEED_LIGHT: f64 = 2.99792458e10;
pub const ELECTRON_CHARGE: f64 = 4.80320680e-10;

/// src/lib.rs:92-107
#[derive(Copy, Clone, Debug, Eq, Hash, PartialEq)]
pub enum Coefficient {
    Emission = 0,
    Absorption = 1,
    Faraday = 2,
}

/// src/lib.rs:75-87
#[derive(Copy, Clone, Debug, Eq, Hash, PartialEq)]
pub enum Stokes {
    I = 0,
    Q = 1,
    V = 2,
}

/// Evaluation mode (`enum rimphony_b200_mode`).
#[derive(Copy, Clone, Debug, Eq, PartialEq)]
pub enum Mode {
    Fast = 0,
    Faithful = 1,
    FusedAll = 2,
    Fused = 3,
}

/// Per-point status bits (`RIMPHONY_B200_STATUS_*`).
pub mod status {
    pub const NAN: i32 = 1;
    pub const CAP_HIT: i32 = 2;
    pub const NORM_FAILED: i32 = 4;
    pub const REROUTED: i32 = 8;
}

fn last_error() -> String {
    unsafe { CStr::from_ptr(ffi::rimphony_b200_last_error()) }.to_string_lossy().into_owned()
}

/// What a distribution hands to the C ABI: its kind and its parameter columns in the order of
/// `enum rimphony_b200_dist_kind`.
pub trait B200Params {
    const KIND: c_int;
    fn b200_params(&self) -> Vec<f64>;
}

/// src/power_law.rs:27-87
#[derive(Copy, Clone, Debug, PartialEq)]
pub struct PowerLawDistribution {
    p: f64,
    gamma_min: f64,
    gamma_max: f64,
    gamma_cutoff: f64,
}

impl PowerLawDistribution {
    pub fn new(p: f64) -> Self {
        PowerLawDistribution { p, gamma_min: 1., gamma_max: 1e12, gamma_cutoff: 1e10 }
    }
    pub fn gamma_limits(mut self, gamma_min: f64, gamma_max: f64, gamma_cutoff: f64) -> Self {
        self.gamma_min = gamma_min;
        self.gamma_max = gamma_max;
        self.gamma_cutoff = gamma_cutoff;
        self
    }
    pub fn full_calculation<L>(self, _logger: L) -> FullSynchrotronCalculator<Self> {
        FullSynchrotronCalculator::new(self)
    }
}

impl B200Params for PowerLawDistribution {
    const KIND: c_int = 0;
    fn b200_params(&self) -> Vec<f64> {
        vec![self.p, self.gamma_min, self.gamma_max, self.gamma_cutoff]
    }
}

/// src/thermal_juettner.rs:23-50
#[derive(Copy, Clone, Debug, PartialEq)]
pub struct ThermalJuettnerDistribution {
    t: f64,
}

impl ThermalJuettnerDistribution {
    pub fn new(t: f64) -> Self {
        ThermalJuettnerDistribution { t }
    }
    pub fn full_calculation<L>(self, _logger: L) -> FullSynchrotronCalculator<Self> {
        FullSynchrotronCalculator::new(self)
    }
}

impl B200Params for ThermalJuettnerDistribution {
    const KIND: c_int = 1;
    fn b200_params(&self) -> Vec<f64> {
        vec![self.t]
    }
}

/// src/pitchy_pl.rs:22-90
#[derive(Copy, Clone, Debug, PartialEq)]
pub struct PitchyPowerLawDistribution {
    p: f64,
    k: f64,
    gamma_min: f64,
    gamma_max: f64,
    gamma_cutoff: f64,
}

impl PitchyPowerLawDistribution {
    pub fn new(p: f64, k: f64) -> Self {
        PitchyPowerLawDistribution { p, k, gamma_min: 1., gamma_max: 1e12, gamma_cutoff: 1e10 }
    }
    pub fn gamma_limits(mut self, gamma_min: f64, gamma_max: f64, gamma_cutoff: f64) -> Self {
        self.gamma_min = gamma_min;
        self.gamma_max = gamma_max;
        self.gamma_cutoff = gamma_cutoff;
        self
    }
    pub fn full_calculation<L>(self, _logger: L) -> FullSynchrotronCalculator<Self> {
        FullSynchrotronCalculator::new(self)
    }
}

impl B200Params for PitchyPowerLawDistribution {
    const KIND: c_int = 2;
    fn b200_params(&self) -> Vec<f64> {
        vec![self.p, self.k, self.gamma_min, self.gamma_max, self.gamma_cutoff]
    }
}

/// A broken power law times sin^k(pitch angle): gamma^-p1 below `gamma_break`,
/// gamma_break^(p2 - p1) gamma^-p2 from it on, built as src/pitchy_pl.rs:22-90 builds its single one.
#[derive(Copy, Clone, Debug, PartialEq)]
pub struct PitchyBrokenPowerLawDistribution {
    p1: f64,
    p2: f64,
    gamma_break: f64,
    k: f64,
    gamma_min: f64,
    gamma_max: f64,
    gamma_cutoff: f64,
}

impl PitchyBrokenPowerLawDistribution {
    pub fn new(p1: f64, p2: f64, gamma_break: f64, k: f64) -> Self {
        PitchyBrokenPowerLawDistribution { p1, p2, gamma_break, k, gamma_min: 1., gamma_max: 1e12, gamma_cutoff: 1e10 }
    }
    pub fn gamma_limits(mut self, gamma_min: f64, gamma_max: f64, gamma_cutoff: f64) -> Self {
        self.gamma_min = gamma_min;
        self.gamma_max = gamma_max;
        self.gamma_cutoff = gamma_cutoff;
        self
    }
    pub fn full_calculation<L>(self, _logger: L) -> FullSynchrotronCalculator<Self> {
        FullSynchrotronCalculator::new(self)
    }
}

impl B200Params for PitchyBrokenPowerLawDistribution {
    const KIND: c_int = 4;
    fn b200_params(&self) -> Vec<f64> {
        vec![self.p1, self.p2, self.gamma_break, self.k, self.gamma_min, self.gamma_max, self.gamma_cutoff]
    }
}

/// src/pitchy_kappa.rs:28-85
#[derive(Copy, Clone, Debug, PartialEq)]
pub struct PitchyKappaDistribution {
    kappa: f64,
    width: f64,
    k: f64,
    gamma_cutoff: f64,
}

impl PitchyKappaDistribution {
    pub fn new(kappa: f64, width: f64, k: f64) -> Self {
        PitchyKappaDistribution { kappa, width, k, gamma_cutoff: 1e10 }
    }
    pub fn gamma_cutoff(mut self, gamma_cutoff: f64) -> Self {
        self.gamma_cutoff = gamma_cutoff;
        self
    }
    pub fn full_calculation<L>(self, _logger: L) -> FullSynchrotronCalculator<Self> {
        FullSynchrotronCalculator::new(self)
    }
}

impl B200Params for PitchyKappaDistribution {
    const KIND: c_int = 3;
    fn b200_params(&self) -> Vec<f64> {
        vec![self.kappa, self.width, self.k, self.gamma_cutoff]
    }
}

/// src/lib.rs:150-210
pub trait SynchrotronCalculator {
    fn compute_dimensionless(&self, coeff: Coefficient, stokes: Stokes, s: f64, theta: f64) -> f64;

    /// src/lib.rs:163-173
    fn compute_cgs(&self, coeff: Coefficient, stokes: Stokes, nu: f64, b: f64, n_e: f64, theta: f64) -> f64 {
        let nu_c = ELECTRON_CHARGE * b / (TWO_PI * MASS_ELECTRON * SPEED_LIGHT);
        let val = self.compute_dimensionless(coeff, stokes, nu / nu_c, theta);
        match coeff {
            Coefficient::Emission => val * n_e * nu,
            Coefficient::Absorption | Coefficient::Faraday => val * n_e / nu,
        }
    }

    /// src/lib.rs:176-191: `[j_I, alpha_I, j_Q, alpha_Q, j_V, alpha_V, rho_Q, rho_V]`
    fn compute_all_dimensionless(&self, s: f64, theta: f64) -> [f64; 8];

    /// src/lib.rs:196-209
    fn compute_all_cgs(&self, nu: f64, b: f64, n_e: f64, theta: f64) -> [f64; 8] {
        let nu_c = ELECTRON_CHARGE * b / (TWO_PI * MASS_ELECTRON * SPEED_LIGHT);
        let mut r = self.compute_all_dimensionless(nu / nu_c, theta);
        for (i, v) in r.iter_mut().enumerate() {
            *v *= if i % 2 == 0 && i < 6 { n_e * nu } else { n_e / nu };
        }
        r
    }
}

/// src/lib.rs:231-247; owns a copy of the distribution.
#[derive(Copy, Clone, Debug, PartialEq)]
pub struct FullSynchrotronCalculator<D> {
    distrib: D,
    mode: Mode,
}

impl<D: B200Params> FullSynchrotronCalculator<D> {
    pub fn new(distrib: D) -> Self {
        FullSynchrotronCalculator { distrib, mode: Mode::Fast }
    }
    pub fn mode(mut self, mode: Mode) -> Self {
        self.mode = mode;
        self
    }
}

impl<D: B200Params> FullSynchrotronCalculator<D> {
    /// Emergent Stokes `[I, Q, U, V]` of `n_rays` rays of `n_cells` cells each of this distribution
    /// (`rimphony_b200_compute_stokes_cgs`): the coefficients of `compute_all_cgs` in every cell, then
    /// `transfer` with no incident radiation, in one call on the device.  `nu`, `b`, `n_e`, `theta`,
    /// `psi` and `ds` hold one value per cell, index `ray * n_cells + cell` (cell 0 where the ray
    /// enters); `n_cells = 1` is a set of uniform slabs.
    pub fn compute_stokes_cgs(&self, n_cells: usize, nu: &[f64], b: &[f64], n_e: &[f64], theta: &[f64],
                              psi: &[f64], ds: &[f64]) -> Result<TransferResult, String>
    {
        let n = nu.len();
        if n_cells == 0 || n % n_cells != 0 {
            return Err(format!("{} cells do not make rays of {} cells", n, n_cells));
        }
        if [b.len(), n_e.len(), theta.len(), psi.len(), ds.len()].iter().any(|&l| l != n) {
            return Err("nu, b, n_e, theta, psi and ds differ in length".into());
        }
        let n_rays = n / n_cells;
        let p = self.distrib.b200_params();
        let ptrs: Vec<*const c_double> = p.iter().map(|v| v as *const f64).collect();
        let opts = ffi::Options {
            struct_size: std::mem::size_of::<ffi::Options>() as u32,
            mode: self.mode as i32,
            param_broadcast_mask: (1u32 << p.len()) - 1,
            ..Default::default()
        };
        let mut soa = vec![f64::NAN; 4 * n_rays];
        let mut status = vec![0i32; n_rays];
        let rc = unsafe {
            ffi::rimphony_b200_compute_stokes_cgs(D::KIND, n_rays as i64, n_cells as i64, nu.as_ptr(), b.as_ptr(),
                                                  n_e.as_ptr(), theta.as_ptr(), psi.as_ptr(), ds.as_ptr(),
                                                  ptrs.as_ptr(), ptrs.len() as c_int, &opts, soa.as_mut_ptr(),
                                                  std::ptr::null_mut(), status.as_mut_ptr())
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok(TransferResult::from_soa(&soa, status))
    }
}

impl<D: B200Params> SynchrotronCalculator for FullSynchrotronCalculator<D> {
    fn compute_dimensionless(&self, coeff: Coefficient, stokes: Stokes, s: f64, theta: f64) -> f64 {
        let p = self.distrib.b200_params();
        let mut out = f64::NAN;
        let rc = unsafe {
            ffi::rimphony_b200_compute_dimensionless(D::KIND, p.as_ptr(), p.len() as c_int, coeff as c_int,
                                                     stokes as c_int, s, theta, &mut out)
        };
        if rc != 0 { f64::NAN } else { out }
    }

    fn compute_all_dimensionless(&self, s: f64, theta: f64) -> [f64; 8] {
        let p = self.distrib.b200_params();
        let cols: Vec<&[f64]> = p.iter().map(std::slice::from_ref).collect();
        match compute_all_dimensionless_batch(D::KIND, &[s], &[theta], &cols, self.mode) {
            Ok(v) => v.values[0],
            Err(_) => [f64::NAN; 8],
        }
    }
}

/// One batched call's results: row i is `compute_all_dimensionless` of point i.
pub struct BatchResult {
    pub values: Vec<[f64; 8]>,
    pub status: Vec<i32>,
}

/// Additive API (the reference has no batch call; replaces the loop body of
/// examples/crank-out-pitchypl.rs:157-172): all eight coefficients for `n` points.  `columns`
/// are the parameter columns of `kind` in the order of include/rimphony_b200.h, each of
/// length `n` or of length 1 (broadcast on the device).
pub fn compute_all_dimensionless_batch(kind: c_int, s: &[f64], theta: &[f64], columns: &[&[f64]], mode: Mode)
    -> Result<BatchResult, String>
{
    let n = s.len();
    if theta.len() != n {
        return Err("s and theta differ in length".into());
    }
    let mut bcast = 0u32;
    for (j, c) in columns.iter().enumerate() {
        if c.len() == 1 && n != 1 {
            bcast |= 1 << j;
        } else if c.len() != n {
            return Err(format!("parameter column {} has length {}, expected {} or 1", j, c.len(), n));
        }
    }
    let ptrs: Vec<*const c_double> = columns.iter().map(|c| c.as_ptr()).collect();
    let mut soa = vec![f64::NAN; 8 * n];
    let mut status = vec![0i32; n];
    let opts = ffi::Options {
        struct_size: std::mem::size_of::<ffi::Options>() as u32,
        mode: mode as i32,
        param_broadcast_mask: bcast,
        ..Default::default()
    };
    let rc = unsafe {
        ffi::rimphony_b200_compute_all_dimensionless(kind, n as i64, s.as_ptr(), theta.as_ptr(), ptrs.as_ptr(),
                                                     ptrs.len() as c_int, &opts, soa.as_mut_ptr(), status.as_mut_ptr())
    };
    if rc != 0 {
        return Err(last_error());
    }
    let values = (0..n).map(|i| { let mut r = [0.0; 8]; for c in 0..8 { r[c] = soa[c * n + i]; } r }).collect();
    Ok(BatchResult { values, status })
}

/// The same batch sharded over `n_devices` GPUs of this box (0 = all): one host thread and stream
/// per device inside the library, no inter-GPU communication, results gathered in place.
pub fn compute_all_dimensionless_multi(kind: c_int, s: &[f64], theta: &[f64], columns: &[&[f64]], n_devices: i32)
    -> Result<BatchResult, String>
{
    let n = s.len();
    let ptrs: Vec<*const c_double> = columns.iter().map(|c| c.as_ptr()).collect();
    let mut soa = vec![f64::NAN; 8 * n];
    let mut status = vec![0i32; n];
    let rc = unsafe {
        ffi::rimphony_b200_compute_all_dimensionless_multi(kind, n as i64, s.as_ptr(), theta.as_ptr(), ptrs.as_ptr(),
                                                           ptrs.len() as c_int, std::ptr::null(), soa.as_mut_ptr(),
                                                           status.as_mut_ptr(), n_devices)
    };
    if rc != 0 {
        return Err(last_error());
    }
    let values = (0..n).map(|i| { let mut r = [0.0; 8]; for c in 0..8 { r[c] = soa[c * n + i]; } r }).collect();
    Ok(BatchResult { values, status })
}

/// Emergent Stokes vectors of a set of rays: `stokes[ray] = [I, Q, U, V]`, and the per-ray status
/// word (`status::NAN` if the ray's vector is NaN).
pub struct TransferResult {
    pub stokes: Vec<[f64; 4]>,
    pub status: Vec<i32>,
}

impl TransferResult {
    fn from_soa(soa: &[f64], status: Vec<i32>) -> Self {
        let n = status.len();
        let stokes = (0..n).map(|r| [soa[r], soa[n + r], soa[2 * n + r], soa[3 * n + r]]).collect();
        TransferResult { stokes, status }
    }
}

/// Polarized transfer through rays of cells with constant coefficients (`rimphony_b200_transfer`; the
/// matrix and its sign convention are in include/rimphony_b200.h).  `coeffs[p]` is the cgs vector of
/// `compute_all_cgs` of cell `p = ray * n_cells + cell`, cell 0 where the ray enters; `psi` and `ds`
/// hold one value per cell; `stokes0` is the incident `[I, Q, U, V]` of each ray (zero if `None`).
pub fn transfer(n_cells: usize, coeffs: &[[f64; 8]], psi: &[f64], ds: &[f64], stokes0: Option<&[[f64; 4]]>)
    -> Result<TransferResult, String>
{
    let n = coeffs.len();
    if n_cells == 0 || n % n_cells != 0 || psi.len() != n || ds.len() != n {
        return Err(format!("{} cells with {} angles and {} lengths do not make rays of {} cells",
                           n, psi.len(), ds.len(), n_cells));
    }
    let n_rays = n / n_cells;
    let mut soa = vec![0.0; 8 * n];
    for (p, c) in coeffs.iter().enumerate() {
        for k in 0..8 {
            soa[k * n + p] = c[k];
        }
    }
    let s0: Option<Vec<f64>> = match stokes0 {
        Some(v) if v.len() != n_rays => return Err("stokes0 needs one vector per ray".into()),
        Some(v) => Some((0..4 * n_rays).map(|i| v[i % n_rays][i / n_rays]).collect()),
        None => None,
    };
    let mut out = vec![f64::NAN; 4 * n_rays];
    let mut status = vec![0i32; n_rays];
    let rc = unsafe {
        ffi::rimphony_b200_transfer(n_rays as i64, n_cells as i64, soa.as_ptr(), psi.as_ptr(), ds.as_ptr(),
                                    s0.as_ref().map_or(std::ptr::null(), |v| v.as_ptr()), out.as_mut_ptr(),
                                    status.as_mut_ptr())
    };
    if rc != 0 {
        return Err(last_error());
    }
    Ok(TransferResult::from_soa(&out, status))
}

/// leung-bessel/src/lib.rs:56-75 on the device: `(J_n(x), J_n'(x))` for arrays of arguments.
pub fn bessel_jn(n: &[f64], x: &[f64]) -> Result<(Vec<f64>, Vec<f64>), String> {
    assert_eq!(n.len(), x.len());
    let mut j = vec![f64::NAN; n.len()];
    let mut dj = vec![f64::NAN; n.len()];
    let rc = unsafe { ffi::rimphony_b200_bessel_jn(n.len() as i64, n.as_ptr(), x.as_ptr(), j.as_mut_ptr(), dj.as_mut_ptr()) };
    if rc != 0 { Err(last_error()) } else { Ok((j, dj)) }
}

/// Release every device buffer, stream and event the library holds.
pub fn shutdown() {
    unsafe { ffi::rimphony_b200_shutdown() }
}

#[allow(dead_code)]
fn _unused(_: *const c_char, _: *mut c_void) {}
