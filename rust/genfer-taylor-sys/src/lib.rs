//! `extern "C"` declarations for `include/genfer_taylor.h` plus a thin safe wrapper (`DevicePoly`)
//! with the value semantics of genfer's `TaylorPoly<F64>` (src/multivariate_taylor.rs).
//!
//! This crate cannot be compiled in the build image (no cargo/rustc there); it is the binding a
//! genfer maintainer adds, see INTEGRATION.md for the patch to `multivariate_taylor.rs`.
#![allow(non_camel_case_types)]
use std::{ffi::CStr, os::raw::{c_char, c_int, c_uint, c_void}, ptr, rc::Rc};

pub const GTP_UNBOUNDED: u64 = u64::MAX; // usize::MAX on 64-bit targets

#[repr(C)] pub struct gtp_ctx { _p: [u8; 0] }
#[repr(C)] pub struct gtp_poly { _p: [u8; 0] }
#[repr(C)] pub struct gtu_series { _p: [u8; 0] }
#[repr(C)] pub struct gtu_program { _p: [u8; 0] }
#[repr(C)] pub struct gtp_sgcl_result { _p: [u8; 0] }
#[repr(C)] pub struct gti_poly { _p: [u8; 0] }

extern "C" {
    // ---- BEGIN GENERATED (tools/gen_rust_externs.py) ----
    pub fn gtp_ctx_create(device: c_int, cuda_stream: *mut c_void, out: *mut *mut gtp_ctx) -> c_int;
    pub fn gtp_ctx_destroy(ctx: *mut gtp_ctx);
    pub fn gtp_last_error(ctx: *mut gtp_ctx) -> *const c_char;
    pub fn gtp_ctx_synchronize(ctx: *mut gtp_ctx) -> c_int;
    pub fn gtp_ctx_trim(ctx: *mut gtp_ctx) -> c_int;
    pub fn gtp_ctx_stream(ctx: *mut gtp_ctx) -> *mut c_void;
    pub fn gtp_ctx_launch_count(ctx: *mut gtp_ctx) -> u64;
    pub fn gtp_ctx_set_fast_mul(ctx: *mut gtp_ctx, enabled: c_int) -> c_int;
    pub fn gtp_nccl_unique_id(out128: *mut c_void) -> c_int;
    pub fn gtp_ctx_create_group(device: c_int, cuda_stream: *mut c_void, rank: c_int, world: c_int, id128: *const c_void, out: *mut *mut gtp_ctx) -> c_int;
    pub fn gtp_ctx_group_info(ctx: *mut gtp_ctx, rank: *mut c_int, world: *mut c_int, partitioned_products: *mut u64, gathers: *mut u64) -> c_int;
    pub fn gtp_ctx_set_partition_threshold(ctx: *mut gtp_ctx, coefficients: u64) -> c_int;
    pub fn gtp_partition_rows(n_rows: u64, world: c_int, rank: c_int, rows_out: *mut u64) -> u64;
    pub fn gtp_partition_block(n_slices: u64, world: c_int, rank: c_int, lo: *mut u64, hi: *mut u64, block: *mut u64);
    pub fn gtp_from_host_block(ctx: *mut gtp_ctx, ndim: c_int, shape: *const u64, degrees_p1: *const u64, block_data: *const f64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_from_device_block(ctx: *mut gtp_ctx, ndim: c_int, shape: *const u64, degrees_p1: *const u64, device_block: *const f64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_is_distributed(p: *const gtp_poly) -> c_int;
    pub fn gtp_replicate(ctx: *mut gtp_ctx, p: *const gtp_poly) -> c_int;
    pub fn gtp_local_rows(p: *const gtp_poly, rows_out: *mut u64) -> u64;
    pub fn gtp_to_host_local(ctx: *mut gtp_ctx, p: *const gtp_poly, out: *mut f64) -> c_int;
    pub fn gtp_from_host(ctx: *mut gtp_ctx, ndim: c_int, shape: *const u64, degrees_p1: *const u64, data: *const f64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_from_device(ctx: *mut gtp_ctx, ndim: c_int, shape: *const u64, degrees_p1: *const u64, device_data: *const f64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_to_host(ctx: *mut gtp_ctx, p: *const gtp_poly, out: *mut f64) -> c_int;
    pub fn gtp_device_ptr(ctx: *mut gtp_ctx, p: *const gtp_poly, out: *mut *const f64) -> c_int;
    pub fn gtp_clone(ctx: *mut gtp_ctx, p: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_free(ctx: *mut gtp_ctx, p: *mut gtp_poly);
    pub fn gtp_ndim(p: *const gtp_poly) -> c_int;
    pub fn gtp_len(p: *const gtp_poly) -> u64;
    pub fn gtp_shape(p: *const gtp_poly, out: *mut u64);
    pub fn gtp_degrees_p1(p: *const gtp_poly, out: *mut u64);
    pub fn gtp_from_scalar(ctx: *mut gtp_ctx, x: f64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_zero_with(ctx: *mut gtp_ctx, ndim: c_int, degrees_p1: *const u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_var(ctx: *mut gtp_ctx, v: u64, x: f64, len: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_var_at_zero(ctx: *mut gtp_ctx, v: u64, len: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_var_with_degrees_p1(ctx: *mut gtp_ctx, v: u64, x: f64, ndim: c_int, degrees_p1: *const u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_add(ctx: *mut gtp_ctx, a: *const gtp_poly, b: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_sub(ctx: *mut gtp_ctx, a: *const gtp_poly, b: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_mul(ctx: *mut gtp_ctx, a: *const gtp_poly, b: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_div(ctx: *mut gtp_ctx, a: *const gtp_poly, b: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_neg(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_exp(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_log(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_pow(ctx: *mut gtp_ctx, a: *const gtp_poly, exp: u32, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_derivative(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, n: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_taylor_expansion_of_coeff(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, n: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_shift_down(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, n: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_coefficients_of_term(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, order: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_taylor_polynomial(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, order: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_taylor_polynomial_terms(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, orders: *const u64, n_orders: c_int, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_subst_var(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, subst: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_truncate_to_degree_p1(ctx: *mut gtp_ctx, a: *const gtp_poly, degree_p1: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_remove_last_variable(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_extend_to_dim(ctx: *mut gtp_ctx, a: *const gtp_poly, ndim: u64, degree_p1: u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_extend(ctx: *mut gtp_ctx, a: *const gtp_poly, ndim: c_int, new_size: *const u64, out: *mut *mut gtp_poly) -> c_int;
    pub fn gtp_constant_term(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut f64) -> c_int;
    pub fn gtp_coefficient(ctx: *mut gtp_ctx, a: *const gtp_poly, index: *const u64, n_index: c_int, out: *mut f64) -> c_int;
    pub fn gtp_gather_axis(ctx: *mut gtp_ctx, a: *const gtp_poly, v: u64, count: u64, out: *mut f64) -> c_int;
    pub fn gtp_extract_constant(ctx: *mut gtp_ctx, a: *const gtp_poly, is_constant: *mut c_int, value: *mut f64) -> c_int;
    pub fn gtp_extract_linear(ctx: *mut gtp_ctx, a: *const gtp_poly, is_linear: *mut c_int, c: *mut f64, m: *mut f64, v: *mut u64) -> c_int;
    pub fn gtp_is_zero(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut c_int) -> c_int;
    pub fn gtp_is_one(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut c_int) -> c_int;
    pub fn gtp_evaluate_all_one(ctx: *mut gtp_ctx, a: *const gtp_poly, out: *mut f64) -> c_int;
    pub fn gtp_eq(ctx: *mut gtp_ctx, a: *const gtp_poly, b: *const gtp_poly, out: *mut c_int) -> c_int;
    pub fn gtp_mul_rows_raw(ctx: *mut gtp_ctx, ndim: c_int, xshape: *const u64, x: *const f64, yshape: *const u64, y: *const f64, rshape: *const u64, row_begin: u64, row_step: u64, row_count: u64, out_rows: *mut f64) -> c_int;
    pub fn gtp_mul_rowlist_raw(ctx: *mut gtp_ctx, ndim: c_int, xshape: *const u64, x: *const f64, yshape: *const u64, y: *const f64, rshape: *const u64, rows: *const u64, n_rows: u64, out_rows: *mut f64) -> c_int;
    pub fn gtp_mul_macs(ndim: c_int, xshape: *const u64, yshape: *const u64, rshape: *const u64) -> f64;
    pub fn gtp_mul_kernel_kind(ctx: *mut gtp_ctx, ndim: c_int, xshape: *const u64, yshape: *const u64, rshape: *const u64) -> c_int;
    pub fn gtp_fp64_peak_probe(ctx: *mut gtp_ctx, kind: c_int, iters: c_int, flops: *mut f64, ms: *mut f64) -> c_int;
    pub fn gtu_constant(ctx: *mut gtp_ctx, x: f64, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_from_coefficients(ctx: *mut gtp_ctx, xs: *const f64, n: u64, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_var(ctx: *mut gtp_ctx, x: f64, order: u64, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_free(ctx: *mut gtp_ctx, s: *mut gtu_series);
    pub fn gtu_is_constant(s: *const gtu_series) -> c_int;
    pub fn gtu_order(s: *const gtu_series) -> u64;
    pub fn gtu_to_host(ctx: *mut gtp_ctx, s: *const gtu_series, out: *mut f64) -> c_int;
    pub fn gtu_coeff(ctx: *mut gtp_ctx, s: *const gtu_series, order: u64, out: *mut f64) -> c_int;
    pub fn gtu_derivative(ctx: *mut gtp_ctx, s: *const gtu_series, order: u64, out: *mut f64) -> c_int;
    pub fn gtu_add(ctx: *mut gtp_ctx, a: *const gtu_series, b: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_sub(ctx: *mut gtp_ctx, a: *const gtu_series, b: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_mul(ctx: *mut gtp_ctx, a: *const gtu_series, b: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_div(ctx: *mut gtp_ctx, a: *const gtu_series, b: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_neg(ctx: *mut gtp_ctx, a: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_exp(ctx: *mut gtp_ctx, a: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_log(ctx: *mut gtp_ctx, a: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_pow(ctx: *mut gtp_ctx, a: *const gtu_series, exp: u32, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_subst(ctx: *mut gtp_ctx, a: *const gtu_series, subst: *const gtu_series, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_taylor_expansion_of_coeff(ctx: *mut gtp_ctx, a: *const gtu_series, n: u64, out: *mut *mut gtu_series) -> c_int;
    pub fn gtu_eq(ctx: *mut gtp_ctx, a: *const gtu_series, b: *const gtu_series, out: *mut c_int) -> c_int;
    pub fn gtu_program_create(ctx: *mut gtp_ctx, out: *mut *mut gtu_program) -> c_int;
    pub fn gtu_program_free(ctx: *mut gtp_ctx, p: *mut gtu_program);
    pub fn gtu_program_constant(ctx: *mut gtp_ctx, p: *mut gtu_program, x: f64, slot: *mut u32) -> c_int;
    pub fn gtu_program_var(ctx: *mut gtp_ctx, p: *mut gtu_program, x: f64, order: u64, slot: *mut u32) -> c_int;
    pub fn gtu_program_from_coefficients(ctx: *mut gtp_ctx, p: *mut gtu_program, xs: *const f64, n: u64, slot: *mut u32) -> c_int;
    pub fn gtu_program_op(ctx: *mut gtp_ctx, p: *mut gtu_program, op: c_int, a: u32, b: u32, exp: u32, slot: *mut u32) -> c_int;
    pub fn gtu_program_slot(p: *const gtu_program, slot: u32, is_constant: *mut c_int, n: *mut u64) -> c_int;
    pub fn gtu_program_run(ctx: *mut gtp_ctx, p: *mut gtu_program, outputs: *const u32, n_outputs: c_int, out: *mut f64) -> c_int;
    pub fn gtp_run_sgcl(ctx: *mut gtp_ctx, source: *const c_char, limit: i64, flags: c_int, unroll: u64, out: *mut *mut gtp_sgcl_result, err: *mut c_char, err_cap: usize) -> c_int;
    pub fn gtp_sgcl_free(r: *mut gtp_sgcl_result);
    pub fn gtp_sgcl_report(r: *const gtp_sgcl_result) -> *const c_char;
    pub fn gtp_sgcl_moments(r: *const gtp_sgcl_result, out11: *mut f64);
    pub fn gtp_sgcl_limit(r: *const gtp_sgcl_result) -> u64;
    pub fn gtp_sgcl_is_normalized(r: *const gtp_sgcl_result) -> c_int;
    pub fn gtp_sgcl_probs(r: *const gtp_sgcl_result, unnormalized: *mut f64, normalized: *mut f64);
    pub fn gtp_sgcl_stats(r: *const gtp_sgcl_result, nodes_evaluated: *mut u64, cache_hits: *mut u64);
    pub fn gtp_sgcl_moment_bounds(r: *const gtp_sgcl_result, out22: *mut f64);
    pub fn gtp_sgcl_prob_bounds(r: *const gtp_sgcl_result, unnormalized_pairs: *mut f64, normalized_pairs: *mut f64);
    pub fn gti_from_scalar(ctx: *mut gtp_ctx, lo: f64, hi: f64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_zero_with(ctx: *mut gtp_ctx, ndim: c_int, degrees_p1: *const u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_var(ctx: *mut gtp_ctx, v: u64, lo: f64, hi: f64, len: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_var_at_zero(ctx: *mut gtp_ctx, v: u64, len: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_var_with_degrees_p1(ctx: *mut gtp_ctx, v: u64, lo: f64, hi: f64, ndim: c_int, degrees_p1: *const u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_from_host(ctx: *mut gtp_ctx, ndim: c_int, shape: *const u64, degrees_p1: *const u64, data: *const f64, pairs: c_int, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_to_host(ctx: *mut gtp_ctx, p: *const gti_poly, out_pairs: *mut f64) -> c_int;
    pub fn gti_free(ctx: *mut gtp_ctx, p: *mut gti_poly);
    pub fn gti_ndim(p: *const gti_poly) -> c_int;
    pub fn gti_len(p: *const gti_poly) -> u64;
    pub fn gti_shape(p: *const gti_poly, out: *mut u64);
    pub fn gti_degrees_p1(p: *const gti_poly, out: *mut u64);
    pub fn gti_add(ctx: *mut gtp_ctx, a: *const gti_poly, b: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_sub(ctx: *mut gtp_ctx, a: *const gti_poly, b: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_mul(ctx: *mut gtp_ctx, a: *const gti_poly, b: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_div(ctx: *mut gtp_ctx, a: *const gti_poly, b: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_neg(ctx: *mut gtp_ctx, a: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_exp(ctx: *mut gtp_ctx, a: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_log(ctx: *mut gtp_ctx, a: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_pow(ctx: *mut gtp_ctx, a: *const gti_poly, e: u32, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_derivative(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, n: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_taylor_expansion_of_coeff(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, n: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_shift_down(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, n: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_coefficients_of_term(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, order: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_taylor_polynomial_terms(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, orders: *const u64, n_orders: c_int, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_subst_var(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, subst: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_truncate_to_degree_p1(ctx: *mut gtp_ctx, a: *const gti_poly, degree_p1: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_remove_last_variable(ctx: *mut gtp_ctx, a: *const gti_poly, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_extend_to_dim(ctx: *mut gtp_ctx, a: *const gti_poly, ndim: u64, degree_p1: u64, out: *mut *mut gti_poly) -> c_int;
    pub fn gti_constant_term(ctx: *mut gtp_ctx, a: *const gti_poly, out2: *mut f64) -> c_int;
    pub fn gti_extract_constant(ctx: *mut gtp_ctx, a: *const gti_poly, is_constant: *mut c_int, out2: *mut f64) -> c_int;
    pub fn gti_gather_axis(ctx: *mut gtp_ctx, a: *const gti_poly, v: u64, count: u64, out_pairs: *mut f64) -> c_int;
    pub fn gtp_run_sgcl_bounds(ctx: *mut gtp_ctx, source: *const c_char, limit: i64, unroll: u64, out12: *mut f64, probs_lohi: *mut f64, err: *mut c_char, err_cap: usize) -> c_int;
    // ---- END GENERATED ----
}

/// One CUDA device + stream; `Rc` because genfer is single threaded (`src/main.rs:96-106`).
pub struct Context(*mut gtp_ctx);
impl Context {
    pub fn new(device: i32) -> Rc<Self> {
        let mut h = ptr::null_mut();
        let rc = unsafe { gtp_ctx_create(device, ptr::null_mut(), &mut h) };
        assert!(rc == 0, "gtp_ctx_create failed ({rc}): no CUDA device -- there is no CPU fallback for the f64 Taylor path");
        Rc::new(Context(h))
    }
    /// Non-zero status becomes a panic, preserving the reference's `assert!` behaviour.
    fn check(&self, rc: c_int) {
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(gtp_last_error(self.0)) }.to_string_lossy().into_owned();
            panic!("libgenfer_taylor error {rc}: {msg}");
        }
    }
}
impl Drop for Context { fn drop(&mut self) { unsafe { gtp_ctx_destroy(self.0) } } }

/// Device-resident `TaylorPoly<F64>`; operators consume by value like the reference.
pub struct DevicePoly { ctx: Rc<Context>, h: *mut gtp_poly }
impl Drop for DevicePoly { fn drop(&mut self) { unsafe { gtp_free(self.ctx.0, self.h) } } }
impl Clone for DevicePoly {
    fn clone(&self) -> Self {
        let mut h = ptr::null_mut();
        self.ctx.check(unsafe { gtp_clone(self.ctx.0, self.h, &mut h) }); // O(1): buffers are immutable + ref-counted
        DevicePoly { ctx: self.ctx.clone(), h }
    }
}
macro_rules! binop { ($name:ident, $f:ident) => {
    pub fn $name(&self, o: &DevicePoly) -> DevicePoly {
        let mut h = ptr::null_mut();
        self.ctx.check(unsafe { $f(self.ctx.0, self.h, o.h, &mut h) });
        DevicePoly { ctx: self.ctx.clone(), h }
    } } }
macro_rules! unop { ($name:ident, $f:ident $(, $a:ident : $t:ty)*) => {
    pub fn $name(&self $(, $a: $t)*) -> DevicePoly {
        let mut h = ptr::null_mut();
        self.ctx.check(unsafe { $f(self.ctx.0, self.h $(, $a)*, &mut h) });
        DevicePoly { ctx: self.ctx.clone(), h }
    } } }
impl DevicePoly {
    /// `data` must be in standard (row-major, contiguous) layout: call `as_standard_layout()` on the
    /// ndarray first -- in-place slicing leaves owned arrays strided (multivariate_taylor.rs:85, :176).
    pub fn from_host(ctx: &Rc<Context>, shape: &[usize], degrees_p1: &[usize], data: &[f64]) -> Self {
        let s: Vec<u64> = shape.iter().map(|&x| x as u64).collect();
        let d: Vec<u64> = degrees_p1.iter().map(|&x| if x == usize::MAX { GTP_UNBOUNDED } else { x as u64 }).collect();
        assert_eq!(data.len(), shape.iter().product::<usize>());
        let mut h = ptr::null_mut();
        ctx.check(unsafe { gtp_from_host(ctx.0, s.len() as c_int, s.as_ptr(), d.as_ptr(), data.as_ptr(), &mut h) });
        DevicePoly { ctx: ctx.clone(), h }
    }
    pub fn to_host(&self) -> (Vec<usize>, Vec<f64>) {
        let n = unsafe { gtp_ndim(self.h) } as usize;
        let mut s = vec![0u64; n.max(1)];
        unsafe { gtp_shape(self.h, s.as_mut_ptr()) };
        let mut out = vec![0f64; unsafe { gtp_len(self.h) } as usize];
        self.ctx.check(unsafe { gtp_to_host(self.ctx.0, self.h, out.as_mut_ptr()) });
        (s[..n].iter().map(|&x| x as usize).collect(), out)
    }
    binop!(add, gtp_add); binop!(sub, gtp_sub); binop!(mul, gtp_mul); binop!(div, gtp_div);
    unop!(neg, gtp_neg); unop!(exp, gtp_exp); unop!(log, gtp_log); unop!(pow, gtp_pow, e: u32);
    unop!(derivative, gtp_derivative, v: u64, n: u64);
    unop!(taylor_expansion_of_coeff, gtp_taylor_expansion_of_coeff, v: u64, n: u64);
    unop!(shift_down, gtp_shift_down, v: u64, n: u64);
    unop!(coefficients_of_term, gtp_coefficients_of_term, v: u64, order: u64);
    unop!(truncate_to_degree_p1, gtp_truncate_to_degree_p1, d: u64);
    unop!(remove_last_variable, gtp_remove_last_variable);
    unop!(extend_to_dim, gtp_extend_to_dim, ndim: u64, d: u64);
    pub fn subst_var(&self, v: u64, subst: &DevicePoly) -> DevicePoly {
        let mut h = ptr::null_mut();
        self.ctx.check(unsafe { gtp_subst_var(self.ctx.0, self.h, v, subst.h, &mut h) });
        DevicePoly { ctx: self.ctx.clone(), h }
    }
    pub fn constant_term(&self) -> f64 {
        let mut x = 0.0;
        self.ctx.check(unsafe { gtp_constant_term(self.ctx.0, self.h, &mut x) });
        x
    }
    /// probs_taylor / moments_taylor read `limit` coefficients along one axis
    /// (generating_function.rs:959-965, :988-993): ONE gather + ONE copy instead of `limit` round trips.
    pub fn gather_axis(&self, v: u64, count: usize) -> Vec<f64> {
        let mut out = vec![0f64; count];
        self.ctx.check(unsafe { gtp_gather_axis(self.ctx.0, self.h, v, count as u64, out.as_mut_ptr()) });
        out
    }
}
