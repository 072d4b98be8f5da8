//! SOURCE ONLY (never compiled in this repository's environment: no rustc).
//! Hand-written `extern "C"` declarations mirroring `include/pg_b200.h` one to one (bindgen is not available either).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

/// `BlsScalar([u64; 4])`: Montgomery limbs, little endian.
#[repr(C)]
#[derive(Copy, Clone, Debug, Default, PartialEq, Eq)]
pub struct pg_fr {
    pub l: [u64; 4],
}
/// G1Affine { x, y } of dusk-bls12_381 without the infinity flag (all-zero = point at infinity).
/// The evaluations of prover round 4 (include/pg_b200.h): dusk-plonk 0.8 ProofEvaluations' fields in order, then quot_eval.
#[repr(C)]
#[derive(Copy, Clone, Debug, Default, PartialEq, Eq)]
pub struct pg_proof_evaluations {
    pub a_eval: pg_fr, pub b_eval: pg_fr, pub c_eval: pg_fr, pub d_eval: pg_fr,
    pub a_next_eval: pg_fr, pub b_next_eval: pg_fr, pub d_next_eval: pg_fr,
    pub q_arith_eval: pg_fr, pub q_c_eval: pg_fr, pub q_l_eval: pg_fr, pub q_r_eval: pg_fr,
    pub left_sigma_eval: pg_fr, pub right_sigma_eval: pg_fr, pub out_sigma_eval: pg_fr,
    pub lin_poly_eval: pg_fr, pub perm_eval: pg_fr, pub quot_eval: pg_fr,
}

#[repr(C)]
#[derive(Copy, Clone, Debug, Default, PartialEq, Eq)]
pub struct pg_g1_affine {
    pub x: [u64; 6],
    pub y: [u64; 6],
}
#[repr(C)]
pub struct pg_ctx {
    _private: [u8; 0],
}
pub type pg_col = u64;

pub const PG_FORM_EVALUATIONS: c_int = 0;
pub const PG_FORM_COEFFICIENTS: c_int = 1;
pub const PG_OK: c_int = 0;
pub const PG_ERR_NON_EXISTING_INVERSE: c_int = 1;
pub const PG_ERR_CUDA: c_int = -1;
pub const PG_ERR_ARG: c_int = -2;
pub const PG_ERR_OOM: c_int = -3;
pub const PG_ERR_MIXED_BITS: c_int = -4;
pub const PG_ERR_NO_DEVICE: c_int = -5;
pub const PG_ERR_STATE: c_int = -6;
pub const PG_CHECK_GENERIC: i32 = 0;
pub const PG_CHECK_SPARSE: i32 = 1;
pub const PG_F_TIMING: u32 = 1;

#[repr(C)]
pub struct pg_cfg {
    pub device: i32,
    pub check_mode: i32,
    pub flags: u32,
    /// UNSTABLE tuning knob (launch shape of the gate-check kernels); keep 0.
    pub check_shape: u32,
    pub stream: *mut c_void,
}
#[repr(C)]
#[derive(Default)]
pub struct pg_timing {
    pub check_ms: f64,
    pub witness_ms: f64,
    pub other_ms: f64,
    pub check_launches: u64,
    pub witness_launches: u64,
    pub other_launches: u64,
    pub check_rows: u64,
}

pub const PG_NZ_UNIFORM: c_int = 0;
pub const PG_NZ_REFERENCE: c_int = 1;
pub const PG_CK_KINDS: usize = 8;
#[repr(C)]
#[derive(Default)]
pub struct pg_check_stats {
    pub launches: [u64; PG_CK_KINDS],
    pub rows: [u64; PG_CK_KINDS],
}

// ---- multi-GPU: sharding plan and collectives
pub const PG_OP_ADD_INPUT: u32 = 0;
pub const PG_OP_RANGE_CHECK: u32 = 1;
pub const PG_OP_MAX_BOUND: u32 = 2;
pub const PG_OP_MAYBE_EQUAL: u32 = 3;
pub const PG_OP_IS_NON_ZERO: u32 = 4;
pub const PG_OP_SELECT_ZERO: u32 = 5;
pub const PG_OP_SELECT_ONE: u32 = 6;
pub const PG_OP_CONSTRAIN: u32 = 7;
pub const PG_OP_RANGE_GATE: u32 = 8;
pub const PG_SHARD_EVEN: c_int = 0;
pub const PG_SHARD_ROWS: c_int = 1;
pub const PG_COMM_ID_BYTES: usize = 128;
#[repr(C)]
#[derive(Copy, Clone, Debug, Default)]
pub struct pg_op {
    pub gadget: u32,
    pub num_bits: u32,
    pub n: u64,
    pub group: u32,
    pub reserved: u32,
}
#[repr(C)]
#[derive(Copy, Clone, Debug, Default, PartialEq, Eq)]
pub struct pg_op_shard {
    pub inst_lo: u64,
    pub inst_hi: u64,
    pub row_base: u64,
    pub var_base: u64,
}

extern "C" {
    pub fn pg_template_get(gadget: u32, num_bits: u32, a: *const pg_fr, b: *const pg_fr, n_rows: *mut u64, n_vars: *mut u64, w_ref: *mut i64,
                           sel: *mut pg_fr, gate: *mut u32) -> c_int;
    pub fn pg_op_shape(gadget: u32, num_bits: u32, rows: *mut u64, vars: *mut u64) -> c_int;
    pub fn pg_shard_plan(ops: *const pg_op, n_ops: u64, world: u32, policy: c_int, out: *mut pg_op_shard) -> c_int;
    pub fn pg_comm_unique_id(id: *mut u8) -> c_int;
    pub fn pg_comm_init(ctx: *mut pg_ctx, id: *const u8, rank: u32, world: u32) -> c_int;
    pub fn pg_comm_destroy(ctx: *mut pg_ctx) -> c_int;
    pub fn pg_check_sharded(ctx: *mut pg_ctx, mine: *const pg_op_shard, n_ops: u64, n_unsat: *mut u64, first_bad_row: *mut u64,
                            n_err: *mut u64) -> c_int;
    pub fn pg_gather_column(ctx: *mut pg_ctx, col: pg_col, dst: *mut pg_fr, capacity: u64, dst_on_device: c_int, counts: *mut u64,
                            total: *mut u64) -> c_int;
    pub fn pg_gather_variables(ctx: *mut pg_ctx, call: u64, dst: *mut pg_fr, capacity: u64, dst_on_device: c_int, total: *mut u64) -> c_int;
    pub fn pg_export_composer(ctx: *mut pg_ctx, path: *const c_char, chunk_rows: u64, flags: u32) -> c_int;
    pub fn pg_abi_version() -> c_int;
    pub fn pg_strerror(code: c_int) -> *const c_char;
    pub fn pg_last_error(ctx: *const pg_ctx) -> *const c_char;
    pub fn pg_ctx_create(cfg: *const pg_cfg, out: *mut *mut pg_ctx) -> c_int;
    pub fn pg_ctx_destroy(ctx: *mut pg_ctx);
    pub fn pg_composer_reset(ctx: *mut pg_ctx) -> c_int;
    pub fn pg_sync(ctx: *mut pg_ctx) -> c_int;
    pub fn pg_add_input_batch(ctx: *mut pg_ctx, n: u64, values: *const pg_fr, on_device: c_int, out: *mut pg_col) -> c_int;
    pub fn pg_range_check_batch(ctx: *mut pg_ctx, min_range: *const pg_fr, max_range: *const pg_fr, n_bounds: u64, on_device: c_int,
                                witness: pg_col, out: *mut pg_col, num_bits: *mut u64) -> c_int;
    pub fn pg_max_bound_batch(ctx: *mut pg_ctx, max_range: *const pg_fr, n_bounds: u64, on_device: c_int, witness: pg_col,
                              out: *mut pg_col, num_bits: *mut u64) -> c_int;
    pub fn pg_maybe_equal_batch(ctx: *mut pg_ctx, a: pg_col, b: pg_col, out: *mut pg_col) -> c_int;
    pub fn pg_is_non_zero_batch(ctx: *mut pg_ctx, var: pg_col, value_assigned: *const pg_fr, on_device: c_int, n_err: *mut u64,
                                first_err: *mut u64) -> c_int;
    pub fn pg_is_non_zero_batch_flags(ctx: *mut pg_ctx, var: pg_col, value_assigned: *const pg_fr, on_device: c_int, err_flags: *mut u8,
                                      layout: c_int, n_err: *mut u64) -> c_int;
    pub fn pg_select_zero_batch(ctx: *mut pg_ctx, x: pg_col, select: pg_col, out: *mut pg_col) -> c_int;
    pub fn pg_select_one_batch(ctx: *mut pg_ctx, y: pg_col, selector: pg_col, out: *mut pg_col) -> c_int;
    pub fn pg_constrain_to_constant_batch(ctx: *mut pg_ctx, a: pg_col, constant: *const pg_fr, n_const: u64, pi: *const pg_fr,
                                          n_pi: u64, on_device: c_int) -> c_int;
    pub fn pg_range_gate_batch(ctx: *mut pg_ctx, witness: pg_col, num_bits: u32) -> c_int;
    pub fn pg_check(ctx: *mut pg_ctx, n_unsat: *mut u64, first_bad_row: *mut u64) -> c_int;
    pub fn pg_check_rows(ctx: *mut pg_ctx, n: u64, w_val: *const pg_fr, sel: *const pg_fr, pi: *const pg_fr, on_device: c_int,
                         n_unsat: *mut u64, first_bad_row: *mut u64) -> c_int;
    pub fn pg_counts(ctx: *const pg_ctx, n_rows: *mut u64, n_vars: *mut u64) -> c_int;
    pub fn pg_col_info(ctx: *const pg_ctx, col: pg_col, n: *mut u64, first_var: *mut u64, stride: *mut u64) -> c_int;
    pub fn pg_col_read(ctx: *mut pg_ctx, col: pg_col, i0: u64, cnt: u64, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_read_variables(ctx: *mut pg_ctx, var0: u64, cnt: u64, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_materialize_rows(ctx: *mut pg_ctx, row0: u64, cnt: u64, w_idx: *mut u64, w_val: *mut pg_fr, sel: *mut pg_fr,
                               pi: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_check_rows_ex(ctx: *mut pg_ctx, n: u64, w_val: *const pg_fr, sel: *const pg_fr, pi: *const pg_fr, q_arith: *const pg_fr,
                            q_range: *const pg_fr, on_device: c_int, n_unsat: *mut u64, first_bad_row: *mut u64) -> c_int;
    pub fn pg_poke_variable(ctx: *mut pg_ctx, var: u64, value: *const pg_fr) -> c_int;
    pub fn pg_materialize_gate_selectors(ctx: *mut pg_ctx, row0: u64, cnt: u64, q_arith: *mut pg_fr, q_range: *mut pg_fr,
                                         dst_on_device: c_int) -> c_int;
    pub fn pg_permutation(ctx: *mut pg_ctx, row0: u64, cnt: u64, sigma: *mut u64, dst_on_device: c_int) -> c_int;
    pub fn pg_fft(ctx: *mut pg_ctx, log_n: u32, inverse: c_int, src: *const pg_fr, dst: *mut pg_fr, on_device: c_int) -> c_int;
    pub fn pg_wire_polynomials(ctx: *mut pg_ctx, log_n: u32, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_sigma_polynomials(ctx: *mut pg_ctx, log_n: u32, form: c_int, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_permutation_z(ctx: *mut pg_ctx, log_n: u32, beta: *const pg_fr, gamma: *const pg_fr, form: c_int, dst: *mut pg_fr,
                            dst_on_device: c_int, closing: *mut pg_fr) -> c_int;
    pub fn pg_permutation_z_rows(ctx: *mut pg_ctx, log_n: u32, n: u64, w_val: *const pg_fr, sigma: *const u64, on_device: c_int,
                                 beta: *const pg_fr, gamma: *const pg_fr, form: c_int, dst: *mut pg_fr, dst_on_device: c_int,
                                 closing: *mut pg_fr) -> c_int;
    pub fn pg_selector_polynomials(ctx: *mut pg_ctx, log_n: u32, form: c_int, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_public_input_polynomial(ctx: *mut pg_ctx, log_n: u32, form: c_int, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_quotient(ctx: *mut pg_ctx, log_n: u32, alpha: *const pg_fr, beta: *const pg_fr, gamma: *const pg_fr, range_challenge: *const pg_fr,
                       dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_prover_openings(ctx: *mut pg_ctx, log_n: u32, challenges: *const pg_fr, t: *const pg_fr, t_on_device: c_int,
                              evals: *mut pg_proof_evaluations, dst: *mut pg_fr, dst_on_device: c_int) -> c_int;
    pub fn pg_msm(ctx: *mut pg_ctx, n: u64, points: *const pg_g1_affine, scalars: *const pg_fr, out: *mut pg_g1_affine, on_device: c_int) -> c_int;
    pub fn pg_srs_powers(ctx: *mut pg_ctx, beta: *const pg_fr, base: *const pg_g1_affine, n: u64, out: *mut pg_g1_affine, out_on_device: c_int) -> c_int;
    pub fn pg_g1_fixed_base_mul(ctx: *mut pg_ctx, n: u64, base: *const pg_g1_affine, scalars: *const pg_fr, out: *mut pg_g1_affine,
                                on_device: c_int) -> c_int;
    pub fn pg_commit_wire_polynomials(ctx: *mut pg_ctx, log_n: u32, powers_of_g: *const pg_g1_affine, n_powers: u64, powers_on_device: c_int,
                                      out4: *mut pg_g1_affine) -> c_int;
    pub fn pg_srs_lagrange(ctx: *mut pg_ctx, beta: *const pg_fr, base: *const pg_g1_affine, log_n: u32, out: *mut pg_g1_affine, out_on_device: c_int) -> c_int;
    pub fn pg_srs_lagrange_from_powers(ctx: *mut pg_ctx, log_n: u32, powers_of_g: *const pg_g1_affine, n_powers: u64, powers_on_device: c_int,
                                       out: *mut pg_g1_affine, out_on_device: c_int) -> c_int;
    pub fn pg_commit_wire_evaluations(ctx: *mut pg_ctx, log_n: u32, lagrange: *const pg_g1_affine, n_points: u64, points_on_device: c_int,
                                      out4: *mut pg_g1_affine) -> c_int;
    pub fn pg_g1_op(ctx: *mut pg_ctx, op: c_int, n: u64, a: *const pg_g1_affine, b: *const pg_g1_affine, out: *mut pg_g1_affine) -> c_int;
    pub fn pg_fr_to_bytes(ctx: *mut pg_ctx, n: u64, src: *const pg_fr, dst: *mut u8, on_device: c_int) -> c_int;
    pub fn pg_fr_from_bytes(ctx: *mut pg_ctx, n: u64, src: *const u8, dst: *mut pg_fr, on_device: c_int, n_invalid: *mut u64,
                            first_invalid: *mut u64) -> c_int;
    pub fn pg_synth(ctx: *mut pg_ctx, seed: u64, stream: u64, n: u64, kind: c_int, bits: u32, dst_device: *mut pg_fr) -> c_int;
    pub fn pg_get_timing(ctx: *mut pg_ctx, out: *mut pg_timing, reset: c_int) -> c_int;
    pub fn pg_get_check_stats(ctx: *mut pg_ctx, out: *mut pg_check_stats, reset: c_int) -> c_int;
    pub fn pg_measure_imad_peak(ctx: *mut pg_ctx, wide_mac_per_s: *mut f64, imad_per_s: *mut f64) -> c_int;
    pub fn pg_microbench(ctx: *mut pg_ctx, mode: c_int, ops_per_s: *mut f64) -> c_int;
    pub fn pg_fr_op(ctx: *mut pg_ctx, op: c_int, n: u64, a: *const pg_fr, b: *const pg_fr, out: *mut pg_fr) -> c_int;
}
