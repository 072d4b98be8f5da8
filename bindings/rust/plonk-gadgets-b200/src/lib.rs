//! SOURCE ONLY (never compiled in this repository's environment).
//!
//! The reference crate (`plonk_gadgets`) stays untouched -- `#![deny(unsafe_code)]` and `#![no_std]` forbid FFI inside
//! it (/root/reference/src/lib.rs:32-33) -- and remains the one-instance path: `AllocatedScalar`, `range_check`,
//! `max_bound`, `is_non_zero`, `maybe_equal`, `conditionally_select_one/zero` keep their signatures.  This crate adds the
//! batched variants with the same names suffixed `_batch`, over a device-resident `BatchComposer`.
//!
//! `Variable(pub(crate) usize)` cannot be forged outside dusk-plonk, so batched calls return `Variables` (a column id plus
//! the reference's Variable numbering `first + i*stride`) instead of `Variable`s.
pub mod import;
use dusk_plonk::prelude::BlsScalar;
pub use plonk_gadgets::{AllocatedScalar, Error};
use plonk_gadgets_b200_sys as sys;
use std::{ffi::CStr, ptr};

/// Engine failures (negative codes of the C ABI).  Never mapped to a gadget `Error`, never a silent CPU fallback.
#[derive(Debug)]
pub struct EngineError {
    pub code: i32,
    pub detail: String,
}

/// `Error::NonExistingInverse` of a batched `is_non_zero`, with what a batch adds: how many instances failed, and the first.
#[derive(Debug)]
pub struct NonZeroBatchError {
    pub error: Error,
    pub n_err: u64,
    pub first_err: u64,
}

/// n `Variable`s, one per gadget instance of the call that produced them.
#[derive(Copy, Clone, Debug)]
pub struct Variables {
    pub col: sys::pg_col,
    pub n: u64,
}

/// Device-resident batched `StandardComposer` (fresh: 3 rows, 5 variables -- `StandardComposer::new()`).
pub struct BatchComposer {
    ctx: *mut sys::pg_ctx,
}

fn as_fr(s: &[BlsScalar]) -> *const sys::pg_fr {
    // BlsScalar is `pub struct Scalar(pub [u64; 4])`: same layout as pg_fr
    s.as_ptr() as *const sys::pg_fr
}

impl BatchComposer {
    pub fn new(device: i32) -> Result<Self, EngineError> {
        let cfg = sys::pg_cfg { device, check_mode: sys::PG_CHECK_GENERIC, flags: 0, check_shape: 0, stream: ptr::null_mut() };
        let mut ctx = ptr::null_mut();
        let rc = unsafe { sys::pg_ctx_create(&cfg, &mut ctx) };
        if rc != sys::PG_OK {
            let detail = unsafe { CStr::from_ptr(sys::pg_strerror(rc)) }.to_string_lossy().into_owned();
            return Err(EngineError { code: rc, detail });
        }
        Ok(BatchComposer { ctx })
    }
    fn ok(&self, rc: i32) -> Result<i32, EngineError> {
        if rc < 0 {
            let detail = unsafe { CStr::from_ptr(sys::pg_last_error(self.ctx)) }.to_string_lossy().into_owned();
            Err(EngineError { code: rc, detail })
        } else {
            Ok(rc)
        }
    }
    /// `AllocatedScalar::allocate` over n scalars.
    pub fn allocate_batch(&mut self, scalars: &[BlsScalar]) -> Result<Variables, EngineError> {
        let mut col = 0;
        self.ok(unsafe { sys::pg_add_input_batch(self.ctx, scalars.len() as u64, as_fr(scalars), 0, &mut col) })?;
        Ok(Variables { col, n: scalars.len() as u64 })
    }
    /// `range_check(composer, min_range, max_range, witness)` for every element of `witness`.
    pub fn range_check_batch(&mut self, min_range: BlsScalar, max_range: BlsScalar, witness: Variables) -> Result<Variables, EngineError> {
        let (mut col, mut k) = (0, 0);
        self.ok(unsafe { sys::pg_range_check_batch(self.ctx, as_fr(&[min_range]), as_fr(&[max_range]), 1, 0, witness.col, &mut col, &mut k) })?;
        Ok(Variables { col, n: witness.n })
    }
    /// `range_check` with one `(min_range, max_range)` pair per instance; all pairs must give the same `num_bits`
    /// (`EngineError { code: PG_ERR_MIXED_BITS, .. }` otherwise, nothing appended).
    pub fn range_check_batch_per_instance(&mut self, min_range: &[BlsScalar], max_range: &[BlsScalar], witness: Variables) -> Result<(Variables, u64), EngineError> {
        assert!(min_range.len() as u64 == witness.n && max_range.len() as u64 == witness.n);
        let (mut col, mut k) = (0, 0);
        self.ok(unsafe { sys::pg_range_check_batch(self.ctx, as_fr(min_range), as_fr(max_range), witness.n, 0, witness.col, &mut col, &mut k) })?;
        Ok((Variables { col, n: witness.n }, k))
    }
    /// `max_bound(composer, max_range, witness) -> (Variable, u64)`.
    pub fn max_bound_batch(&mut self, max_range: BlsScalar, witness: Variables) -> Result<(Variables, u64), EngineError> {
        let (mut col, mut k) = (0, 0);
        self.ok(unsafe { sys::pg_max_bound_batch(self.ctx, as_fr(&[max_range]), 1, 0, witness.col, &mut col, &mut k) })?;
        Ok((Variables { col, n: witness.n }, k))
    }
    pub fn maybe_equal_batch(&mut self, a: Variables, b: Variables) -> Result<Variables, EngineError> {
        let mut col = 0;
        self.ok(unsafe { sys::pg_maybe_equal_batch(self.ctx, a.col, b.col, &mut col) })?;
        Ok(Variables { col, n: a.n })
    }
    /// `for i { is_non_zero(composer, var_i, value_assigned_i)?; }` -- `Ok(Err(..))` mirrors the gadget error of the first zero
    /// `value_assigned` (the composer then holds what that loop leaves behind); the error carries how many instances of the batch
    /// have a zero `value_assigned` and the index of the first one.
    pub fn is_non_zero_batch(&mut self, var: Variables, value_assigned: &[BlsScalar]) -> Result<Result<(), NonZeroBatchError>, EngineError> {
        let (mut n_err, mut first_err) = (0, 0);
        let rc = self.ok(unsafe { sys::pg_is_non_zero_batch(self.ctx, var.col, as_fr(value_assigned), 0, &mut n_err, &mut first_err) })?;
        Ok(if rc == sys::PG_ERR_NON_EXISTING_INVERSE { Err(NonZeroBatchError { error: Error::NonExistingInverse, n_err, first_err }) } else { Ok(()) })
    }
    /// `value_assigned.iter().map(|v| is_non_zero(composer, var_i, *v))` with every `Result` kept: the batch does not stop at a
    /// zero.  `reference_layout`: errored calls leave the 1 variable + 1 row the reference appends before returning `Err`
    /// (ragged numbering); otherwise every instance appends 3 variables + 3 rows and an errored one fails its last row.
    pub fn is_non_zero_each(&mut self, var: Variables, value_assigned: &[BlsScalar], reference_layout: bool) -> Result<Vec<Result<(), Error>>, EngineError> {
        let mut flags = vec![0u8; value_assigned.len()];
        let mut n_err = 0;
        let layout = if reference_layout { sys::PG_NZ_REFERENCE } else { sys::PG_NZ_UNIFORM };
        self.ok(unsafe { sys::pg_is_non_zero_batch_flags(self.ctx, var.col, as_fr(value_assigned), 0, flags.as_mut_ptr(), layout, &mut n_err) })?;
        Ok(flags.iter().map(|&f| if f != 0 { Err(Error::NonExistingInverse) } else { Ok(()) }).collect())
    }
    pub fn conditionally_select_zero_batch(&mut self, x: Variables, select: Variables) -> Result<Variables, EngineError> {
        let mut col = 0;
        self.ok(unsafe { sys::pg_select_zero_batch(self.ctx, x.col, select.col, &mut col) })?;
        Ok(Variables { col, n: x.n })
    }
    pub fn conditionally_select_one_batch(&mut self, y: Variables, selector: Variables) -> Result<Variables, EngineError> {
        let mut col = 0;
        self.ok(unsafe { sys::pg_select_one_batch(self.ctx, y.col, selector.col, &mut col) })?;
        Ok(Variables { col, n: y.n })
    }
    /// `for w in witness { composer.range_gate(w, num_bits) }` -- dusk-plonk's native quad-accumulator range gate (the path
    /// `plonk_gadgets::range` recommends for power-of-two bounds).  `num_bits` even, 2..=256.
    pub fn range_gate_batch(&mut self, witness: Variables, num_bits: usize) -> Result<(), EngineError> {
        self.ok(unsafe { sys::pg_range_gate_batch(self.ctx, witness.col, num_bits as u32) })?;
        Ok(())
    }
    /// Satisfaction verdict: (unsatisfied rows, first unsatisfied row).
    pub fn check(&mut self) -> Result<(u64, Option<u64>), EngineError> {
        let (mut bad, mut first) = (0, 0);
        self.ok(unsafe { sys::pg_check(self.ctx, &mut bad, &mut first) })?;
        Ok((bad, if first == u64::MAX { None } else { Some(first) }))
    }
    /// Joins the communicator of the box's ranks (one process and one `BatchComposer` per GPU).  `id`: `comm_unique_id()` of rank 0.
    pub fn comm_init(&mut self, id: &[u8; sys::PG_COMM_ID_BYTES], rank: u32, world: u32) -> Result<(), EngineError> {
        self.ok(unsafe { sys::pg_comm_init(self.ctx, id.as_ptr(), rank, world) })?;
        Ok(())
    }
    /// Verdict of the WHOLE sharded circuit on every rank: local gate check, then the NCCL all-reduce (sum of unsatisfied rows and of
    /// `NonExistingInverse` errors, min of the first bad row in the sequential composer's numbering).  `mine`: this rank's row of
    /// `shard_plan(..)`; `n_err`: this rank's error count.
    pub fn check_sharded(&mut self, mine: &[sys::pg_op_shard], n_err: u64) -> Result<(u64, Option<u64>, u64), EngineError> {
        let (mut bad, mut first, mut err) = (0, 0, n_err);
        self.ok(unsafe { sys::pg_check_sharded(self.ctx, mine.as_ptr(), mine.len() as u64, &mut bad, &mut first, &mut err) })?;
        Ok((bad, if first == u64::MAX { None } else { Some(first) }, err))
    }
    /// All-gather of a column's values (per-instance results of a call) from every rank, in instance order of the whole batch.
    pub fn gather_column(&mut self, v: Variables, total: usize) -> Result<Vec<BlsScalar>, EngineError> {
        let mut out = vec![BlsScalar::zero(); total];
        let mut got = 0u64;
        self.ok(unsafe { sys::pg_gather_column(self.ctx, v.col, out.as_mut_ptr() as *mut sys::pg_fr, total as u64, 0, std::ptr::null_mut(), &mut got) })?;
        out.truncate(got as usize);
        Ok(out)
    }
    /// Gather of witness shards: the Variables batched call number `call` appended on every rank, in the sequential composer's order.
    pub fn gather_variables(&mut self, call: u64, total: usize) -> Result<Vec<BlsScalar>, EngineError> {
        let mut out = vec![BlsScalar::zero(); total];
        let mut got = 0u64;
        self.ok(unsafe { sys::pg_gather_variables(self.ctx, call, out.as_mut_ptr() as *mut sys::pg_fr, total as u64, 0, &mut got) })?;
        out.truncate(got as usize);
        Ok(out)
    }
    /// Writes the whole composer (calls, Variable values, wire ids, selector columns, dense PI) to `path` for `import::import_into`.
    pub fn export(&mut self, path: &std::path::Path, with_sigma: bool) -> Result<(), EngineError> {
        let c = std::ffi::CString::new(path.to_str().expect("utf-8 path")).expect("no NUL in path");
        self.ok(unsafe { sys::pg_export_composer(self.ctx, c.as_ptr(), 0, if with_sigma { 1 } else { 0 }) })?;
        Ok(())
    }
    /// Rows and variables appended so far (`circuit_size()`, `variables.len()`).
    pub fn counts(&self) -> (u64, u64) {
        let (mut rows, mut vars) = (0, 0);
        unsafe { sys::pg_counts(self.ctx, &mut rows, &mut vars) };
        (rows, vars)
    }
    /// log2 of `EvaluationDomain::new(circuit_size).size()`.
    pub fn domain_log_size(&self) -> u32 {
        self.counts().0.next_power_of_two().trailing_zeros()
    }
    /// Prover round 1, first half: coefficients of w_l, w_r, w_o, w_4 (`domain.ifft` of the zero-padded wire columns),
    /// four vectors of 2^log_n scalars.
    pub fn wire_polynomials(&mut self, log_n: u32) -> Result<Vec<Vec<BlsScalar>>, EngineError> {
        let n = 1usize << log_n;
        let mut flat = vec![BlsScalar::zero(); 4 * n];
        self.ok(unsafe { sys::pg_wire_polynomials(self.ctx, log_n, flat.as_mut_ptr() as *mut sys::pg_fr, 0) })?;
        Ok(flat.chunks(n).map(|c| c.to_vec()).collect())
    }
    /// Preprocessing's sigma polynomials (`compute_permutation_lagrange`, or with `coefficients` `compute_sigma_polynomials`) of
    /// the composer's rows over the domain 2^log_n: four vectors of 2^log_n scalars.
    pub fn sigma_polynomials(&mut self, log_n: u32, coefficients: bool) -> Result<Vec<Vec<BlsScalar>>, EngineError> {
        let n = 1usize << log_n;
        let form = if coefficients { sys::PG_FORM_COEFFICIENTS } else { sys::PG_FORM_EVALUATIONS };
        let mut flat = vec![BlsScalar::zero(); 4 * n];
        self.ok(unsafe { sys::pg_sigma_polynomials(self.ctx, log_n, form, flat.as_mut_ptr() as *mut sys::pg_fr, 0) })?;
        Ok(flat.chunks(n).map(|c| c.to_vec()).collect())
    }
    /// Prover round 2: the grand-product polynomial z over the domain 2^log_n (`compute_fast_permutation_poly`, or with
    /// `coefficients` `compute_permutation_poly`) for the transcript's beta and gamma, and the product of all 2^log_n ratios
    /// (one on every composer this API builds).
    pub fn permutation_z(&mut self, log_n: u32, beta: &BlsScalar, gamma: &BlsScalar, coefficients: bool) -> Result<(Vec<BlsScalar>, BlsScalar), EngineError> {
        let form = if coefficients { sys::PG_FORM_COEFFICIENTS } else { sys::PG_FORM_EVALUATIONS };
        let mut z = vec![BlsScalar::zero(); 1usize << log_n];
        let mut closing = BlsScalar::zero();
        self.ok(unsafe {
            sys::pg_permutation_z(self.ctx, log_n, beta as *const BlsScalar as *const sys::pg_fr, gamma as *const BlsScalar as *const sys::pg_fr, form,
                                  z.as_mut_ptr() as *mut sys::pg_fr, 0, &mut closing as *mut BlsScalar as *mut sys::pg_fr)
        })?;
        Ok((z, closing))
    }
    /// Preprocessing's selector polynomials q_m q_l q_r q_o q_4 q_c q_arith q_range (padding rows zero) over the domain 2^log_n,
    /// evaluations or (`coefficients`) their ifft: eight vectors of 2^log_n scalars.
    pub fn selector_polynomials(&mut self, log_n: u32, coefficients: bool) -> Result<Vec<Vec<BlsScalar>>, EngineError> {
        let n = 1usize << log_n;
        let form = if coefficients { sys::PG_FORM_COEFFICIENTS } else { sys::PG_FORM_EVALUATIONS };
        let mut flat = vec![BlsScalar::zero(); 8 * n];
        self.ok(unsafe { sys::pg_selector_polynomials(self.ctx, log_n, form, flat.as_mut_ptr() as *mut sys::pg_fr, 0) })?;
        Ok(flat.chunks(n).map(|c| c.to_vec()).collect())
    }
    /// `construct_dense_pi_vec` padded to 2^log_n, or (`coefficients`) PI(X).
    pub fn public_input_polynomial(&mut self, log_n: u32, coefficients: bool) -> Result<Vec<BlsScalar>, EngineError> {
        let form = if coefficients { sys::PG_FORM_COEFFICIENTS } else { sys::PG_FORM_EVALUATIONS };
        let mut pi = vec![BlsScalar::zero(); 1usize << log_n];
        self.ok(unsafe { sys::pg_public_input_polynomial(self.ctx, log_n, form, pi.as_mut_ptr() as *mut sys::pg_fr, 0) })?;
        Ok(pi)
    }
    /// Prover round 3: t_1 .. t_4 (`split_tx_poly`), four vectors of 2^log_n coefficients, for the transcript's alpha, beta, gamma
    /// and range separation challenge; log_n <= 30.
    pub fn quotient(&mut self, log_n: u32, alpha: &BlsScalar, beta: &BlsScalar, gamma: &BlsScalar, range_challenge: &BlsScalar)
                    -> Result<Vec<Vec<BlsScalar>>, EngineError> {
        let n = 1usize << log_n;
        let mut flat = vec![BlsScalar::zero(); 4 * n];
        let p = |x: &BlsScalar| x as *const BlsScalar as *const sys::pg_fr;
        self.ok(unsafe { sys::pg_quotient(self.ctx, log_n, p(alpha), p(beta), p(gamma), p(range_challenge), flat.as_mut_ptr() as *mut sys::pg_fr, 0) })?;
        Ok(flat.chunks(n).map(|c| c.to_vec()).collect())
    }
    /// Prover rounds 4 and 5 for round 3's t_1 .. t_4 and the transcript's alpha, beta, gamma, range separation challenge, z_challenge
    /// and the two aggregation challenges v (opening at z) and v' (opening at z*w): the evaluations, and W_z, W_zw and r as
    /// vectors of 2^log_n coefficients; log_n <= 30.
    pub fn prover_openings(&mut self, log_n: u32, t: &[Vec<BlsScalar>], challenges: &[BlsScalar; 7])
                           -> Result<(sys::pg_proof_evaluations, Vec<Vec<BlsScalar>>), EngineError> {
        let n = 1usize << log_n;
        assert!(t.len() == 4 && t.iter().all(|c| c.len() == n), "t: four vectors of 2^log_n coefficients");
        let flat_t: Vec<BlsScalar> = t.iter().flatten().copied().collect();
        let mut ev = sys::pg_proof_evaluations::default();
        let mut flat = vec![BlsScalar::zero(); 3 * n];
        self.ok(unsafe {
            sys::pg_prover_openings(self.ctx, log_n, challenges.as_ptr() as *const sys::pg_fr, flat_t.as_ptr() as *const sys::pg_fr, 0, &mut ev,
                                    flat.as_mut_ptr() as *mut sys::pg_fr, 0)
        })?;
        Ok((ev, flat.chunks(n).map(|c| c.to_vec()).collect()))
    }
    /// Prover round 1, second half: `commit_key.commit(&w_l_poly)` .. `w_4`.  `powers_of_g` are the CommitKey's G1Affine
    /// powers in the layout of `sys::pg_g1_affine` (x, y Montgomery limbs; all-zero = infinity).
    pub fn commit_wire_polynomials(&mut self, log_n: u32, powers_of_g: &[sys::pg_g1_affine]) -> Result<[sys::pg_g1_affine; 4], EngineError> {
        let mut out = [sys::pg_g1_affine::default(); 4];
        self.ok(unsafe { sys::pg_commit_wire_polynomials(self.ctx, log_n, powers_of_g.as_ptr(), powers_of_g.len() as u64, 0, out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// The Lagrange-basis form of the SRS for the domain 2^log_n from the CommitKey's monomial powers alone (beta unknown):
    /// `out[i] = (1/n) sum_j w^(-ij) powers_of_g[j]` over the first n = 2^log_n powers, by an inverse FFT over G1 on the GPU.
    pub fn srs_lagrange_from_powers(&mut self, log_n: u32, powers_of_g: &[sys::pg_g1_affine]) -> Result<Vec<sys::pg_g1_affine>, EngineError> {
        let n = if log_n <= 32 { 1usize << log_n } else { 0 };           // log_n > 32: the call returns PG_ERR_ARG
        let mut out = vec![sys::pg_g1_affine::default(); n];
        self.ok(unsafe {
            sys::pg_srs_lagrange_from_powers(self.ctx, log_n, powers_of_g.as_ptr(), powers_of_g.len() as u64, 0, out.as_mut_ptr(), 0)
        })?;
        Ok(out)
    }
    /// The same four commitments from the wire values against the Lagrange-basis form of the SRS (`lagrange[i] = L_i(beta) * g`,
    /// exactly 2^log_n points): no FFT, and bits / short accumulators leave most windows of the multi-scalar multiplication empty.
    pub fn commit_wire_evaluations(&mut self, log_n: u32, lagrange: &[sys::pg_g1_affine]) -> Result<[sys::pg_g1_affine; 4], EngineError> {
        let mut out = [sys::pg_g1_affine::default(); 4];
        self.ok(unsafe { sys::pg_commit_wire_evaluations(self.ctx, log_n, lagrange.as_ptr(), lagrange.len() as u64, 0, out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// `msm_variable_base(points, scalars)`.
    pub fn msm(&mut self, points: &[sys::pg_g1_affine], scalars: &[BlsScalar]) -> Result<sys::pg_g1_affine, EngineError> {
        assert_eq!(points.len(), scalars.len());
        let mut out = sys::pg_g1_affine::default();
        self.ok(unsafe { sys::pg_msm(self.ctx, points.len() as u64, points.as_ptr(), as_fr(scalars), &mut out, 0) })?;
        Ok(out)
    }
    /// `composer.variables[var]` of a column.
    pub fn values(&mut self, v: Variables) -> Result<Vec<BlsScalar>, EngineError> {
        let mut out = vec![BlsScalar::zero(); v.n as usize];
        self.ok(unsafe { sys::pg_col_read(self.ctx, v.col, 0, v.n, out.as_mut_ptr() as *mut sys::pg_fr, 0) })?;
        Ok(out)
    }
}
/// `ncclGetUniqueId` through the C ABI: rank 0 calls it and hands the bytes to the other ranks (any channel).
pub fn comm_unique_id() -> Option<[u8; sys::PG_COMM_ID_BYTES]> {
    let mut id = [0u8; sys::PG_COMM_ID_BYTES];
    if unsafe { sys::pg_comm_unique_id(id.as_mut_ptr()) } == sys::PG_OK { Some(id) } else { None }
}
/// Splits a mixed circuit (a list of batched calls) over `world` GPUs: `plan[rank][k]` = the instance range of call k that rank runs
/// and the row / Variable index of its first instance in the sequential composer (prefix sums over the calls).  Pure host code.
pub fn shard_plan(ops: &[sys::pg_op], world: u32, by_rows: bool) -> Option<Vec<Vec<sys::pg_op_shard>>> {
    let mut flat = vec![sys::pg_op_shard::default(); ops.len() * world as usize];
    let policy = if by_rows { sys::PG_SHARD_ROWS } else { sys::PG_SHARD_EVEN };
    if unsafe { sys::pg_shard_plan(ops.as_ptr(), ops.len() as u64, world, policy, flat.as_mut_ptr()) } != sys::PG_OK { return None; }
    Some(flat.chunks(ops.len().max(1)).map(|c| c.to_vec()).collect())
}
impl Drop for BatchComposer {
    fn drop(&mut self) {
        unsafe { sys::pg_ctx_destroy(self.ctx) }
    }
}
