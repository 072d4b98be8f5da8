/*
 * pg_b200.h -- C ABI of the B200-native batched gadget engine for plonk_gadgets' hot path
 * (witness generation + arithmetic-gate constraint evaluation over BLS12-381 Fr).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch/C++ types.  A Rust `-sys` crate binds exactly these
 * symbols (see INTEGRATION.md); the C++ mirror of the reference API lives in plonk_gadgets_b200/host/plonk_gadgets.hpp
 * and the Python (ctypes) mirror used by the tests in plonk_gadgets_b200/api.py.
 *
 * The reference has no FFI of its own: its "operator interface" is the crate's public Rust functions, all of which take
 * `composer: &mut StandardComposer` first.  Each entry point below cites the reference function it replaces; `ref:` is a path
 * inside the dusk-network/plonk_gadgets v0.6.0 source tree (ref:src/range.rs:27 = src/range.rs line 27 of that crate), [dusk-plonk]
 * marks behaviour of its dusk-plonk 0.8 dependency.
 *
 * Model.  A pg_ctx owns ONE device-resident composer (dusk-plonk StandardComposer, arithmetic-row subset) on one GPU.
 * Every *_batch call appends n independent gadget instances and is defined to be EQUAL to the sequential program
 *         for i in 0..n { gadget(&mut composer, .., operand_i) }
 * run on the reference composer: same Variable numbering, same wire columns, same selector rows, same values.
 * Operands that are `Variable`s in the reference are *columns* here (pg_col): the n variables, one per instance, that an
 * earlier call produced.  The composer is stored as (row template per gadget and bit width) x (per-instance variable
 * table in structure-of-arrays form, bits packed); pg_materialize_rows / pg_read_variables expand any range of it into
 * the reference's own representation (`Vec<BlsScalar>` columns, `Vec<Variable>` wires).
 *
 * Scalars cross the boundary as pg_fr: the raw in-memory form of `BlsScalar([u64;4])` (little-endian limbs of
 * a*2^256 mod q, fully reduced).  Inputs must be fully reduced (< q), as every BlsScalar is.  Single scalars (uniform bounds,
 * constants, pg_poke_variable) are checked on the host: PG_ERR_ARG.  Batches are checked on the device by the kernel that ingests
 * them, without a synchronisation: an unreduced scalar is counted, and the next call that reads the device counters -- pg_check,
 * pg_sync, pg_is_non_zero_batch*, a range gadget with per-instance bounds, pg_fr_from_bytes, pg_check_rows* -- returns PG_ERR_ARG
 * (pg_last_error names the count and the first index).  The composer then holds values the reference type cannot represent:
 * reset it.
 *
 * A mixed circuit is a sequence of *_batch calls on one ctx (each call one "op" of n instances): there is no separate
 * pg_circuit_run(op list) entry point, the composer model is that list.  pg_shard_plan splits such a list over GPUs.
 *
 * Threading: a pg_ctx is not thread-safe (the reference API is `&mut`).  All work is enqueued on the ctx's CUDA
 * stream; calls that return host values synchronise that stream.  There is no CPU fallback: every entry point fails
 * with PG_ERR_NO_DEVICE / PG_ERR_CUDA when the GPU is unavailable.
 */
#ifndef PG_B200_H
#define PG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PG_B200_ABI_VERSION 7

/* BlsScalar: ref:src/allocated_scalar.rs:9-12 (dusk_plonk::bls12_381::BlsScalar) */
typedef struct pg_fr { uint64_t l[4]; } pg_fr;

typedef struct pg_ctx pg_ctx;

/* A column of variables: variable `i` of the column is the one instance i of the producing call allocated.
 * 0 is never a valid column. */
typedef uint64_t pg_col;

/* Return codes.  > 0 : gadget-level errors of the reference (ref:src/errors.rs:13-18).
 *                < 0 : engine errors (never a silent fallback). */
enum {
    PG_OK = 0,
    PG_ERR_NON_EXISTING_INVERSE = 1, /* Error::NonExistingInverse, ref:src/scalar.rs:79 */
    PG_ERR_CUDA = -1,                /* a CUDA call failed; pg_last_error() has the driver's message */
    PG_ERR_ARG = -2,                 /* bad argument (null pointer, unknown column, length mismatch, ...) */
    PG_ERR_OOM = -3,                 /* device allocation failed */
    PG_ERR_MIXED_BITS = -4,          /* per-instance bounds of one call do not share one bit width (num_bits) */
    PG_ERR_NO_DEVICE = -5,           /* no CUDA device / wrong architecture */
    PG_ERR_STATE = -6                /* call not valid in the composer's current state */
};

/* How the gate equation is evaluated by pg_check (results are identical; only the work differs):
 *   GENERIC : q_m*a*b + q_l*a + q_r*b + q_o*c + q_4*d + q_c + PI for arbitrary selector values, no selector inspected (what
 *             dusk-plonk's check_circuit_satisfied / quotient evaluation do); evaluated as a*(q_m*b + q_l) + q_r*b + q_o*c +
 *             q_4*d with one Montgomery multiplication and one four-term dot product sharing a single reduction.
 *   SPARSE  : structure-aware.  Decisions are taken on the row TEMPLATE (never on witness data): a term whose selector is the
 *             constant 0, or whose wire is the zero variable, is skipped (the wire is not loaded); selectors +-1 become add / sub;
 *             a wire that is one of the 256 packed bit variables of a decomposition is read as the bit the table stores for it,
 *             i.e. it is boolean by construction (b*b = b: the boolean_gate rows of ref:src/range.rs:144 fold to "holds").  Those
 *             variables cannot be overwritten through pg_poke_variable, so the assumption cannot be violated from outside.
 *             Runs of rows  sel_j*bit_j + x_j - x_{j+1} = 0  over consecutive Variables (the accumulator rows of ref:src/range.rs:146-152)
 *             are evaluated as one loop with x_{j+1} kept in registers (one 32-byte load per row), as  x_j + t == x_{j+1} (mod q)
 *             without a reduction.  Rows of the range widget (pg_range_gate_batch): D(f) = f(f-1)(f-2)(f-3) vanishes iff f is a base-4
 *             digit, so a row whose four differences are digits holds without a multiplication; any other row is evaluated through
 *             the polynomial.  Same verdict as GENERIC on every composer state this API can produce. */
enum { PG_CHECK_GENERIC = 0, PG_CHECK_SPARSE = 1 };

enum {
    PG_F_TIMING = 1u,       /* record CUDA events around every kernel class (pg_get_timing) */
    PG_F_FUSED_CHECK = 2u   /* with PG_CHECK_SPARSE: the gadgets' witness kernels also evaluate the rows they generate (on the values they hold
                               in registers, structure-aware arithmetic) -- range_check, max_bound, maybe_equal, is_non_zero (the _flags call in
                               the uniform layout), conditionally_select_* -- so the variable table is written once and never read again for
                               the verdict; pg_check / pg_check_sharded then only launch for what was not verified that way (the fresh rows,
                               constrain_to_constant and range_gate rows, is_non_zero with `?` semantics) and add the recorded verdict.
                               pg_poke_variable drops the record: every segment present at that moment goes back to the check kernels (calls
                               made afterwards are recorded afresh).  Same verdict as without the flag on every composer state this API can
                               produce. */
};

typedef struct pg_cfg {
    int32_t device;         /* CUDA ordinal */
    int32_t check_mode;     /* PG_CHECK_* */
    uint32_t flags;         /* PG_F_* */
    uint32_t check_shape;   /* UNSTABLE tuning knob, keep 0: launch shape (threads x blocks per SM, loads in flight) of the gate-check kernels
                               (1..4 = alternatives, kernels.cuh CheckShape / ProgDepth); never changes results */
    void *stream;           /* cudaStream_t to enqueue on; NULL = the engine creates its own non-blocking stream */
} pg_cfg;

/* ---- lifetime --------------------------------------------------------------------------------------------------- */
int pg_abi_version(void);
const char *pg_strerror(int code);
const char *pg_last_error(const pg_ctx *ctx);          /* detail of the last engine error on this ctx ("" if none) */
/* StandardComposer::new() [dusk-plonk]: zero variable + two dummy rows => 3 rows, 5 variables (SURVEY.md App. A.2) */
int pg_ctx_create(const pg_cfg *cfg, pg_ctx **out);
void pg_ctx_destroy(pg_ctx *ctx);
/* Back to a fresh composer; device buffers are kept in the ctx's pool for reuse. */
int pg_composer_reset(pg_ctx *ctx);
/* Blocks until everything enqueued so far has finished. */
int pg_sync(pg_ctx *ctx);

/* ---- gadgets ------------------------------------------------------------------------------------------------------
 * `on_device` != 0: the pointer arguments of the call are 32-byte aligned device pointers on cfg.device (read asynchronously on the
 * ctx stream; keep them alive until pg_sync); == 0: host pointers (copied with cudaMemcpyAsync; pinned memory makes that copy
 * asynchronous -- keep the buffer alive and unchanged until the next call that returns data or pg_sync).  pg_add_input_batch copies
 * host batches of 2^20 scalars or more in chunks on a separate input stream, and a range gadget called on that column next starts on
 * the chunks that have arrived; every other operation waits for the whole copy first. */

/* AllocatedScalar::allocate / composer.add_input over n scalars -- ref:src/allocated_scalar.rs:27-30.
 * Appends n variables, no rows. */
int pg_add_input_batch(pg_ctx *ctx, uint64_t n, const pg_fr *values, int on_device, pg_col *out);

/* range_check(composer, min_range, max_range, witness) -- ref:src/range.rs:27-43.
 * n_bounds == 1: one public (min,max) pair for all instances; n_bounds == n: per-instance bounds, which must all give the
 * same num_bits (else PG_ERR_MIXED_BITS and nothing is appended).  Per instance 4k+11 rows, 2k+523 variables.
 * *out: the returned Variable (value 1 iff min <= x < max within k bits); *num_bits: k (may be NULL). */
int pg_range_check_batch(pg_ctx *ctx, const pg_fr *min_range, const pg_fr *max_range, uint64_t n_bounds, int on_device,
                         pg_col witness, pg_col *out, uint64_t *num_bits);

/* max_bound(composer, max_range, witness) -> (Variable, u64) -- ref:src/range.rs:82-113.  2k+5 rows, k+261 vars. */
int pg_max_bound_batch(pg_ctx *ctx, const pg_fr *max_range, uint64_t n_bounds, int on_device, pg_col witness,
                       pg_col *out, uint64_t *num_bits);

/* maybe_equal(composer, a, b) -- ref:src/scalar.rs:105-140.  3 rows, 3 variables; *out = 1 iff a == b.
 * (The AllocatedScalar's host-side `scalar` is the column's own value.) */
int pg_maybe_equal_batch(pg_ctx *ctx, pg_col a, pg_col b, pg_col *out);

/* for i { is_non_zero(composer, var_i, value_assigned_i)?; } -- ref:src/scalar.rs:63-97.
 * 3 rows, 3 variables per instance.  If some value_assigned is zero the call returns PG_ERR_NON_EXISTING_INVERSE and the
 * composer holds what the reference loop leaves behind: the instances before the first zero complete, plus the
 * 1 variable + 1 row the failing call had already appended (scalar.rs:69-71).  *n_err = number of zero values in the
 * whole batch, *first_err = index of the first one (either may be NULL). */
int pg_is_non_zero_batch(pg_ctx *ctx, pg_col var, const pg_fr *value_assigned, int on_device, uint64_t *n_err,
                         uint64_t *first_err);

/* for i { results[i] = is_non_zero(composer, var_i, value_assigned_i); } -- ref:src/scalar.rs:63-97 with every Result KEPT instead of
 * propagated with `?`: a batch does not abort on one zero (ref:src/errors.rs:13-18).  err_flags (n bytes, host or device memory like
 * value_assigned; may be NULL): 1 where the call returned Err(NonExistingInverse), else 0; *n_err = their number.  Returns PG_OK.
 *   PG_NZ_UNIFORM  : every instance appends the full 3 variables + 3 rows (Variable numbering stays first + 3*i).  For an errored
 *                    instance: var_assigned = 0, inv = 0 (invert().unwrap_or(zero), the convention of ref:src/scalar.rs:122), one = 1;
 *                    its row var*inv - 1 = 0 is unsatisfied, so pg_check reports it too.  One segment, one kernel launch.  This is NOT
 *                    what the reference appends for an errored call; it is the layout for throughput (BASELINE config C4).
 *   PG_NZ_REFERENCE: the composer that loop leaves behind, bit for bit: an errored call has appended var_assigned and the assert_equal
 *                    row only (1 variable + 1 row, ref:src/scalar.rs:69-71 before the return at :79), so numbering is ragged.  The
 *                    device table is described as 2*n_err + 1 segment views; cost grows with n_err (at most 2^19 errors). */
enum { PG_NZ_UNIFORM = 0, PG_NZ_REFERENCE = 1 };
int pg_is_non_zero_batch_flags(pg_ctx *ctx, pg_col var, const pg_fr *value_assigned, int on_device, uint8_t *err_flags, int layout,
                               uint64_t *n_err);

/* conditionally_select_zero(composer, x, select) -- ref:src/scalar.rs:21-27.  1 row, 1 variable. */
int pg_select_zero_batch(pg_ctx *ctx, pg_col x, pg_col select, pg_col *out);
/* conditionally_select_one(composer, y, selector) -- ref:src/scalar.rs:36-59.  4 rows, 4 variables. */
int pg_select_one_batch(pg_ctx *ctx, pg_col y, pg_col selector, pg_col *out);

/* composer.constrain_to_constant(a, constant, pi) [dusk-plonk] as used by the reference's tests
 * (ref:tests/range_gadgets_tests.rs:26,:43; tests/scalar_gadgets_tests.rs:30,:78,:135).  1 row, no variable.
 * n_const / n_pi: 1 (uniform) or n; pi == NULL: no public input. */
int pg_constrain_to_constant_batch(pg_ctx *ctx, pg_col a, const pg_fr *constant, uint64_t n_const, const pg_fr *pi,
                                   uint64_t n_pi, int on_device);

/* for i { composer.range_gate(witness_i, num_bits); } -- StandardComposer::range_gate [dusk-plonk 0.8 src/constraint_system/range.rs],
 * the native quad-accumulator range gate that ref:src/range.rs:9-12 recommends over range_check when the bound is a
 * power of two (SURVEY.md section 8f item 4).  Per instance: num_bits/2 accumulator variables a_j = 4*a_{j-1} + quad_j (base-4
 * digits of the witness, most significant first) laid out four per gate on w_4, w_o, w_r, w_l after 1..4 leading zero wires;
 * ceil(num_bits/8) gates with q_range = 1 (all arithmetic selectors and q_arith 0), one closing gate with q_range = 0, and
 * assert_equal(last accumulator, witness): ceil(num_bits/8) + 2 rows.  The circuit is satisfied iff the witness < 2^num_bits.
 * num_bits must be even (the reference asserts) and in 2..256, else PG_ERR_ARG.  Nothing is returned (the reference returns ()). */
int pg_range_gate_batch(pg_ctx *ctx, pg_col witness, uint32_t num_bits);

/* ---- verdict ------------------------------------------------------------------------------------------------------ */
/* Arithmetic and range parts of check_circuit_satisfied [dusk-plonk]: evaluates, on every row of the composer,
 *   q_arith*(q_m*a*b + q_l*a + q_r*b + q_o*c + q_4*d + PI + q_c) + q_range*(D(c - 4d) + D(b - 4c) + D(a - 4b) + D(d_next - 4a)),
 * D(f) = f(f-1)(f-2)(f-3), d_next = fourth wire of the next row (q_range is non-zero only on rows appended by pg_range_gate_batch).
 * *n_unsat = number of rows with a non-zero value; *first_bad_row = smallest such row index or UINT64_MAX. */
int pg_check(pg_ctx *ctx, uint64_t *n_unsat, uint64_t *first_bad_row);
/* Same equation over caller-supplied materialised rows (w_val: 4 x n wire values, sel: 6 x n selectors in the order
 * q_m q_l q_r q_o q_4 q_c, pi: n or NULL), column-major. */
int pg_check_rows(pg_ctx *ctx, uint64_t n, const pg_fr *w_val, const pg_fr *sel, const pg_fr *pi, int on_device,
                  uint64_t *n_unsat, uint64_t *first_bad_row);

/* The full equation of pg_check (arithmetic + range widget) over caller-supplied rows: q_arith and q_range are n scalars each
 * (NULL q_arith = 1 everywhere, NULL q_range = 0 everywhere); d_next of row i is w_val[3][(i + 1) mod n]. */
int pg_check_rows_ex(pg_ctx *ctx, uint64_t n, const pg_fr *w_val, const pg_fr *sel, const pg_fr *pi, const pg_fr *q_arith,
                     const pg_fr *q_range, int on_device, uint64_t *n_unsat, uint64_t *first_bad_row);

/* ---- row templates ------------------------------------------------------------------------------------------------------------
 * What ONE instance of a gadget appends, in the reference's order (SURVEY.md 8a: the structure depends only on public data -- the
 * property the reference's verifier-side circuit rebuild relies on, ref:tests/scalar_gadgets_tests.rs:43,:60): pure host code, no ctx.
 * a / b: the public scalars of the call -- range_check: (min_range, max_range); max_bound: (NULL, max_range); constrain_to_constant:
 * (pi or NULL, constant); others: ignored.  num_bits: range_gate's width; for range_check / max_bound 0 or the width the bound implies.
 * w_ref (4 x n_rows, column-major w_l w_r w_o w_4): 0 = the zero variable, 1 + j = the j-th Variable the instance allocates,
 * -1 - e = operand e (witness / a, b / x, select / var).  sel (6 x n_rows): q_m q_l q_r q_o q_4 q_c.  gate (n_rows): 0 arithmetic
 * (q_arith = 1), 1 range widget (q_range = 1), 2 neither.  Output buffers may be NULL (sizes only). */
int pg_template_get(uint32_t gadget, uint32_t num_bits, const pg_fr *a, const pg_fr *b, uint64_t *n_rows, uint64_t *n_vars,
                    int64_t *w_ref, pg_fr *sel, uint32_t *gate);

/* ---- multi-GPU: sharding plan and the two collectives (SURVEY.md section 8e) -------------------------------------------------
 * One process and one pg_ctx per GPU.  Gadget instances are independent (ref:src/range.rs:119-158 allocates its own accumulators,
 * ref:src/scalar.rs:41, :83 their own constant one), so the instances of every batched call are cut into contiguous ranges, one per
 * rank; a rank makes the same sequence of *_batch calls on its ranges.  No communication inside the kernels; the ranks meet in
 *   - the all-reduce of the verdict (sum of unsatisfied rows and of NonExistingInverse errors, min of the first bad row), and
 *   - the gather of per-instance results / witness shards,
 * both NCCL over NVLink 5 / NVSwitch on the ctx's stream (NCCL is bound at run time: "libnccl.so.2").
 *
 * pg_shard_plan is pure host code (no ctx, no GPU): a mixed circuit is a list of calls (pg_op: gadget, num_bits for the range
 * gadgets, instance count, group); calls with the same `group` share one instance index space (an add_input column and the gadgets
 * applied to it) and are cut at the same places.  out[rank * n_ops + k] = the instance range of call k that `rank` runs, and the
 * row / Variable index its first instance has in the SEQUENTIAL composer of the whole circuit (3 rows + 5 variables of the fresh
 * composer, then call after call: prefix sums of n * rows / n * variables per instance) -- the numbering the reference would
 * produce.  Policies: PG_SHARD_EVEN cuts every group into equal instance ranges; PG_SHARD_ROWS lays the groups end to end weighted by
 * rows per instance and cuts that line into equal parts at instance boundaries, so a rank owns a contiguous ~1/world of the rows. */
enum { PG_OP_ADD_INPUT = 0, PG_OP_RANGE_CHECK = 1, PG_OP_MAX_BOUND = 2, PG_OP_MAYBE_EQUAL = 3, PG_OP_IS_NON_ZERO = 4,
       PG_OP_SELECT_ZERO = 5, PG_OP_SELECT_ONE = 6, PG_OP_CONSTRAIN = 7, PG_OP_RANGE_GATE = 8 };
enum { PG_SHARD_EVEN = 0, PG_SHARD_ROWS = 1 };
typedef struct pg_op { uint32_t gadget; uint32_t num_bits; uint64_t n; uint32_t group; uint32_t reserved; } pg_op;
typedef struct pg_op_shard { uint64_t inst_lo, inst_hi; uint64_t row_base, var_base; } pg_op_shard;
/* rows and variables one instance of the gadget appends (SURVEY.md 8a: range_check 4k+11 / 2k+523, max_bound 2k+5 / k+261, ...) */
int pg_op_shape(uint32_t gadget, uint32_t num_bits, uint64_t *rows, uint64_t *vars);
int pg_shard_plan(const pg_op *ops, uint64_t n_ops, uint32_t world, int policy, pg_op_shard *out);

/* Communicator of the ranks of one box.  pg_comm_unique_id (rank 0; no ctx needed) fills a 128-byte id to be handed to the other
 * ranks out of band; every rank then calls pg_comm_init on its ctx (collective).  Without a communicator the calls below behave as a
 * world of one rank and NCCL is never loaded. */
#define PG_COMM_ID_BYTES 128
int pg_comm_unique_id(uint8_t *id);
int pg_comm_init(pg_ctx *ctx, const uint8_t *id, uint32_t rank, uint32_t world);
int pg_comm_destroy(pg_ctx *ctx);
/* pg_check on a sharded composer followed by the all-reduce: every rank receives the verdict of the WHOLE circuit.  mine = this
 * rank's row of the plan (n_ops entries; call k since the last reset must be op k and hold inst_hi - inst_lo instances): rows are
 * numbered from row_base, so *first_bad_row is the index in the sequential composer; mine == NULL: local numbering.  The fresh
 * composer's three rows are checked by rank 0 only.  *n_err: in = this rank's NonExistingInverse count, out = the sum (may be NULL). */
int pg_check_sharded(pg_ctx *ctx, const pg_op_shard *mine, uint64_t n_ops, uint64_t *n_unsat, uint64_t *first_bad_row, uint64_t *n_err);
/* All-gather of a column (per-instance results of a call): dst receives the shards of all ranks in rank order = instance order of
 * the whole batch.  capacity: scalars dst can hold (PG_ERR_ARG if too small); counts: `world` entries or NULL; *total = their sum. */
int pg_gather_column(pg_ctx *ctx, pg_col col, pg_fr *dst, uint64_t capacity, int dst_on_device, uint64_t *counts, uint64_t *total);
/* Gather of witness shards: the Variables that call number `call` (0-based since the last reset) appended on every rank, in the
 * sequential composer's Variable order -- variables[var_base of rank 0's shard ...) of that call. */
int pg_gather_variables(pg_ctx *ctx, uint64_t call, pg_fr *dst, uint64_t capacity, int dst_on_device, uint64_t *total);

/* ---- reading the composer back in the reference's representation --------------------------------------------------- */
int pg_counts(const pg_ctx *ctx, uint64_t *n_rows, uint64_t *n_vars);        /* composer.circuit_size(), variables.len() */
/* Column geometry: Variable id of instance i = first_var + i * stride. */
int pg_col_info(const pg_ctx *ctx, pg_col col, uint64_t *n, uint64_t *first_var, uint64_t *stride);
/* Values of instances [i0, i0+cnt) of a column (what `composer.variables[var]` holds).
 * dst_on_device: 0 = host memory (returns when the data has arrived), 1 = device memory, 2 = PINNED host memory, asynchronous:
 * the copy runs on a second stream, overlaps with kernels enqueued afterwards (e.g. pg_check) and is complete after pg_sync. */
int pg_col_read(pg_ctx *ctx, pg_col col, uint64_t i0, uint64_t cnt, pg_fr *dst, int dst_on_device);
/* variables[var0 .. var0+cnt) in Variable order. */
int pg_read_variables(pg_ctx *ctx, uint64_t var0, uint64_t cnt, pg_fr *dst, int dst_on_device);
/* Rows [row0, row0+cnt): any of the outputs may be NULL.  w_idx: 4 x cnt Variable ids (w_l,w_r,w_o,w_4), w_val: 4 x cnt
 * wire values, sel: 6 x cnt (q_m,q_l,q_r,q_o,q_4,q_c), pi: cnt (dense public inputs), all column-major.  On every row
 * q_logic = q_fixed_group_add = q_variable_group_add = 0; q_arith = 1 and q_range = 0 except on the rows of pg_range_gate_batch
 * (pg_materialize_gate_selectors returns those two columns). */
int pg_materialize_rows(pg_ctx *ctx, uint64_t row0, uint64_t cnt, uint64_t *w_idx, pg_fr *w_val, pg_fr *sel, pg_fr *pi,
                        int dst_on_device);

/* q_arith and q_range of rows [row0, row0+cnt) (cnt scalars each; either pointer may be NULL). */
int pg_materialize_gate_selectors(pg_ctx *ctx, uint64_t row0, uint64_t cnt, pg_fr *q_arith, pg_fr *q_range, int dst_on_device);

/* ---- copy constraints (SURVEY.md section 8f item 1) ----------------------------------------------------------------------
 * The permutation argument's input: dusk-plonk appends the four wire positions of every row to perm.variable_map[var]
 * (add_variables_to_map, called by every gate method listed above) and links the positions of one Variable into a cycle.
 * sigma is 4 x cnt, column-major: sigma[w*cnt + t] = successor, in that cycle, of wire w (0 w_l, 1 w_r, 2 w_o, 3 w_4) of
 * row row0 + t, encoded as row*4 + wire.  A position whose Variable is used once maps to itself, and so do the three zero wires
 * (w_l, w_r, w_o) of a range gate's closing row, which dusk-plonk pushes without a map entry. */
int pg_permutation(pg_ctx *ctx, uint64_t row0, uint64_t cnt, uint64_t *sigma, int dst_on_device);

/* ---- composer export (SURVEY.md section 8f item 1: the import adapter's input) -----------------------------------------------
 * The reference's tests hand the composer to dusk-plonk: prover.mut_cs() -> gadget calls -> preprocess -> prove
 * (ref:tests/range_gadgets_tests.rs:82-91).  `Variable(pub(crate) usize)` cannot be forged outside dusk-plonk, so a batch built here
 * reaches a real StandardComposer by REPLAY: pg_export_composer writes the whole composer -- the list of calls, every Variable's value
 * as BlsScalar::to_bytes, and per row the four wire Variables, q_m q_l q_r q_o q_4 q_c q_arith q_range and the dense public input
 * (construct_dense_pi_vec, ref:tests/scalar_gadgets_tests.rs:151), optionally the permutation (flags bit 0) -- to one little-endian
 * file, in chunks of chunk_rows rows (0 = 2^20); layout: csrc/engine.hpp export_composer.  bindings/rust/plonk-gadgets-b200/src/import.rs
 * (source only) replays it with add_input / poly_gate / range_gate and checks the Variable numbering as it goes. */
enum { PG_EXPORT_SIGMA = 1u };
int pg_export_composer(pg_ctx *ctx, const char *path, uint64_t chunk_rows, uint32_t flags);

/* ---- evaluation domain (SURVEY.md section 8f item 2, first half) -------------------------------------------------------------
 * The step that follows the gadget hot path inside Prover::prove [DEP dusk-plonk 0.8, reached from
 * ref:tests/range_gadgets_tests.rs:90-91 and tests/scalar_gadgets_tests.rs (prover.prove)]:
 *     let w_l_scalar = &[&self.to_scalars(&self.cs.w_l)[..], &pad].concat();       // pad = zeros up to domain.size()
 *     let w_l_poly = Polynomial::from_coefficients_vec(domain.ifft(w_l_scalar));   // same for w_r, w_o, w_4
 * pg_fft is EvaluationDomain::fft (inverse == 0) / ifft (inverse != 0) [DEP src/fft/domain.rs] of a vector of 2^log_n
 * scalars, natural order in and out, over the subgroup generated by ROOT_OF_UNITY^(2^(32-log_n)), ROOT_OF_UNITY =
 * 7^((q-1)/2^32); log_n <= 32 (TWO_ADICITY) or PG_ERR_ARG.  src and dst are both host or both device pointers and may be
 * the same buffer.
 * pg_wire_polynomials writes the coefficient vectors of w_l, w_r, w_o, w_4 (4 x 2^log_n scalars, column-major) for the
 * composer's current rows; 2^log_n must be >= the circuit size (EvaluationDomain::new(circuit_size) takes the next power of
 * two: pass ceil(log2(n_rows)) for the reference's domain).  Their commitments: next section. */
int pg_fft(pg_ctx *ctx, uint32_t log_n, int inverse, const pg_fr *src, pg_fr *dst, int on_device);
int pg_wire_polynomials(pg_ctx *ctx, uint32_t log_n, pg_fr *dst, int dst_on_device);

/* ---- permutation argument (SURVEY.md section 8f item 2, continued) ----------------------------------------------------------
 * Preprocessing's sigma polynomials and round 2 of Prover::prove [DEP dusk-plonk 0.8 src/permutation/permutation.rs, recalled
 * like the rest of [DEP]].  Domain H = <w> of size N = 2^log_n as in pg_fft; rows n_rows .. N are padding (wire value 0, every
 * position a fixed point of sigma: pad() pushes zero-variable wires without touching the variable map -- recalled, unpinned).
 * Coset constants k = (1, K1, K2, K3) = (1, 7, 13, 17) for w_l, w_r, w_o, w_4 (permutation/constants.rs, recalled); the identity of
 * wire position (i, w) is k_w * w^i.
 * pg_sigma_polynomials: sigma_w(w^i) = k_{w'} * w^{r'}, r'*4 + w' = pg_permutation's successor of (i, w)
 *   (compute_permutation_lagrange); PG_FORM_COEFFICIENTS: domain.ifft of that (compute_sigma_polynomials).  dst: 4 x N, column-major.
 * pg_permutation_z: with wire values v_w(i) and the caller's beta, gamma (host pointers; the transcript is not built):
 *     num_i = prod_w (v_w(i) + beta*k_w*w^i + gamma),  den_i = prod_w (v_w(i) + beta*sigma_w(w^i) + gamma)
 *     z_0 = 1,  z_{i+1} = z_i * num_i / den_i                      (compute_fast_permutation_poly; coefficients: compute_permutation_poly)
 *   dst: N scalars.  *closing (host, may be NULL) = prod_{i<N} num_i / den_i, the element the reference drops: 1 on every composer
 *   this API builds, for any beta and gamma.  A zero den_i (the reference panics in invert().unwrap(), e.g. beta = gamma = 0 on a row
 *   with the zero variable) is PG_ERR_ARG and pg_last_error names the first such row.
 * Both: PG_ERR_ARG when 2^log_n < the circuit size or log_n > 32, or beta / gamma is not fully reduced; PG_ERR_STATE on a ctx with a
 *   communicator of more than one rank (a sharded z needs the other ranks' carries: not built).  They synchronise the ctx stream.
 * pg_permutation_z_rows: the same over caller-supplied rows (the pg_check_rows counterpart): w_val 4 x n wire values, sigma 4 x n
 *   positions in pg_permutation's encoding (row*4 + wire), column-major, both host or both device memory; rows n .. N are padding.
 *   A sigma entry >= 4*N or an unreduced wire value is counted on the device and reported as PG_ERR_ARG by this call. */
enum { PG_FORM_EVALUATIONS = 0, PG_FORM_COEFFICIENTS = 1 };
int pg_sigma_polynomials(pg_ctx *ctx, uint32_t log_n, int form, pg_fr *dst, int dst_on_device);
int pg_permutation_z(pg_ctx *ctx, uint32_t log_n, const pg_fr *beta, const pg_fr *gamma, int form, pg_fr *dst, int dst_on_device,
                     pg_fr *closing);
int pg_permutation_z_rows(pg_ctx *ctx, uint32_t log_n, uint64_t n, const pg_fr *w_val, const uint64_t *sigma, int on_device,
                          const pg_fr *beta, const pg_fr *gamma, int form, pg_fr *dst, int dst_on_device, pg_fr *closing);

/* ---- quotient polynomial (SURVEY.md section 8f item 2, continued) ------------------------------------------------------------
 * Preprocessing's selector and public-input polynomials and round 3 of Prover::prove [DEP dusk-plonk 0.8 src/proof_system/
 * quotient_poly.rs (compute, compute_circuit_satisfiability_equation, compute_permutation_checks, split_tx_poly), recalled like
 * the rest of [DEP]: parity unpinned].  H = <w> of size N = 2^log_n as above; rows n_rows .. N are padding with zero wires,
 * zero selectors (q_arith included) and zero PI (pad(), recalled).
 * pg_selector_polynomials: q_m q_l q_r q_o q_4 q_c q_arith q_range of rows 0 .. N, 8 x N column-major, PG_FORM_EVALUATIONS or the
 *   domain.ifft of each (PG_FORM_COEFFICIENTS).  q_logic, q_fixed_group_add and q_variable_group_add are 0 on every row (see
 *   pg_materialize_rows): their polynomials and widget terms vanish.
 * pg_public_input_polynomial: the dense public inputs (construct_dense_pi_vec) padded to N, or their ifft PI(X): N scalars.
 * pg_quotient: with the caller's challenges alpha, beta, gamma and the range separation challenge rho (host pointers to one scalar
 *   each; the transcript is not built), kappa = rho^2, Delta(f) = f(f-1)(f-2)(f-3), k = (1, 7, 13, 17), L_1(X) = (X^N - 1)/(N(X - 1)),
 *   z(X) = pg_permutation_z's polynomial for the same beta, gamma, and at every point x of the coset g*<zeta> (zeta^4 = w, g = 7 =
 *   dusk-bls12_381 GENERATOR; EvaluationDomain::coset_fft of the 4N domain):
 *     arith = q_arith (q_m a b + q_l a + q_r b + q_o c + q_4 d + q_c) + PI                 (PI outside the q_arith factor)
 *     range = rho q_range (Delta(c - 4d) + kappa Delta(b - 4c) + kappa^2 Delta(a - 4b) + kappa^3 Delta(d(xw) - 4a))
 *     perm  = alpha z(x) prod_w (v_w + beta k_w x + gamma) - alpha z(xw) prod_w (v_w + beta sigma_w(x) + gamma) + alpha^2 L_1(x) (z(x) - 1)
 *     t(x)  = (arith + range + perm) / (x^N - 1)
 *   With no blinding deg t <= 4N - 5 on an honest composer.  dst: t_1 = t[0 .. N), t_2 = t[N .. 2N), t_3, t_4 (split_tx_poly), 4 x N
 *   coefficients column-major.  The call does not judge the witness: on a composer that violates a gate or a copy constraint it
 *   returns PG_OK and a t whose top coefficients are not zero (a verifier rejects it), like the reference's prover.
 * All three: PG_ERR_ARG when 2^log_n < the circuit size or a null buffer; PG_ERR_STATE on a ctx whose communicator has more than one
 *   rank.  pg_quotient also: PG_ERR_ARG when log_n > 30 (the 4N coset needs 2-adicity log_n + 2 <= 32), an unreduced challenge, or a
 *   zero z denominator (from the z computation it makes; pg_last_error names the row).  They synchronise the ctx stream. */
int pg_selector_polynomials(pg_ctx *ctx, uint32_t log_n, int form, pg_fr *dst, int dst_on_device);
int pg_public_input_polynomial(pg_ctx *ctx, uint32_t log_n, int form, pg_fr *dst, int dst_on_device);
int pg_quotient(pg_ctx *ctx, uint32_t log_n, const pg_fr *alpha, const pg_fr *beta, const pg_fr *gamma, const pg_fr *range_challenge,
                pg_fr *dst, int dst_on_device);

/* ---- openings: prover rounds 4 and 5 (SURVEY.md section 8f item 2, continued) ---------------------------------------------------
 * [DEP dusk-plonk 0.8 Prover::prove (the evaluations, compute_quotient_opening_poly / compute_aggregate_witness), linearisation_poly::
 * compute, the widgets' compute_linearisation and Polynomial::ruffini, recalled like the rest of [DEP]: parity unpinned.]
 * H, N, the padding, alpha, beta, gamma, rho, kappa = rho^2, Delta and k = (1, 7, 13, 17) are those of pg_quotient; w generates H.
 * challenges: 7 host scalars alpha beta gamma rho zeta v v' (zeta: the evaluation challenge; v, v': the aggregation challenges of the
 * openings at zeta and at zeta*w; the transcript is not built).  t: pg_quotient's 4 x N output for the same alpha, beta, gamma, rho.
 * Z_H(zeta) = zeta^N - 1, L_1(zeta) = Z_H(zeta) / (N (zeta - 1)).
 * Evaluations (pg_proof_evaluations, ProofEvaluations' order, then quot_eval):
 *   a b c d = w_l w_r w_o w_4 at zeta;  a_w b_w d_w = w_l w_r w_4 at zeta*w;  q_arith q_c q_l q_r at zeta;  sigma_1..3 at zeta;
 *   lin = r(zeta);  perm = z(zeta*w);  quot = t_1(zeta) + zeta^N t_2(zeta) + zeta^2N t_3(zeta) + zeta^3N t_4(zeta).
 * Linearisation polynomial (PI is not in r; the verifier adds PI(zeta)):
 *   r(X) = q_arith (a b q_m + a q_l + b q_r + c q_o + d q_4 + q_c)
 *        + rho (Delta(c - 4d) + kappa Delta(b - 4c) + kappa^2 Delta(a - 4b) + kappa^3 Delta(d_w - 4a)) q_range
 *        + (alpha prod_w (v_w + beta k_w zeta + gamma) + alpha^2 L_1(zeta)) z
 *        - alpha beta perm (a + beta sigma_1 + gamma)(b + beta sigma_2 + gamma)(c + beta sigma_3 + gamma) sigma_4
 *   with the scalars above (v_w = a b c d), the polynomials q_*, z, sigma_4 of X.
 * Opening witnesses, ruffini(f, p) = the quotient of f by (X - p) without the remainder (q_(N-2) = f_(N-1), q_(i-1) = f_i + p q_i),
 * N coefficients with q_(N-1) = 0:
 *   W_zeta   = ruffini(t_1 + zeta^N t_2 + zeta^2N t_3 + zeta^3N t_4 + v r + v^2 w_l + v^3 w_r + v^4 w_o + v^5 w_4
 *                      + v^6 sigma_1 + v^7 sigma_2 + v^8 sigma_3, zeta)
 *   W_zeta_w = ruffini(z + v' w_l + v'^2 w_r + v'^3 w_4, zeta*w)
 * The quotient identity.  By pg_quotient's definition, on an honest composer t(X) Z_H(X) = arith + range + perm as polynomials, so at
 * zeta: quot * Z_H(zeta) = arith(zeta) + range(zeta) + perm(zeta).  Substituting the evaluations, arith(zeta) + range(zeta) is r's first
 * two lines plus PI(zeta); perm(zeta) = alpha z(zeta) prod_w (v_w + beta k_w zeta + gamma) - alpha perm prod_(w<4) (v_w + beta sigma_w + gamma)
 * + alpha^2 L_1(zeta) (z(zeta) - 1), where r's third line is the terms with z(zeta) and the last factor (d + beta sigma_4 + gamma) splits
 * into r's fourth line and -alpha perm (...)(...)(...)(d + gamma).  Hence
 *   quot * Z_H(zeta) = lin + PI(zeta) - alpha^2 L_1(zeta) - alpha perm (a + beta sigma_1 + gamma)(b + beta sigma_2 + gamma)(c + beta sigma_3 + gamma)(d + gamma),
 * which is what the verifier's compute_quotient_evaluation checks.  On a composer that violates a constraint it fails (t is then not
 * the exact quotient), as the verifier would see.
 * pg_prover_openings: evals (host) and dst = [W_zeta, W_zeta_w, r], 3 x N coefficients column-major.  It rebuilds the wire, z, sigma and
 * selector coefficient vectors (as pg_quotient does) and takes t as input.  The remainder of each division is the aggregate's value at
 * its point; the call compares it with the same sum formed from the evaluations and reports a mismatch as PG_ERR_CUDA.  It does not
 * judge the witness.  PG_ERR_ARG: 2^log_n < the circuit size or log_n > 30, a null buffer, an unreduced challenge, an unreduced
 * coefficient of t (counted on the device; pg_last_error names the first, as index r*N + m), zeta^N = 1 (zeta in H: the reference's
 * L_1 inversion panics at zeta = 1 and the verifier divides by Z_H(zeta)), or a zero z denominator (pg_last_error names the row).
 * PG_ERR_STATE on a ctx whose communicator has more than one rank.  It synchronises the ctx stream. */
typedef struct pg_proof_evaluations {
    pg_fr a_eval, b_eval, c_eval, d_eval, a_next_eval, b_next_eval, d_next_eval, q_arith_eval, q_c_eval, q_l_eval, q_r_eval,
          left_sigma_eval, right_sigma_eval, out_sigma_eval, lin_poly_eval, perm_eval, quot_eval;
} pg_proof_evaluations;
int pg_prover_openings(pg_ctx *ctx, uint32_t log_n, const pg_fr *challenges, const pg_fr *t, int t_on_device, pg_proof_evaluations *evals,
                       pg_fr *dst, int dst_on_device);

/* ---- commitments (SURVEY.md section 8f item 2, second half) -----------------------------------------------------------------
 * KZG commitments of coefficient vectors in the BLS12-381 group G1 [DEP dusk-plonk 0.8 CommitKey::commit =
 * dusk-bls12_381 msm_variable_base(&powers_of_g, &poly.coeffs); Prover::prove computes w_l_poly_commit .. w_4_poly_commit right
 * after the wire polynomials; reached from ref:tests/range_gadgets_tests.rs:90-91].
 * pg_g1_affine = the in-memory G1Affine { x: Fp, y: Fp } of dusk-bls12_381 (Fp([u64; 6]), Montgomery form, R = 2^384) without
 * its `infinity` flag byte: the point at infinity is the all-zero pair.
 * pg_msm: out = sum_i scalars[i] * points[i] (one point, written to HOST memory); points/scalars both host or both device.
 * pg_srs_powers: out[i] = beta^i * base, base == NULL meaning the G1 generator (PublicParameters::setup: powers_of_g).
 * pg_g1_fixed_base_mul: out[i] = scalars[i] * base.  base and beta are host pointers to one element.
 * pg_commit_wire_polynomials: the four commitments of the composer's wire polynomials over the domain 2^log_n against
 * powers_of_g[0 .. 2^log_n), written to host memory (w_l, w_r, w_o, w_4); PG_ERR_ARG when n_powers < 2^log_n (the reference's
 * check_commit_degree_is_within_bounds / Error::PolynomialDegreeTooLarge).  The reference blinds nothing in this version.
 * Points are taken as given: no on-curve / subgroup check (the reference validates when it deserialises; use pg_g1_op(1, ..)). */
typedef struct pg_g1_affine { uint64_t x[6]; uint64_t y[6]; } pg_g1_affine;
int pg_msm(pg_ctx *ctx, uint64_t n, const pg_g1_affine *points, const pg_fr *scalars, pg_g1_affine *out, int on_device);
int pg_srs_powers(pg_ctx *ctx, const pg_fr *beta, const pg_g1_affine *base, uint64_t n, pg_g1_affine *out, int out_on_device);
int pg_g1_fixed_base_mul(pg_ctx *ctx, uint64_t n, const pg_g1_affine *base, const pg_fr *scalars, pg_g1_affine *out, int on_device);
int pg_commit_wire_polynomials(pg_ctx *ctx, uint32_t log_n, const pg_g1_affine *powers_of_g, uint64_t n_powers, int powers_on_device,
                               pg_g1_affine *out4);
/* Evaluation-form commitments.  With the Lagrange-basis form of the SRS for a domain, lagrange[i] = L_i(beta) * base, the
 * commitment of a polynomial is sum_i f(w^i) * lagrange[i] -- the same group element as sum_j coeff_j * powers_of_g[j] -- so the
 * wire commitments can be taken from the wire VALUES directly: no FFT, and bits / short accumulators leave most windows empty.
 * pg_srs_lagrange builds that form for local setups that know beta (like PublicParameters::setup; PG_ERR_ARG if beta lies on the
 * domain).  pg_srs_lagrange_from_powers derives it from the monomial powers alone, for a trusted setup whose beta nobody knows.
 * pg_commit_wire_evaluations returns the same four points as pg_commit_wire_polynomials; n_points must be exactly 2^log_n. */
int pg_srs_lagrange(pg_ctx *ctx, const pg_fr *beta, const pg_g1_affine *base, uint32_t log_n, pg_g1_affine *out, int out_on_device);
/* pg_srs_lagrange_from_powers: out[i] = (1/n) sum_{j<n} w^(-ij) * powers_of_g[j], i < n = 2^log_n, w the domain generator of pg_fft
 * (EvaluationDomain::group_gen).  Only the first n powers are read (like the trimmed CommitKey).  When powers_of_g[j] = beta^j * base
 * the result is pg_srs_lagrange(beta, base, log_n) bit for bit (canonical affine limbs, infinity all-zero).  log_n = 0 copies
 * powers_of_g[0].  The work is an inverse FFT over G1 with a 255-bit scalar multiplication per butterfly (about
 * (n/2) log n + n of them); it needs n x 192 bytes of device scratch.  Points are taken as given (no on-curve check, like pg_msm).
 * It uses no composer state, so a sharded ctx may call it.  PG_ERR_ARG: a null pointer, log_n > 32, n_powers < 2^log_n.
 * It synchronises the ctx stream. */
int pg_srs_lagrange_from_powers(pg_ctx *ctx, uint32_t log_n, const pg_g1_affine *powers_of_g, uint64_t n_powers, int powers_on_device,
                                pg_g1_affine *out, int out_on_device);
int pg_commit_wire_evaluations(pg_ctx *ctx, uint32_t log_n, const pg_g1_affine *lagrange, uint64_t n_points, int points_on_device,
                               pg_g1_affine *out4);
/* self-test helper: op 0: out[i] = a[i] + b[i]; op 1: out[i].x[0] = 1 if a[i] is on the curve (or infinity) else 0.  Host buffers. */
int pg_g1_op(pg_ctx *ctx, int op, uint64_t n, const pg_g1_affine *a, const pg_g1_affine *b, pg_g1_affine *out);

/* ---- wire format (SURVEY.md section 8f item 3) -------------------------------------------------------------------------
 * BlsScalar::to_bytes / from_bytes [dusk_bytes::Serializable<32>, called at ref:src/range.rs:163]: the canonical
 * little-endian 32-byte encoding used for witness / selector / public-input dumps exchanged with Rust tooling.  n scalars;
 * src and dst are both host (on_device == 0; dst may be unaligned-safe only for host) or both device pointers.
 * from_bytes rejects encodings >= q like the reference: they are counted in *n_invalid (first index in *first_invalid, or
 * UINT64_MAX) and decode to 0. */
int pg_fr_to_bytes(pg_ctx *ctx, uint64_t n, const pg_fr *src, uint8_t *dst, int on_device);
int pg_fr_from_bytes(pg_ctx *ctx, uint64_t n, const uint8_t *src, pg_fr *dst, int on_device, uint64_t *n_invalid,
                     uint64_t *first_invalid);

/* ---- fault injection ----------------------------------------------------------------------------------------------------------
 * Overwrites composer.variables[var] with *value (host pointer), leaving every row as it is: the way to present pg_check with a
 * witness that violates a constraint (the gadgets themselves only ever produce consistent ones).  Variables stored as packed
 * bits (the 256 bit variables of a decomposition) cannot be overwritten: PG_ERR_ARG. */
int pg_poke_variable(pg_ctx *ctx, uint64_t var, const pg_fr *value);

/* ---- measurement helpers ------------------------------------------------------------------------------------------- */
/* Deterministic synthetic scalars (SplitMix64 counter stream): kind 0 = uniform Fr (512-bit draw reduced mod q, as
 * BlsScalar::from_bytes_wide), kind 1 = uniform integer of `bits` bits (bits <= 254), kind 2 = even index kind 1 / odd
 * index kind 0, kind 3 = `bits`-bit integer with the top bit forced to 1.  dst is a device pointer (n scalars). */
int pg_synth(pg_ctx *ctx, uint64_t seed, uint64_t stream, uint64_t n, int kind, uint32_t bits, pg_fr *dst_device);

typedef struct pg_timing {
    double check_ms;        /* gate-check kernels */
    double witness_ms;      /* witness-generation kernels (incl. batch inversion) */
    double other_ms;        /* layout / materialise / synth kernels */
    uint64_t check_launches, witness_launches, other_launches;
    uint64_t check_rows;    /* rows evaluated by the gate-check kernels */
} pg_timing;
int pg_get_timing(pg_ctx *ctx, pg_timing *out, int reset);   /* needs PG_F_TIMING; synchronises */

/* Which kernel evaluated how many rows since the last reset (counted at launch, no synchronisation).  Kinds:
 * one thread per instance -- generic equation (k_check), per-row structure-aware terms, compiled structure-aware row program
 * (k_check_prog); one thread per (instance, row) for segments too small to fill the chip (k_check_rowpar); segments with
 * range-widget rows (k_check_gates); rows evaluated inside witness generation (PG_F_FUSED_CHECK). */
enum { PG_CK_INSTANCE_GENERIC = 0, PG_CK_INSTANCE_TERMS = 1, PG_CK_PROGRAM = 2, PG_CK_ROWPAR = 3, PG_CK_GATES = 4, PG_CK_FUSED = 5, PG_CK_KINDS = 8 };
typedef struct pg_check_stats { uint64_t launches[PG_CK_KINDS]; uint64_t rows[PG_CK_KINDS]; } pg_check_stats;
int pg_get_check_stats(pg_ctx *ctx, pg_check_stats *out, int reset);

/* Integer-multiply roofline denominators measured on this GPU: 32x32+64->64 multiply-accumulates per second with
 * IMAD.WIDE.U32 chains, and 32-bit IMAD (lo) per second. */
int pg_measure_imad_peak(pg_ctx *ctx, double *wide_mac_per_s, double *imad_per_s);
/* Pipe micro-benchmarks (operations per second on all SMs): mode 0 IMAD lo, 1 IMAD.WIDE product only, 2 IMAD.WIDE with
 * 64-bit accumulate, 3 IMAD.HI, 4 the mad.lo.cc/madc.hi.cc carry-chain rows of the Fr multiplier (per 32x32 product),
 * 5 IADD3, 6 Fr Montgomery multiplications (device multiplier), 7 the same through the portable CIOS code, 8 Fr additions,
 * 9 fp64 DFMA, 10 IMAD.WIDE and DFMA interleaved 1:1 (both counted). */
int pg_microbench(pg_ctx *ctx, int mode, double *ops_per_s);

/* Element-wise Fr self-test kernels (op: 0 mul, 1 add, 2 sub, 3 neg, 4 invert-or-zero (batch inversion), 5 from_mont,
 * 6 mul via the portable CIOS path, 7 exclusive prefix product out[0] = 1, out[i] = a[0]*..*a[i-1] (the grand-product scan of
 * pg_permutation_z), 8 division by (X - b[0]): out[0 .. n-1) = ruffini(a, b[0]) and out[n-1] = the remainder a(b[0]) (the Ruffini scan of
 * pg_prover_openings; b holds one scalar)).  a, b, out: host arrays of n scalars. */
int pg_fr_op(pg_ctx *ctx, int op, uint64_t n, const pg_fr *a, const pg_fr *b, pg_fr *out);

#ifdef __cplusplus
}
#endif
#endif /* PG_B200_H */
