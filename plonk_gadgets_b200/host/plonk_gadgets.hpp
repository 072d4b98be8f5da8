// plonk_gadgets.hpp -- C++17 host-side mirror of the reference crate's public interface, over the C ABI (include/pg_b200.h).
//
// The reference is a Rust library; there is no Rust toolchain in this environment, so the host layer above the C ABI is
// written in C++ (the Rust `-sys`/wrapper crates are shipped as source under bindings/rust, see INTEGRATION.md).
// Names, argument order and error behaviour follow /root/reference/src/lib.rs:37-45:
//
//   plonk_gadgets::AllocatedScalar::allocate        /root/reference/src/allocated_scalar.rs:27-30
//   plonk_gadgets::RangeGadgets::range_check        /root/reference/src/range.rs:27-43
//   plonk_gadgets::RangeGadgets::max_bound          /root/reference/src/range.rs:82-113
//   plonk_gadgets::ScalarGadgets::{conditionally_select_zero, conditionally_select_one, is_non_zero, maybe_equal}
//                                                   /root/reference/src/scalar.rs:21-140
//   plonk_gadgets::Error::NonExistingInverse        /root/reference/src/errors.rs:13-18
//
// Every gadget takes `StandardComposer&` first, like the reference takes `&mut StandardComposer`; operands are columns of
// n variables (one gadget instance per element) instead of single `Variable`s.  Header-only; link with libpg_b200.so.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>
#include "../../include/pg_b200.h"
#include "../csrc/fr.cuh"      // host-side Fr (portable Montgomery arithmetic) for BlsScalar construction only

namespace plonk_gadgets {

// dusk_plonk::bls12_381::BlsScalar: Montgomery limbs.  Only what callers of the gadgets need to build inputs.
struct BlsScalar {
    pg_fr raw;
    static BlsScalar from_fr(const pg::Fr& f) {
        BlsScalar s;
        for (int i = 0; i < 4; i++) s.raw.l[i] = (uint64_t)f.v[2 * i] | ((uint64_t)f.v[2 * i + 1] << 32);
        return s;
    }
    pg::Fr fr() const {
        pg::Fr f;
        for (int i = 0; i < 4; i++) { f.v[2 * i] = (uint32_t)raw.l[i]; f.v[2 * i + 1] = (uint32_t)(raw.l[i] >> 32); }
        return f;
    }
    static BlsScalar zero() { return from_fr(pg::fr_zero()); }
    static BlsScalar one() { return from_fr(pg::fr_one()); }
    static BlsScalar from(uint64_t v) { pg::Fr r = {{(uint32_t)v, (uint32_t)(v >> 32), 0, 0, 0, 0, 0, 0}}; return from_fr(pg::fr_to_mont(r)); }
    static BlsScalar pow_of_2(uint64_t by) { pg::Fr r = pg::fr_one(); for (uint64_t i = 0; i < by; i++) r = pg::fr_add(r, r); return from_fr(r); }
    BlsScalar operator+(const BlsScalar& o) const { return from_fr(pg::fr_add(fr(), o.fr())); }
    BlsScalar operator-(const BlsScalar& o) const { return from_fr(pg::fr_sub(fr(), o.fr())); }
    BlsScalar operator*(const BlsScalar& o) const { return from_fr(pg::fr_mul(fr(), o.fr())); }
    BlsScalar operator-() const { return from_fr(pg::fr_neg(fr())); }
    bool operator==(const BlsScalar& o) const { return pg::fr_eq(fr(), o.fr()); }
};
static_assert(sizeof(BlsScalar) == 32, "BlsScalar must be layout-compatible with pg_fr");

/// /root/reference/src/errors.rs:13-18
enum class Error { NonExistingInverse };

/// Engine failures (negative codes of the C ABI): never mapped onto a gadget error, never a silent fallback.
struct EngineError : std::runtime_error {
    int code;
    EngineError(int c, const std::string& what) : std::runtime_error(what), code(c) {}
};

class StandardComposer;

/// n `Variable`s, one per gadget instance.
struct Variables {
    pg_col col = 0;
    uint64_t n = 0;
};

/// Device-resident batched StandardComposer (fresh: 3 rows, 5 variables).
class StandardComposer {
public:
    explicit StandardComposer(int device = 0, int check_mode = PG_CHECK_GENERIC, bool fused_check = false) {
        pg_cfg cfg{}; cfg.device = device; cfg.check_mode = check_mode; cfg.flags = fused_check ? PG_F_FUSED_CHECK : 0u;
        int rc = pg_ctx_create(&cfg, &ctx_);
        if (rc != PG_OK) throw EngineError(rc, std::string("pg_ctx_create: ") + pg_strerror(rc));
    }
    ~StandardComposer() { pg_ctx_destroy(ctx_); }
    StandardComposer(const StandardComposer&) = delete;
    StandardComposer& operator=(const StandardComposer&) = delete;

    pg_ctx* raw() { return ctx_; }
    int ok(int rc, const char* what) {
        if (rc < 0) throw EngineError(rc, std::string(what) + ": " + pg_last_error(ctx_));
        return rc;
    }
    /// composer.add_input over n scalars
    Variables add_input(const std::vector<BlsScalar>& scalars) {
        Variables v; v.n = scalars.size();
        ok(pg_add_input_batch(ctx_, v.n, reinterpret_cast<const pg_fr*>(scalars.data()), 0, &v.col), "pg_add_input_batch");
        return v;
    }
    /// composer.range_gate(witness, num_bits) per instance [dusk-plonk; recommended at /root/reference/src/range.rs:9-12]
    void range_gate(Variables witness, size_t num_bits) { ok(pg_range_gate_batch(ctx_, witness.col, (uint32_t)num_bits), "pg_range_gate_batch"); }
    /// composer.constrain_to_constant(a, constant, pi) per instance; `pi` empty = None
    void constrain_to_constant(Variables a, const std::vector<BlsScalar>& constant, const std::vector<BlsScalar>& pi = {}) {
        ok(pg_constrain_to_constant_batch(ctx_, a.col, reinterpret_cast<const pg_fr*>(constant.data()), constant.size(),
                                          pi.empty() ? nullptr : reinterpret_cast<const pg_fr*>(pi.data()), pi.size(), 0),
           "pg_constrain_to_constant_batch");
    }
    uint64_t circuit_size() const { uint64_t r = 0, v = 0; pg_counts(ctx_, &r, &v); return r; }
    uint64_t num_variables() const { uint64_t r = 0, v = 0; pg_counts(ctx_, &r, &v); return v; }
    /// arithmetic part of check_circuit_satisfied: (unsatisfied rows, first unsatisfied row or UINT64_MAX)
    std::pair<uint64_t, uint64_t> check_circuit_satisfied() {
        uint64_t bad = 0, first = 0;
        ok(pg_check(ctx_, &bad, &first), "pg_check");
        return {bad, first};
    }
    std::vector<BlsScalar> values(Variables v) {
        std::vector<BlsScalar> out(v.n);
        ok(pg_col_read(ctx_, v.col, 0, v.n, reinterpret_cast<pg_fr*>(out.data()), 0), "pg_col_read");
        return out;
    }
    void reset() { ok(pg_composer_reset(ctx_), "pg_composer_reset"); }
    /// composer.variables[var0 .. var0 + cnt) in Variable order
    std::vector<BlsScalar> variables(uint64_t var0, uint64_t cnt) {
        std::vector<BlsScalar> out(cnt);
        ok(pg_read_variables(ctx_, var0, cnt, reinterpret_cast<pg_fr*>(out.data()), 0), "pg_read_variables");
        return out;
    }
    /// The hand-over to a real dusk-plonk StandardComposer (prover.mut_cs(), /root/reference/tests/range_gadgets_tests.rs:82-91):
    /// the whole composer in one file, replayed by bindings/rust/plonk-gadgets-b200/src/import.rs
    void export_to(const std::string& path, bool with_sigma = false) { ok(pg_export_composer(ctx_, path.c_str(), 0, with_sigma ? PG_EXPORT_SIGMA : 0u), "pg_export_composer"); }

    // ---- several GPUs: one process and one composer per GPU (include/pg_b200.h, "multi-GPU") ----
    void comm_init(const uint8_t* unique_id, uint32_t rank, uint32_t world) { ok(pg_comm_init(ctx_, unique_id, rank, world), "pg_comm_init"); }
    struct Verdict { uint64_t n_unsat, first_bad_row, n_err; };
    /// verdict of the WHOLE sharded circuit on every rank; `mine`: this rank's row of shard_plan(..) (empty: local numbering)
    Verdict check_sharded(const std::vector<pg_op_shard>& mine, uint64_t n_err_local = 0) {
        Verdict v{0, 0, n_err_local};
        ok(pg_check_sharded(ctx_, mine.empty() ? nullptr : mine.data(), mine.size(), &v.n_unsat, &v.first_bad_row, &v.n_err), "pg_check_sharded");
        return v;
    }
    /// the per-instance results of a call from every rank, in instance order of the whole batch (`total` = sum of the ranks' lengths)
    std::vector<BlsScalar> gather_column(Variables v, uint64_t total) {
        std::vector<BlsScalar> out(total); uint64_t got = 0;
        ok(pg_gather_column(ctx_, v.col, reinterpret_cast<pg_fr*>(out.data()), total, 0, nullptr, &got), "pg_gather_column");
        out.resize(got);
        return out;
    }
    /// gather of witness shards: the Variables of call number `call` from every rank, in the sequential composer's order
    std::vector<BlsScalar> gather_variables(uint64_t call, uint64_t total) {
        std::vector<BlsScalar> out(total); uint64_t got = 0;
        ok(pg_gather_variables(ctx_, call, reinterpret_cast<pg_fr*>(out.data()), total, 0, &got), "pg_gather_variables");
        out.resize(got);
        return out;
    }

    // ---- the prover's first round ([DEP] dusk-plonk 0.8 Prover::prove: to_scalars + pad, domain.ifft, commit_key.commit) ----
    /// log2 of EvaluationDomain::new(circuit_size).size()
    uint32_t domain_log_size() const { uint32_t l = 0; while ((1ull << l) < circuit_size()) l++; return l; }
    /// coefficients of w_l, w_r, w_o, w_4: 4 x 2^log_n scalars, column after column
    std::vector<BlsScalar> wire_polynomials(uint32_t log_n) {
        std::vector<BlsScalar> out((size_t)4 << log_n);
        ok(pg_wire_polynomials(ctx_, log_n, reinterpret_cast<pg_fr*>(out.data()), 0), "pg_wire_polynomials");
        return out;
    }
    /// preprocessing's sigma polynomials over the domain 2^log_n (evaluations, or coefficients): 4 x 2^log_n scalars
    std::vector<BlsScalar> sigma_polynomials(uint32_t log_n, bool coefficients = false) {
        std::vector<BlsScalar> out((size_t)4 << log_n);
        ok(pg_sigma_polynomials(ctx_, log_n, coefficients ? PG_FORM_COEFFICIENTS : PG_FORM_EVALUATIONS, reinterpret_cast<pg_fr*>(out.data()), 0),
           "pg_sigma_polynomials");
        return out;
    }
    /// prover round 2: z over the domain 2^log_n for the caller's beta, gamma; *closing = product of all ratios (may be null)
    std::vector<BlsScalar> permutation_z(uint32_t log_n, const BlsScalar& beta, const BlsScalar& gamma, bool coefficients = false,
                                         BlsScalar* closing = nullptr) {
        std::vector<BlsScalar> out((size_t)1 << log_n);
        ok(pg_permutation_z(ctx_, log_n, reinterpret_cast<const pg_fr*>(&beta), reinterpret_cast<const pg_fr*>(&gamma),
                            coefficients ? PG_FORM_COEFFICIENTS : PG_FORM_EVALUATIONS, reinterpret_cast<pg_fr*>(out.data()), 0,
                            reinterpret_cast<pg_fr*>(closing)), "pg_permutation_z");
        return out;
    }
    /// preprocessing's q_m q_l q_r q_o q_4 q_c q_arith q_range over the domain 2^log_n (evaluations, or coefficients): 8 x 2^log_n scalars
    std::vector<BlsScalar> selector_polynomials(uint32_t log_n, bool coefficients = false) {
        std::vector<BlsScalar> out((size_t)8 << log_n);
        ok(pg_selector_polynomials(ctx_, log_n, coefficients ? PG_FORM_COEFFICIENTS : PG_FORM_EVALUATIONS, reinterpret_cast<pg_fr*>(out.data()), 0),
           "pg_selector_polynomials");
        return out;
    }
    /// the dense public inputs padded to 2^log_n (evaluations), or PI(X) (coefficients)
    std::vector<BlsScalar> public_input_polynomial(uint32_t log_n, bool coefficients = false) {
        std::vector<BlsScalar> out((size_t)1 << log_n);
        ok(pg_public_input_polynomial(ctx_, log_n, coefficients ? PG_FORM_COEFFICIENTS : PG_FORM_EVALUATIONS, reinterpret_cast<pg_fr*>(out.data()), 0),
           "pg_public_input_polynomial");
        return out;
    }
    /// prover round 3: t_1 .. t_4, 4 x 2^log_n coefficients, for the caller's alpha, beta, gamma and range separation challenge
    std::vector<BlsScalar> quotient(uint32_t log_n, const BlsScalar& alpha, const BlsScalar& beta, const BlsScalar& gamma, const BlsScalar& range_challenge) {
        std::vector<BlsScalar> out((size_t)4 << log_n);
        auto p = [](const BlsScalar& x) { return reinterpret_cast<const pg_fr*>(&x); };
        ok(pg_quotient(ctx_, log_n, p(alpha), p(beta), p(gamma), p(range_challenge), reinterpret_cast<pg_fr*>(out.data()), 0), "pg_quotient");
        return out;
    }
    /// prover rounds 4 and 5 for pg_quotient's t (4 x 2^log_n) and the challenges alpha beta gamma rho zeta v v': the 17 evaluations
    /// (ProofEvaluations' order, then quot_eval) and [W_zeta, W_zeta_w, r], 3 x 2^log_n coefficients
    std::pair<pg_proof_evaluations, std::vector<BlsScalar>> prover_openings(uint32_t log_n, const std::vector<BlsScalar>& t, const BlsScalar (&challenges)[7]) {
        if (t.size() != ((size_t)4 << log_n)) throw std::invalid_argument("prover_openings: t must hold 4 x 2^log_n scalars");
        pg_proof_evaluations ev;
        std::vector<BlsScalar> out((size_t)3 << log_n);
        ok(pg_prover_openings(ctx_, log_n, reinterpret_cast<const pg_fr*>(challenges), reinterpret_cast<const pg_fr*>(t.data()), 0, &ev,
                              reinterpret_cast<pg_fr*>(out.data()), 0), "pg_prover_openings");
        return {ev, out};
    }
    /// EvaluationDomain::fft / ifft of 2^k scalars
    std::vector<BlsScalar> fft(const std::vector<BlsScalar>& v, bool inverse) {
        uint32_t log_n = 0; while ((1ull << log_n) < v.size()) log_n++;
        if (v.empty() || (1ull << log_n) != v.size()) throw EngineError(PG_ERR_ARG, "fft: the length must be a power of two");
        std::vector<BlsScalar> out(v.size());
        ok(pg_fft(ctx_, log_n, inverse ? 1 : 0, reinterpret_cast<const pg_fr*>(v.data()), reinterpret_cast<pg_fr*>(out.data()), 0), "pg_fft");
        return out;
    }
    /// PublicParameters::setup: powers_of_g[i] = beta^i * G1 generator
    std::vector<pg_g1_affine> srs_powers(const BlsScalar& beta, uint64_t n) {
        std::vector<pg_g1_affine> out(n);
        ok(pg_srs_powers(ctx_, reinterpret_cast<const pg_fr*>(&beta), nullptr, n, out.data(), 0), "pg_srs_powers");
        return out;
    }
    /// Lagrange-basis form of the SRS for the domain 2^log_n: out[i] = L_i(beta) * G1 generator
    std::vector<pg_g1_affine> srs_lagrange(const BlsScalar& beta, uint32_t log_n) {
        std::vector<pg_g1_affine> out((size_t)1 << log_n);
        ok(pg_srs_lagrange(ctx_, reinterpret_cast<const pg_fr*>(&beta), nullptr, log_n, out.data(), 0), "pg_srs_lagrange");
        return out;
    }
    /// the same form from the monomial powers alone (a trusted setup's powers_of_g, beta unknown): the first 2^log_n powers are read
    std::vector<pg_g1_affine> srs_lagrange_from_powers(const std::vector<pg_g1_affine>& powers_of_g, uint32_t log_n) {
        std::vector<pg_g1_affine> out((size_t)1 << log_n);
        ok(pg_srs_lagrange_from_powers(ctx_, log_n, powers_of_g.data(), powers_of_g.size(), 0, out.data(), 0), "pg_srs_lagrange_from_powers");
        return out;
    }
    /// the same four commitments as commit_wire_polynomials, from the wire values against the Lagrange-basis SRS (no FFT)
    std::vector<pg_g1_affine> commit_wire_evaluations(const std::vector<pg_g1_affine>& lagrange, uint32_t log_n) {
        std::vector<pg_g1_affine> out(4);
        ok(pg_commit_wire_evaluations(ctx_, log_n, lagrange.data(), lagrange.size(), 0, out.data()), "pg_commit_wire_evaluations");
        return out;
    }
    /// CommitKey::commit of a coefficient vector (msm_variable_base)
    pg_g1_affine commit(const std::vector<pg_g1_affine>& powers_of_g, const std::vector<BlsScalar>& coeffs) {
        if (coeffs.size() > powers_of_g.size()) throw EngineError(PG_ERR_ARG, "commit: polynomial degree exceeds the SRS");
        pg_g1_affine out{};
        ok(pg_msm(ctx_, coeffs.size(), powers_of_g.data(), reinterpret_cast<const pg_fr*>(coeffs.data()), &out, 0), "pg_msm");
        return out;
    }
    /// w_l_poly_commit .. w_4_poly_commit
    std::vector<pg_g1_affine> commit_wire_polynomials(const std::vector<pg_g1_affine>& powers_of_g, uint32_t log_n) {
        std::vector<pg_g1_affine> out(4);
        ok(pg_commit_wire_polynomials(ctx_, log_n, powers_of_g.data(), powers_of_g.size(), 0, out.data()), "pg_commit_wire_polynomials");
        return out;
    }

private:
    pg_ctx* ctx_ = nullptr;
};

/// /root/reference/src/allocated_scalar.rs:17-31
struct AllocatedScalar {
    Variables var;
    static AllocatedScalar allocate(StandardComposer& composer, const std::vector<BlsScalar>& scalar) {
        return AllocatedScalar{composer.add_input(scalar)};
    }
};

namespace RangeGadgets {
/// /root/reference/src/range.rs:27-43.  min_range/max_range: 1 (uniform) or n scalars of one bit width.
inline Variables range_check(StandardComposer& composer, const std::vector<BlsScalar>& min_range, const std::vector<BlsScalar>& max_range,
                             AllocatedScalar witness) {
    if (min_range.size() != max_range.size()) throw EngineError(PG_ERR_ARG, "range_check: min/max length mismatch");
    Variables out; out.n = witness.var.n;
    composer.ok(pg_range_check_batch(composer.raw(), reinterpret_cast<const pg_fr*>(min_range.data()),
                                     reinterpret_cast<const pg_fr*>(max_range.data()), max_range.size(), 0, witness.var.col, &out.col, nullptr),
                "pg_range_check_batch");
    return out;
}
/// /root/reference/src/range.rs:82-113 -> (Variable, num_bits)
inline std::pair<Variables, uint64_t> max_bound(StandardComposer& composer, const std::vector<BlsScalar>& max_range, AllocatedScalar witness) {
    Variables out; out.n = witness.var.n; uint64_t k = 0;
    composer.ok(pg_max_bound_batch(composer.raw(), reinterpret_cast<const pg_fr*>(max_range.data()), max_range.size(), 0, witness.var.col, &out.col, &k),
                "pg_max_bound_batch");
    return {out, k};
}
}  // namespace RangeGadgets

namespace ScalarGadgets {
/// /root/reference/src/scalar.rs:21-27
inline Variables conditionally_select_zero(StandardComposer& composer, Variables x, Variables select) {
    Variables out; out.n = x.n;
    composer.ok(pg_select_zero_batch(composer.raw(), x.col, select.col, &out.col), "pg_select_zero_batch");
    return out;
}
/// /root/reference/src/scalar.rs:36-59
inline Variables conditionally_select_one(StandardComposer& composer, Variables y, Variables selector) {
    Variables out; out.n = y.n;
    composer.ok(pg_select_one_batch(composer.raw(), y.col, selector.col, &out.col), "pg_select_one_batch");
    return out;
}
/// /root/reference/src/scalar.rs:63-97 -- Result<(), Error>: returns true on Ok(()), false + *err on Err (like `is_non_zero(..)?` in a loop)
inline bool is_non_zero(StandardComposer& composer, Variables var, const std::vector<BlsScalar>& value_assigned, Error* err = nullptr,
                        uint64_t* first_err = nullptr) {
    uint64_t n_err = 0, first = 0;
    int rc = composer.ok(pg_is_non_zero_batch(composer.raw(), var.col, reinterpret_cast<const pg_fr*>(value_assigned.data()), 0, &n_err, &first),
                         "pg_is_non_zero_batch");
    if (rc == PG_ERR_NON_EXISTING_INVERSE) { if (err) *err = Error::NonExistingInverse; if (first_err) *first_err = first; return false; }
    return true;
}
/// The same loop with every Result kept (a batch does not abort on one zero, /root/reference/src/errors.rs:13-18): errs[i] is true
/// where is_non_zero(composer, var_i, value_assigned_i) returned Err(NonExistingInverse).  reference_layout: errored calls leave the
/// 1 variable + 1 row of scalar.rs:69-71 behind, as the reference does; otherwise 3 + 3 everywhere (the errored instance fails its last row).
inline std::vector<bool> is_non_zero_each(StandardComposer& composer, Variables var, const std::vector<BlsScalar>& value_assigned, bool reference_layout = false) {
    std::vector<uint8_t> flags(value_assigned.size()); uint64_t n_err = 0;
    composer.ok(pg_is_non_zero_batch_flags(composer.raw(), var.col, reinterpret_cast<const pg_fr*>(value_assigned.data()), 0, flags.data(),
                                           reference_layout ? PG_NZ_REFERENCE : PG_NZ_UNIFORM, &n_err), "pg_is_non_zero_batch_flags");
    return std::vector<bool>(flags.begin(), flags.end());
}
/// /root/reference/src/scalar.rs:105-140
inline Variables maybe_equal(StandardComposer& composer, AllocatedScalar a, AllocatedScalar b) {
    Variables out; out.n = a.var.n;
    composer.ok(pg_maybe_equal_batch(composer.raw(), a.var.col, b.var.col, &out.col), "pg_maybe_equal_batch");
    return out;
}
}  // namespace ScalarGadgets

/// Cuts a mixed circuit (a list of batched calls) over `world` GPUs: plan[rank][k] = the instance range of call k that rank runs and
/// the row / Variable index of its first instance in the sequential composer (pure host code).
inline std::vector<std::vector<pg_op_shard>> shard_plan(const std::vector<pg_op>& ops, uint32_t world, bool by_rows = false) {
    std::vector<pg_op_shard> flat(ops.size() * world);
    const int rc = pg_shard_plan(ops.data(), ops.size(), world, by_rows ? PG_SHARD_ROWS : PG_SHARD_EVEN, flat.data());
    if (rc != PG_OK) throw EngineError(rc, std::string("pg_shard_plan: ") + pg_strerror(rc));
    std::vector<std::vector<pg_op_shard>> plan(world);
    for (uint32_t r = 0; r < world; r++) plan[r].assign(flat.begin() + (size_t)r * ops.size(), flat.begin() + (size_t)(r + 1) * ops.size());
    return plan;
}

}  // namespace plonk_gadgets
