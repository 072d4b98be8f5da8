// reference_tests.cpp -- the reference crate's integration tests, replayed through the C++ mirror on the GPU.
//
// Mirrors /root/reference/tests/range_gadgets_tests.rs (max_bound_test :46-107, range_check_test :108-201) and
// /root/reference/tests/scalar_gadgets_tests.rs (test_maybe_equal :13-68, test_conditionally_select_0 :70-122,
// test_conditionally_select_1 :124-178, test_is_not_zero :180-236).  The reference decides each case with a
// prove -> verify round trip (out of scope here, SURVEY.md section 2 row 8); the verdict of this engine is "every row
// satisfies the gate equation", which is equivalent for these circuits (copy constraints hold by construction).
// All cases of one test are batched into ONE gadget call (one instance per case).  Exit code 0 = all verdicts as expected.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <unistd.h>
#include "plonk_gadgets.hpp"

using namespace plonk_gadgets;
using RangeGadgets::max_bound;
using RangeGadgets::range_check;
using namespace ScalarGadgets;

static int failures = 0;
#define EXPECT(cond, msg) do { if (!(cond)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, msg); failures++; } } while (0)

static BlsScalar two_pow(uint64_t e) { return BlsScalar::pow_of_2(e); }     // BlsScalar::from(2).pow(&[e,0,0,0])

// constrain every instance's output to the claimed boolean and return the verdict (tests/range_gadgets_tests.rs:22-26)
static bool satisfied_with_claims(StandardComposer& c, Variables res, const std::vector<bool>& claims) {
    std::vector<BlsScalar> outcome;
    for (bool b : claims) outcome.push_back(b ? BlsScalar::one() : BlsScalar::zero());
    c.constrain_to_constant(res, outcome);
    return c.check_circuit_satisfied().first == 0;
}

static void max_bound_test() {
    struct TestCase { BlsScalar max_range, witness; bool expected_result; };
    std::vector<TestCase> cases = {
        {two_pow(128) - BlsScalar::one(), two_pow(127), true},
        {BlsScalar::from(200), BlsScalar::from(100), true},
        {BlsScalar::from(100), BlsScalar::from(200), false},
        {two_pow(128) - BlsScalar::one(), two_pow(130), false},
    };
    // bounds of different bit widths cannot share one batched call: one call per case (n = 1), as in the reference's loop
    for (auto& tc : cases) {
        for (bool flip : {false, true}) {
            StandardComposer composer;
            auto witness = AllocatedScalar::allocate(composer, {tc.witness});
            auto res = max_bound(composer, {tc.max_range}, witness).first;
            bool ok = satisfied_with_claims(composer, res, {tc.expected_result != flip});
            EXPECT(ok == !flip, "max_bound verdict");
        }
    }
}

static void range_check_test() {
    struct TestCase { BlsScalar min_range, max_range, witness; bool expected_result; };
    std::vector<TestCase> cases = {
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(50001), true},
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(250001), false},
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(250000), false},
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(249000), true},
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(50000), true},
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(49999), false},
        {BlsScalar::from(50000), BlsScalar::from(250000), BlsScalar::from(18598), false},
    };
    // the seven cases with the same public bounds run as ONE batched call
    StandardComposer composer;
    std::vector<BlsScalar> w; std::vector<bool> claims;
    for (auto& tc : cases) { w.push_back(tc.witness); claims.push_back(tc.expected_result); }
    auto witness = AllocatedScalar::allocate(composer, w);
    auto res = range_check(composer, {cases[0].min_range}, {cases[0].max_range}, witness);
    EXPECT(composer.circuit_size() == 3 + 7 * (4 * 19 + 11), "row count 4k+11, k=19");
    EXPECT(satisfied_with_claims(composer, res, claims), "range_check verdicts");
    // and the negated claims are all rejected: 7 unsatisfied rows
    StandardComposer c2;
    auto w2 = AllocatedScalar::allocate(c2, w);
    auto r2 = range_check(c2, {cases[0].min_range}, {cases[0].max_range}, w2);
    std::vector<BlsScalar> neg;
    for (bool b : claims) neg.push_back(b ? BlsScalar::zero() : BlsScalar::one());
    c2.constrain_to_constant(r2, neg);
    EXPECT(c2.check_circuit_satisfied().first == 7, "negated claims rejected");
    // the 127-bit case (tests/range_gadgets_tests.rs:158-163)
    StandardComposer c3;
    auto w3 = AllocatedScalar::allocate(c3, {two_pow(127) - BlsScalar::one()});
    auto r3 = range_check(c3, {two_pow(126)}, {two_pow(127) + BlsScalar::one()}, w3);
    EXPECT(satisfied_with_claims(c3, r3, {true}), "127-bit range");
}

static void test_maybe_equal() {
    StandardComposer composer;
    auto a = AllocatedScalar::allocate(composer, {BlsScalar::from(100), BlsScalar::from(20)});
    auto b = AllocatedScalar::allocate(composer, {BlsScalar::from(100), BlsScalar::from(3330)});
    auto bit = maybe_equal(composer, a, b);
    EXPECT(satisfied_with_claims(composer, bit, {true, false}), "maybe_equal");
}

static void test_conditionally_select_0() {
    StandardComposer composer;
    BlsScalar rnd = BlsScalar::from(0x1234567890abcdefULL) * BlsScalar::from(0xfedcba9876543211ULL);
    auto value = composer.add_input({rnd, rnd});
    auto selector = composer.add_input({BlsScalar::zero(), BlsScalar::one()});
    auto res = conditionally_select_zero(composer, value, selector);
    composer.constrain_to_constant(res, {BlsScalar::zero()});
    auto v = composer.check_circuit_satisfied();
    // selector 0 -> 0 (ok); selector 1 with a random value -> the claim "0" is rejected (scalar_gadgets_tests.rs:106,:119)
    EXPECT(v.first == 1, "select_zero: exactly the selector=1 instance violates res == 0");
}

static void test_conditionally_select_1() {
    StandardComposer composer;
    BlsScalar rnd = BlsScalar::from(0x0123456789abcdefULL) * BlsScalar::from(0x1111111111111111ULL);
    auto value = composer.add_input({rnd, rnd});
    auto selector = composer.add_input({BlsScalar::zero(), BlsScalar::one()});
    auto res = conditionally_select_one(composer, value, selector);
    // constrain_to_constant(res, 0, Some(-expected)): selector 0 -> 1, selector 1 -> value
    composer.constrain_to_constant(res, {BlsScalar::zero()}, {-BlsScalar::one(), -rnd});
    EXPECT(composer.check_circuit_satisfied().first == 0, "select_one");
}

static void test_is_not_zero() {
    BlsScalar r1 = BlsScalar::from(77) * BlsScalar::from(0xabcdef0123456789ULL), r2 = BlsScalar::from(78) * BlsScalar::from(0xabcdef0123456789ULL);
    {   // zero -> Err(NonExistingInverse)
        StandardComposer composer;
        auto value = composer.add_input({BlsScalar::zero()});
        Error e; EXPECT(!is_non_zero(composer, value, {BlsScalar::zero()}, &e) && e == Error::NonExistingInverse, "is_non_zero(0) errs");
        EXPECT(composer.circuit_size() == 3 + 1 && composer.num_variables() == 5 + 1 + 1, "partial append: 1 var + 1 row");
    }
    {   // different value / value_assigned -> Ok, but unsatisfied
        StandardComposer composer;
        auto value = composer.add_input({r1});
        EXPECT(is_non_zero(composer, value, {r2}), "is_non_zero mismatch returns Ok");
        EXPECT(composer.check_circuit_satisfied().first != 0, "is_non_zero mismatch rejected");
    }
    {   // equal and non-zero -> satisfied
        StandardComposer composer;
        auto value = composer.add_input({r1});
        EXPECT(is_non_zero(composer, value, {r1}), "is_non_zero ok");
        EXPECT(composer.check_circuit_satisfied().first == 0, "is_non_zero satisfied");
    }
}

// What the reference tests do next is prover.prove(&ck) (range_gadgets_tests.rs:90-91).  Its first round -- wire polynomials by
// ifft, then their KZG commitments -- is checked here through the structure of the SRS: against powers_of_g[i] = beta^i * G
// the commitment of a polynomial is poly(beta) * G.
static void prover_first_round_test() {
    StandardComposer composer;
    auto witness = AllocatedScalar::allocate(composer, {BlsScalar::from(50001), BlsScalar::from(250001)});
    range_check(composer, {BlsScalar::from(50000)}, {BlsScalar::from(250000)}, witness);
    EXPECT(composer.check_circuit_satisfied().first == 0, "range_check satisfied before the prover round");
    const uint32_t k = composer.domain_log_size();
    const uint64_t n = 1ull << k;
    EXPECT(n >= composer.circuit_size() && n / 2 < composer.circuit_size(), "domain = next power of two");
    const BlsScalar beta = BlsScalar::from(0x5eed5eed5eedULL) * BlsScalar::from(0x9e3779b97f4a7c15ULL);
    const auto powers = composer.srs_powers(beta, n);
    const auto polys = composer.wire_polynomials(k);
    const auto commits = composer.commit_wire_polynomials(powers, k);
    for (int w = 0; w < 4; w++) {
        BlsScalar at_beta = BlsScalar::zero();
        for (uint64_t i = n; i-- > 0;) at_beta = at_beta * beta + polys[(size_t)w * n + i];        // Horner
        const pg_g1_affine want = composer.commit({powers[0]}, {at_beta});
        EXPECT(std::memcmp(&want, &commits[w], sizeof(want)) == 0, "commit(w_poly) == w_poly(beta) * G");
    }
    // the same commitments from the wire values against the Lagrange-basis form of the SRS
    const auto from_values = composer.commit_wire_evaluations(composer.srs_lagrange(beta, k), k);
    for (int w = 0; w < 4; w++) EXPECT(std::memcmp(&from_values[w], &commits[w], sizeof(pg_g1_affine)) == 0, "evaluation-form commitment == coefficient-form commitment");
    // ifft then fft is the identity on a wire-polynomial column
    std::vector<BlsScalar> col(polys.begin(), polys.begin() + n);
    const auto evals = composer.fft(col, false);
    EXPECT(composer.fft(evals, true) == col, "ifft(fft(x)) == x");
}

// The native range gate the reference points to for power-of-two bounds (range.rs:9-12): composer.range_gate(witness, num_bits)
// is satisfied iff the witness fits num_bits.  One composer per case, as a failing case spoils the whole circuit.
static void range_gate_test() {
    struct TestCase { BlsScalar witness; size_t num_bits; bool fits; };
    std::vector<TestCase> cases = {
        {BlsScalar::from(0), 2, true}, {BlsScalar::from(3), 2, true}, {BlsScalar::from(4), 2, false},
        {BlsScalar::from(1023), 10, true}, {BlsScalar::from(1024), 10, false},
        {two_pow(64) - BlsScalar::one(), 64, true}, {two_pow(64), 64, false},
        {BlsScalar::zero() - BlsScalar::one(), 254, false}, {BlsScalar::zero() - BlsScalar::one(), 256, true},
    };
    for (auto& tc : cases) {
        StandardComposer composer;
        const uint64_t rows0 = composer.circuit_size();
        auto witness = AllocatedScalar::allocate(composer, {tc.witness});
        composer.range_gate(witness.var, tc.num_bits);
        EXPECT(composer.circuit_size() - rows0 == (tc.num_bits + 7) / 8 + 2, "range_gate rows");
        EXPECT((composer.check_circuit_satisfied().first == 0) == tc.fits, "range_gate verdict");
    }
}

// Round 2: every Result of a batched is_non_zero kept (scalar_gadgets_tests.rs:199: zero -> Err, without stopping the batch), the
// structure-aware and fused checks, the sharded verdict / gathers as a world of one rank, and the export for the import adapter.
static void batch_extensions_test() {
    const BlsScalar r1 = BlsScalar::from(77) * BlsScalar::from(0xabcdef0123456789ULL);
    {
        StandardComposer composer;
        std::vector<BlsScalar> vals = {r1, BlsScalar::zero(), r1 + r1, BlsScalar::zero(), r1};
        auto v = composer.add_input(vals);
        const auto errs = is_non_zero_each(composer, v, vals);
        EXPECT(errs == std::vector<bool>({false, true, false, true, false}), "per-instance NonExistingInverse flags");
        EXPECT(composer.circuit_size() == 3 + 3 * 5 && composer.check_circuit_satisfied().first == 2, "errored instances fail their last row");
        StandardComposer ref_layout;
        auto v2 = ref_layout.add_input(vals);
        is_non_zero_each(ref_layout, v2, vals, true);
        EXPECT(ref_layout.circuit_size() == 3 + 3 * 3 + 2 * 1 && ref_layout.num_variables() == 5 + 5 + 3 * 3 + 2 * 1, "reference layout: 1 variable + 1 row per errored call");
    }
    for (int fused = 0; fused < 2; fused++) {
        StandardComposer composer(0, PG_CHECK_SPARSE, fused != 0);
        std::vector<BlsScalar> w;
        for (uint64_t i = 0; i < 300; i++) w.push_back(i % 2 ? -BlsScalar::from(i + 1) : BlsScalar::from(50000 + i));
        auto witness = AllocatedScalar::allocate(composer, w);
        auto res = range_check(composer, {BlsScalar::from(50000)}, {BlsScalar::from(250000)}, witness);
        const std::vector<pg_op> ops = {{PG_OP_ADD_INPUT, 0, 300, 0, 0}, {PG_OP_RANGE_CHECK, 19, 300, 0, 0}};
        const auto plan = shard_plan(ops, 1, true);
        EXPECT(plan[0][1].row_base == 3 && plan[0][1].var_base == 5 + 300 && plan[0][1].inst_hi == 300, "shard plan of one rank = the whole circuit");
        const auto v = composer.check_sharded(plan[0]);
        EXPECT(v.n_unsat == 0 && v.first_bad_row == UINT64_MAX, "sharded verdict (world of one)");
        const auto all = composer.gather_column(res, 300);
        EXPECT(all == composer.values(res) && all[0] == BlsScalar::one() && all[1] == BlsScalar::zero(), "gathered results");
        const uint64_t vars_per = 2 * 19 + 523;
        EXPECT(composer.gather_variables(1, 300 * vars_per) == composer.variables(5 + 300, 300 * vars_per), "gathered witness shard == the composer's variables");
        // a file of this run's own: a fixed name would collide with (or be left unwritable by) another user's run on the same host
        const char* tmpdir = std::getenv("TMPDIR");
        std::string path = std::string(tmpdir && *tmpdir ? tmpdir : "/tmp") + "/pg_cpp_mirror_export_XXXXXX";
        const int fd = mkstemp(&path[0]);
        EXPECT(fd >= 0, "temporary export file");
        if (fd < 0) continue;
        close(fd);
        composer.export_to(path, true);
        FILE* f = std::fopen(path.c_str(), "rb");
        char magic[8] = {0}; uint32_t ver = 0, flags = 0; uint64_t head[3] = {0, 0, 0};
        const bool read_ok = f && std::fread(magic, 1, 8, f) == 8 && std::fread(&ver, 4, 1, f) == 1 && std::fread(&flags, 4, 1, f) == 1 && std::fread(head, 8, 3, f) == 3;
        if (f) std::fclose(f);
        std::remove(path.c_str());
        EXPECT(read_ok && std::memcmp(magic, "PGB2EXP1", 8) == 0 && ver == 1 && flags == 1 && head[0] == composer.circuit_size() && head[1] == composer.num_variables() && head[2] == 3,
               "export header: rows, variables, calls (fresh + add_input + range_check)");
    }
}

int main() {
    try {
        range_gate_test(); batch_extensions_test();
        max_bound_test(); range_check_test(); test_maybe_equal();
        test_conditionally_select_0(); test_conditionally_select_1(); test_is_not_zero();
        prover_first_round_test();
    } catch (const EngineError& e) {
        std::printf("EngineError %d: %s\n", e.code, e.what());
        return 2;
    }
    std::printf(failures ? "reference tests: %d FAILED\n" : "reference tests: all passed\n", failures);
    return failures ? 1 : 0;
}
