// engine.hpp -- host logic of the device-resident batched composer, generic over a Backend.
//
// The shipped library (engine.cu) instantiates Engine<CudaBackend> only.  tests/emu instantiates the same logic over a
// host backend that runs the per-instance bodies in a loop, which lets template construction, Variable/row numbering,
// operand resolution and witness arithmetic be tested without a GPU; that build is test infrastructure and is never
// loaded by the package.
//
// Backend concept:
//   bool init(const pg_cfg&), void shutdown(), const char* error()
//   void* alloc(size_t), void release(void*)                       -- device memory
//   bool h2d(void*, const void*, size_t), bool d2h(void*, const void*, size_t) [d2h returns after the data arrived]
//   bool d2d(void*, const void*, size_t), bool sync()
//   template<class Body> bool run_simple(const typename Body::Args&, uint64_t n, int cls)
//   bool run_batch_inv(const BatchInvArgs&, int cls)            -- out_slot = in_slot^-1 (or 0) over table slots
//   bool run_check(const CheckArgs&, const SparseProg&), bool run_check_rows(const CheckRowsBody::Args&)
//   bool run_check_gates(const CheckArgs&)                        -- segments with rows of the range widget (GateRowsCheckBody)
//   bool sort_pairs(const uint32_t* keys, const uint32_t* vals, uint32_t* keys_out, uint32_t* vals_out, uint64_t n, uint32_t key_bits)
//   bool run_msm_buckets(const MsmBucketBody::Args&)             -- one thread per part of a bucket run (launch shape chosen by the backend)
//   bool exclusive_sum(const uint32_t* in, uint32_t* out, uint64_t n)
//   bool run_ntt_pass(const NttPassArgs&, uint64_t n_blocks)    -- one group of butterfly stages over all tiles (ntt.cuh)
//   bool run_fr_scan(const uint4* in, uint4* out, uint64_t n, uint4* total, uint4* scratch) -- exclusive prefix product (scan.cuh);
//        optional: a backend without it (the test-only loop backend) runs FrScanSerialBody, the defining serial loop
//   bool run_fr_ruffini(const uint4* in, uint4* out, uint64_t n, const uint4* pw, uint4* rem, uint4* scratch) -- division by (X - p)
//        (scan.cuh); optional like run_fr_scan: without it FrRuffiniSerialBody runs
//   bool upload_pow2(const Fr*), bool imad_peak(double*, double*), bool ubench(int, double*), timing(pg_timing*, bool reset)
#pragma once
#include <stdio.h>
#include <algorithm>
#include <stdexcept>
#include <map>
#include <string>
#include <vector>
#include <type_traits>
#include "../../include/pg_b200.h"
#include "templates.hpp"
#include "shard.hpp"
#include "ntt.cuh"
#include "scan.cuh"
#include "msm.cuh"
#include "g1fft.cuh"

namespace pg {

enum { CLS_CHECK = 0, CLS_WITNESS = 1, CLS_OTHER = 2 };

struct Column { uint32_t seg; uint32_t local; uint64_t inst_off; uint64_t n; };
constexpr uint64_t INPUT_CHUNKS = 4, INPUT_CHUNK_MIN = 1ull << 20;     // host inputs of at least 2^20 scalars (32 MiB) are copied in four chunks

struct Segment {
    Template t;
    uint64_t n_inst = 0, n_alloc = 0, base_row = 0, base_var = 0;
    uint4* fr = nullptr; uint32_t* bits = nullptr; uint4* param = nullptr;
    DevRow* d_rows = nullptr; uint32_t* d_varloc = nullptr; uint32_t* d_pool = nullptr; Fr* d_fold = nullptr;   // views into d_image
    void* d_image = nullptr;
    DevTab tabs[MAX_TABS] = {};
    std::vector<DevRow> rows;
    std::vector<SpOp> sp_ops; SpOp* d_sp = nullptr;    // structure-aware row program (PG_CHECK_SPARSE only)
    std::vector<Column> operands;       // the columns bound as operands (for the permutation map)
    bool other_gates = false;           // some row belongs to another widget than the arithmetic one (GATE_RANGE / GATE_NONE)
    bool fused_ok = false;              // PG_F_FUSED_CHECK: every row was evaluated while the witness was generated, and no Variable was overwritten since
    bool owns_table = true;             // false: fr / bits / param and d_image are views into buffers another segment owns
};
// a pre-allocated variable table (and image memory) for a segment that is a VIEW of another segment's storage: instance i of the
// view is instance first + i of the owner (the SoA stride is the owner's)
struct SegmentView { uint4* fr; uint64_t n_alloc; unsigned char* image; size_t image_bytes; };

// Range templates are expensive to build on the host (k = 253: 1019 rows, 514 pool entries, ~0.2 ms with the structure-aware program),
// and a caller that repeats a circuit (a prover loop, the benches) repeats them: the built template, and the resolved segment image
// (rows with addresses, structure-aware program, extended pool) when the tables sit at the same device addresses, are kept.
struct RangeTemplateKey {
    int range_check; uint32_t k; int uniform; Fr m, negmin;
    bool operator==(const RangeTemplateKey& o) const { return range_check == o.range_check && k == o.k && uniform == o.uniform && fr_eq(m, o.m) && fr_eq(negmin, o.negmin); }
};
struct ResolvedKey {
    uint64_t n_alloc; const void *fr, *bits, *param; int check_mode; DevTab tab1; uint32_t op_loc, op_local;     // operand: its table, location and local index
    bool operator==(const ResolvedKey& o) const {
        return n_alloc == o.n_alloc && fr == o.fr && bits == o.bits && param == o.param && check_mode == o.check_mode && tab1.fr == o.tab1.fr &&
               tab1.bits == o.tab1.bits && tab1.stride == o.tab1.stride && op_loc == o.op_loc && op_local == o.op_local;
    }
};
struct CachedRange {
    RangeTemplateKey key; Template t; uint32_t result_local = 0;
    bool resolved = false; ResolvedKey rkey{}; std::vector<DevRow> rows; std::vector<SpOp> sp_ops; std::vector<Fr> pool; std::vector<unsigned char> img;
    uint64_t stamp = 0;
};
constexpr size_t RANGE_CACHE_SLOTS = 16;

inline Fr fr_from_pg(const pg_fr& x) {
    Fr r;
    for (int i = 0; i < 4; i++) { r.v[2 * i] = (uint32_t)x.l[i]; r.v[2 * i + 1] = (uint32_t)(x.l[i] >> 32); }
    return r;
}

static_assert(sizeof(pg_proof_evaluations) == 17 * sizeof(pg_fr), "pg_proof_evaluations is 17 consecutive scalars");
inline pg_fr fr_to_pg(const Fr& x) {
    pg_fr r;
    for (int i = 0; i < 4; i++) r.l[i] = (uint64_t)x.v[2 * i] | ((uint64_t)x.v[2 * i + 1] << 32);
    return r;
}

// whether a backend brings its own device-wide prefix product (Engine::fr_scan)
template <class B, class = void> struct has_fr_scan : std::false_type {};
template <class B> struct has_fr_scan<B, std::void_t<decltype(&B::run_fr_scan)>> : std::true_type {};
// whether a backend brings its own device-wide Ruffini division (Engine::fr_ruffini)
template <class B, class = void> struct has_fr_ruffini : std::false_type {};
template <class B> struct has_fr_ruffini<B, std::void_t<decltype(&B::run_fr_ruffini)>> : std::true_type {};

template <class BE>
class Engine {
public:
    BE be;
    pg_cfg cfg{};
    std::string err;
    std::vector<Segment> segs;
    std::vector<Column> cols;
    std::vector<DevSeg> dsegs;
    DevSeg* d_segs = nullptr; size_t d_segs_cap = 0; bool dsegs_dirty = true;
    unsigned long long* d_counters = nullptr;
    uint64_t n_rows = 0, n_vars = 0;
    std::multimap<size_t, void*> pool_free;          // size -> buffer (exact-size reuse across composer resets)
    std::map<void*, size_t> pool_live;
    std::vector<void*> scratch;                      // temporaries that must outlive the enqueued work (freed on reset)

    std::vector<CachedRange> range_cache; uint64_t cache_clock = 0;
    CachedRange* range_cache_get(const RangeTemplateKey& key) {            // the slot of `key`, built on a miss (the least recently used slot is replaced)
        for (auto& c : range_cache) if (c.key == key) { c.stamp = ++cache_clock; return &c; }
        CachedRange* slot;
        if (range_cache.size() < RANGE_CACHE_SLOTS) { range_cache.emplace_back(); slot = &range_cache.back(); }
        else { slot = &range_cache[0]; for (auto& c : range_cache) if (c.stamp < slot->stamp) slot = &c; *slot = CachedRange(); }
        slot->key = key; slot->stamp = ++cache_clock;
        slot->t = make_range_template(key.range_check != 0, key.k, key.uniform != 0, key.m, key.negmin, &slot->result_local);
        return slot;
    }

    // ------------------------------------------------------------------------------------------------ memory
    void* dalloc(size_t bytes) {
        if (bytes == 0) bytes = 16;
        auto it = pool_free.find(bytes);
        void* p;
        if (it != pool_free.end()) { p = it->second; pool_free.erase(it); }
        else {
            p = be.alloc(bytes);
            if (!p && !pool_free.empty()) {          // out of memory with idle buffers parked in the pool: give them back and retry
                be.sync();
                for (auto& kv : pool_free) be.release(kv.second);
                pool_free.clear();
                p = be.alloc(bytes);
            }
        }
        if (p) pool_live[p] = bytes;
        return p;
    }
    void dfree(void* p) {
        if (!p) return;
        auto it = pool_live.find(p);
        if (it == pool_live.end()) return;
        pool_free.insert({it->second, p});
        pool_live.erase(it);
    }
    // give back temporaries allocated since `mark`; only valid right after a call that synchronised the stream (d2h)
    void release_scratch_from(size_t mark) {
        for (size_t k = mark; k < scratch.size(); k++) dfree(scratch[k]);
        scratch.resize(mark);
    }
    int fail(int code, const std::string& what) { err = what; if (code == PG_ERR_CUDA && be.error()[0]) err += std::string(": ") + be.error(); return code; }

    // ------------------------------------------------------------------------------------------------ lifetime
    int create(const pg_cfg& c) {
        cfg = c;
        if (!be.init(cfg)) return fail(be.no_device() ? PG_ERR_NO_DEVICE : PG_ERR_CUDA, "backend init");
        // 2^i * R table (selectors of range.rs:146 and accumulator increments)
        h_pow2[0] = fr_one();
        for (int i = 1; i < 256; i++) h_pow2[i] = fr_add(h_pow2[i - 1], h_pow2[i - 1]);
        if (!be.upload_pow2(h_pow2)) return fail(PG_ERR_CUDA, "upload 2^i table");
        d_counters = (unsigned long long*)dalloc(CNT_WORDS * sizeof(unsigned long long));
        if (!d_counters) return fail(PG_ERR_OOM, "counters");
        return reset();
    }
    void destroy() {
        be.sync();
        release_segments();
        dfree(d_counters); dfree(d_segs); dfree(ntt_tw); ntt_tw = nullptr; dfree(fb_table_gen); fb_table_gen = nullptr;
        for (auto& kv : pool_free) be.release(kv.second);
        for (auto& kv : pool_live) be.release(kv.first);
        pool_free.clear(); pool_live.clear();
        be.shutdown();
    }
    void release_segments() {
        for (auto& s : segs) if (s.owns_table) { dfree(s.fr); dfree(s.bits); dfree(s.param); dfree(s.d_image); }
        for (void* p : scratch) dfree(p);
        scratch.clear(); segs.clear(); cols.clear(); dsegs.clear(); dsegs_dirty = true;
        be.drop_result_chunks();
        n_rows = 0; n_vars = 0;
    }
    // StandardComposer::new(): 5 variables, 3 rows
    int reset() {
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        release_segments();
        { const int rcc = reset_counters(true); if (rcc) return rcc; }
        validation_pending = false;
        std::vector<Fr> vals;
        Template t = make_preamble_template(&vals);
        int rc = push_segment(std::move(t), 1, nullptr, 0);
        if (rc) return rc;
        Segment& s = segs.back();
        std::vector<uint4> img(2 * vals.size());
        for (size_t j = 0; j < vals.size(); j++) {
            img[2 * j] = make_uint4(vals[j].v[0], vals[j].v[1], vals[j].v[2], vals[j].v[3]);
            img[2 * j + 1] = make_uint4(vals[j].v[4], vals[j].v[5], vals[j].v[6], vals[j].v[7]);
        }
        if (!be.h2d(s.fr, img.data(), img.size() * sizeof(uint4)) || !be.sync()) return fail(PG_ERR_CUDA, "preamble upload");
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ segments
    const Column* column(pg_col c) const { return (c >= 1 && c <= cols.size()) ? &cols[c - 1] : nullptr; }
    pg_col new_column(uint32_t seg, uint32_t local, uint64_t n) { cols.push_back(Column{seg, local, 0, n}); return (pg_col)cols.size(); }

    DevTab view_of(const Column& c) const {
        const Segment& s = segs[c.seg];
        DevTab v;
        v.fr = s.fr ? s.fr + 2 * c.inst_off : nullptr;
        v.bits = s.bits ? s.bits + c.inst_off : nullptr;
        v.stride = s.n_alloc; v.var_base = s.base_var + c.inst_off * s.t.n_vars; v.var_stride = s.t.n_vars;
        return v;
    }
    uint32_t loc_of(const Column& c) const { return segs[c.seg].t.var_loc[c.local]; }

    // Compiles the resolved rows of a segment into the structure-aware program (layout.h SpOp, bodies.cuh SparseProgBody):
    // per term -- selector 0 or zero-variable wire: nothing; packed bit variables: masks (b*b = b; the selectors of all terms
    // on the same bits are summed on the host, a sum of 0 removes them); selector +-1: add / subtract; otherwise one
    // multiplication -- then q_c and PI.  The last operation of a row carries SP_ROW_END; rows left without any operation
    // hold for every witness and are merged into SP_TRIVIAL runs.  Folded selector sums are appended to the segment's pool.
    static void build_sparse_program(Segment& s) {
        auto mem = [](uint8_t op, uint64_t addr, uint32_t stride, uint16_t sel, uint8_t sh) { SpOp o; o.addr = addr; o.stride = stride; o.sel = sel; o.op = op; o.sh = sh; return o; };
        auto pool_index = [&](const Fr& c) -> uint16_t {
            for (size_t k = 0; k < s.t.pool.size(); k++) if (fr_eq(s.t.pool[k], c)) return (uint16_t)k;
            s.t.pool.push_back(c);
            return (uint16_t)(s.t.pool.size() - 1);
        };
        struct BitTerm { uint64_t addr[2]; uint8_t sh[2]; int n; Fr sum; };
        auto& out = s.sp_ops; out.clear();
        for (const DevRow& d : s.rows) {
            const size_t row_start = out.size();
            std::vector<BitTerm> bit_terms;
            for (int k = 0; k < 5; k++) {
                const uint16_t si = d.sel[k];
                if (si == POOL_ZERO) continue;
                int wires[2], nw = 0;
                wires[nw++] = k ? k - 1 : 0;
                if (k == 0) wires[nw++] = 1;
                bool zero = false; int bits[2], nb = 0, frs[2], nf = 0;
                for (int j = 0; j < nw; j++) {
                    const uint32_t kind = loc_kind(d.loc[wires[j]]);
                    if (kind == LOC_ZERO) zero = true; else if (kind == LOC_BIT) bits[nb++] = wires[j]; else frs[nf++] = wires[j];
                }
                if (zero) continue;
                if (nb == 2 && d.addr[bits[0]] == d.addr[bits[1]] && (d.loc[bits[0]] & 31u) == (d.loc[bits[1]] & 31u)) nb = 1;   // b*b = b
                const bool general = si != POOL_ONE && si != POOL_MINUS_ONE;
                auto bit_op = [&](uint8_t op, int w, uint16_t sel) { return mem(op, d.addr[w], 4, sel, (uint8_t)(d.loc[w] & 31u)); };
                if (nf == 0) {                                      // bits only: selector * (product of bits); fold equal bit sets
                    BitTerm bt; bt.n = nb; bt.sum = s.t.pool[si];
                    for (int j = 0; j < nb; j++) { bt.addr[j] = d.addr[bits[j]]; bt.sh[j] = (uint8_t)(d.loc[bits[j]] & 31u); }
                    if (nb == 2 && (bt.addr[0] > bt.addr[1] || (bt.addr[0] == bt.addr[1] && bt.sh[0] > bt.sh[1]))) { std::swap(bt.addr[0], bt.addr[1]); std::swap(bt.sh[0], bt.sh[1]); }
                    bool merged = false;
                    for (BitTerm& o : bit_terms) {
                        bool same = o.n == bt.n;
                        for (int j = 0; same && j < bt.n; j++) same = o.addr[j] == bt.addr[j] && o.sh[j] == bt.sh[j];
                        if (same) { o.sum = fr_add(o.sum, bt.sum); merged = true; break; }
                    }
                    if (!merged) bit_terms.push_back(bt);
                    continue;
                }
                for (int j = 0; j < nb; j++) out.push_back(bit_op(SP_MASK, bits[j], 0));
                if (nf == 1 && nb == 0) {
                    out.push_back(mem(si == POOL_ONE ? SP_ADD_FR : si == POOL_MINUS_ONE ? SP_SUB_FR : SP_MUL_SEL_FR, d.addr[frs[0]], 32, si, 0));
                    continue;
                }
                out.push_back(mem(SP_LOAD_FR, d.addr[frs[0]], 32, 0, 0));
                if (nf == 2) out.push_back(mem(SP_MUL_FR, d.addr[frs[1]], 32, 0, 0));
                if (general) out.push_back(mem(SP_MULSEL_V, 0, 0, si, 0));
                out.push_back(mem(SP_ADD_V, 0, 0, 0, si == POOL_MINUS_ONE ? 1 : 0));
            }
            for (const BitTerm& bt : bit_terms) {
                if (fr_is_zero(bt.sum)) continue;                   // e.g. b*b - b: (1 + -1) * b
                const uint16_t sel = pool_index(bt.sum);
                for (int j = 0; j + 1 < bt.n; j++) out.push_back(mem(SP_MASK, bt.addr[j], 4, 0, bt.sh[j]));
                out.push_back(mem(SP_BITSEL, bt.addr[bt.n - 1], 4, sel, bt.sh[bt.n - 1]));
            }
            auto param_addr = [&](int slot) { return (uint64_t)(uintptr_t)(s.param + 2 * ((uint64_t)slot * s.n_alloc)); };
            if (d.qc_param >= 0) out.push_back(mem(SP_ADD_FR, param_addr(d.qc_param), 32, 0, 0));
            else if (d.sel[5] != POOL_ZERO) out.push_back(mem(SP_ADD_POOL, 0, 0, d.sel[5], 0));
            if (d.pi_param >= 0) out.push_back(mem(SP_ADD_FR, param_addr(d.pi_param), 32, 0, 0));
            else if (d.pi_sel != POOL_ZERO) out.push_back(mem(SP_ADD_POOL, 0, 0, d.pi_sel, 0));
            if (out.size() > row_start) { out.back().op |= SP_ROW_END; continue; }
            if (!out.empty() && out.back().op == SP_TRIVIAL) out.back().stride++;      // `stride` of SP_TRIVIAL counts the rows (no memory operand: addr = 0)
            else out.push_back(mem(SP_TRIVIAL, 0, 1, 0, 0));
        }
        fold_chains(s);
    }
    // Peephole pass over the compiled program: runs of  [TRIVIAL(t)] ADD_FR(x_j) SUB_FR(x_{j+1}) BITSEL|ROW_END(bit_j, sel_j)  with consecutive
    // scalar slots and consecutive packed bits become one SP_CHAIN (layout.h).  Purely structural: nothing is assumed about the gadget
    // that produced the rows.  The L selectors are copied into a contiguous run of the pool (shared by chains with the same selectors).
    static void fold_chains(Segment& s) {
        const std::vector<SpOp> in = s.sp_ops;
        std::vector<SpOp>& out = s.sp_ops; out.clear();
        const uint64_t slot_step = (uint64_t)s.n_alloc * 32, word_step = (uint64_t)s.n_alloc * 4;
        std::vector<std::pair<std::vector<uint16_t>, uint16_t>> runs;          // selector lists already copied -> first pool index
        auto elem = [&](size_t p, uint32_t& triv) -> bool {                     // does a chain element start at p?  (4 operations, or 3 without leading trivial rows)
            triv = 0;
            if (p < in.size() && in[p].op == SP_TRIVIAL) { triv = in[p].stride; p++; }
            return p + 2 < in.size() && in[p].op == SP_ADD_FR && in[p + 1].op == SP_SUB_FR && in[p + 2].op == (SP_BITSEL | SP_ROW_END) &&
                   in[p].stride == 32 && in[p + 1].addr == in[p].addr + slot_step;
        };
        size_t p = 0;
        while (p < in.size()) {
            uint32_t triv = 0;
            if (!elem(p, triv) || triv + 1 > 255) { out.push_back(in[p++]); continue; }
            // extend the run
            const size_t width = triv ? 4 : 3;
            size_t L = 1, e = p;
            std::vector<uint16_t> sels;
            auto at = [&](size_t k, int which) -> const SpOp& { return in[p + k * width + (triv ? 1 : 0) + which]; };
            sels.push_back(at(0, 2).sel);
            while (L < 256) {
                uint32_t t2 = 0;
                if (!elem(p + L * width, t2) || t2 != triv) break;
                const SpOp &prev_bit = at(L - 1, 2), &bit = at(L, 2);
                const bool next_bit = (bit.addr == prev_bit.addr && bit.sh == prev_bit.sh + 1) || (prev_bit.sh == 31 && bit.sh == 0 && bit.addr == prev_bit.addr + word_step);
                if (!next_bit || at(L, 0).addr != at(L - 1, 1).addr) break;
                sels.push_back(bit.sel);
                L++;
            }
            (void)e;
            if (L < SP_CHAIN_MIN || s.t.pool.size() + L > 2000) { out.push_back(in[p++]); continue; }
            uint16_t first = 0xffff;
            for (auto& kv : runs) if (kv.first.size() >= L && std::equal(sels.begin(), sels.end(), kv.first.begin())) { first = kv.second; break; }
            if (first == 0xffff) {
                first = (uint16_t)s.t.pool.size();
                for (uint16_t si : sels) { const Fr c = s.t.pool[si]; s.t.pool.push_back(c); }
                runs.push_back({sels, first});
            }
            SpOp c0, c1, c2;
            c0.addr = at(0, 0).addr; c0.stride = 32; c0.sel = first; c0.op = SP_CHAIN; c0.sh = at(0, 2).sh;
            c1.addr = at(0, 2).addr; c1.stride = 4; c1.sel = (uint16_t)L; c1.op = SP_CHAIN_AUX; c1.sh = (uint8_t)(triv + 1);
            c2.addr = slot_step; c2.stride = 0; c2.sel = 0; c2.op = SP_CHAIN_AUX; c2.sh = 0;
            out.push_back(c0); out.push_back(c1); out.push_back(c2);
            p += L * width;
        }
    }
    // Appends a segment of n instances of template t whose operands are the given columns.  Allocates the variable
    // table, resolves the symbolic wires and uploads the row program.  The witness kernels run afterwards.
    static size_t image_bytes_bound(const Template& T) {      // upper bound of a segment image (the structure-aware program has at most ~12 operations per row)
        const size_t fold = 8 * std::min(T.rows.size(), T.pool.size());     // fold table: 8 constants per distinct q_m
        return (T.rows.size() * (sizeof(DevRow) + 12 * sizeof(SpOp)) + T.var_loc.size() * sizeof(uint32_t) + (T.pool.size() + 8 * T.rows.size() + fold) * sizeof(Fr) + 255) & ~(size_t)255;
    }
    int push_segment(Template&& t, uint64_t n, const Column* operands, uint32_t n_operands, const SegmentView* view = nullptr, CachedRange* cache = nullptr) {
        Segment s;
        s.t = std::move(t);
        s.n_inst = n; s.n_alloc = n ? n : 1;
        s.base_row = n_rows; s.base_var = n_vars;
        const Template& T = s.t;
        if (view) {                                   // storage exists already (templates with fr slots only)
            if (T.n_planes || T.n_params) return fail(PG_ERR_STATE, "segment views hold scalar slots only");
            s.owns_table = false; s.fr = view->fr; s.n_alloc = view->n_alloc;
        }
        else if (T.n_fr) { s.fr = (uint4*)dalloc((size_t)T.n_fr * 2 * s.n_alloc * sizeof(uint4)); if (!s.fr) return fail(PG_ERR_OOM, "variable table"); }
        if (T.n_planes) { s.bits = (uint32_t*)dalloc((size_t)T.n_planes * 8 * s.n_alloc * sizeof(uint32_t)); if (!s.bits) return fail(PG_ERR_OOM, "bit planes"); }
        if (T.n_params) { s.param = (uint4*)dalloc((size_t)T.n_params * 2 * s.n_alloc * sizeof(uint4)); if (!s.param) return fail(PG_ERR_OOM, "parameter table"); }
        s.tabs[0].fr = s.fr; s.tabs[0].bits = s.bits; s.tabs[0].stride = s.n_alloc; s.tabs[0].var_base = s.base_var; s.tabs[0].var_stride = T.n_vars;
        for (uint32_t e = 0; e < n_operands; e++) { s.tabs[e + 1] = view_of(operands[e]); s.operands.push_back(operands[e]); }
        ResolvedKey rk; memset(&rk, 0, sizeof(rk));
        rk.n_alloc = s.n_alloc; rk.fr = s.fr; rk.bits = s.bits; rk.param = s.param; rk.check_mode = cfg.check_mode; rk.tab1 = s.tabs[1];
        if (cache && n_operands == 1) { rk.op_loc = loc_of(operands[0]); rk.op_local = operands[0].local; }
        std::vector<unsigned char> img;
        if (cache && n_operands == 1 && !view && cache->resolved && cache->rkey == rk) {      // same template over tables at the same addresses: the image is known
            s.rows = cache->rows; s.sp_ops = cache->sp_ops; s.t.pool = cache->pool; img = cache->img;
        } else {
        s.rows.resize(T.rows.size());
        std::map<uint16_t, uint16_t> fold_of;        // q_m pool index -> its entry in the fold table (order of first use)
        std::vector<Fr> fold;
        for (size_t r = 0; r < T.rows.size(); r++) {
            const RowT& src = T.rows[r]; DevRow d; memset(&d, 0, sizeof(d));
            for (int w = 0; w < 4; w++) {
                const WireRef& wr = src.w[w];
                if (wr.src == 0) { d.loc[w] = loc_make(LOC_ZERO, 0, 0); d.var[w] = 0; }
                else if (wr.src == 1) { d.loc[w] = T.var_loc[wr.idx]; d.var[w] = wr.idx; }
                else { const uint32_t e = wr.src - 2u; d.loc[w] = loc_with_tab(loc_of(operands[e]), e + 1); d.var[w] = operands[e].local; }
            }
            for (int k = 0; k < 6; k++) d.sel[k] = src.sel[k];
            d.pi_sel = src.pi_sel; d.qc_param = src.qc_param; d.pi_param = src.pi_param; d.gate = src.gate;
            auto f = fold_of.find(src.sel[0]);
            if (f == fold_of.end()) {
                f = fold_of.emplace(src.sel[0], (uint16_t)fold_of.size()).first;
                fold.resize(fold.size() + 8);
                fr_fold_constants(&fold[fold.size() - 8], T.pool[src.sel[0]]);
            }
            d.fold = f->second;
            if (src.gate != GATE_ARITH) s.other_gates = true;
            for (int w = 0; w < 4; w++) {            // instance-0 address of each wire value (see DevRow::addr)
                const uint32_t kind = loc_kind(d.loc[w]), pay = loc_payload(d.loc[w]);
                const DevTab& tb = s.tabs[loc_tab(d.loc[w])];
                if (kind == LOC_FR) d.addr[w] = (uint64_t)(uintptr_t)(tb.fr + 2 * ((uint64_t)pay * tb.stride));
                else if (kind == LOC_BIT) d.addr[w] = (uint64_t)(uintptr_t)(tb.bits + (uint64_t)((pay >> 8) * 8 + ((pay & 255u) >> 5)) * tb.stride);
                else d.addr[w] = 0;
            }
            s.rows[r] = d;
        }
        if (cfg.check_mode == PG_CHECK_SPARSE && !s.other_gates) build_sparse_program(s);   // segments with range rows have their own check body
        // rows | variable map | selector pool | fold table | structure-aware program go up in ONE copy (one staging image per segment);
        // every section starts 32-byte aligned (fr_load_fold reads the fold table with 256-bit loads)
        const size_t b_rows0 = s.rows.size() * sizeof(DevRow), b_var0 = (T.var_loc.size() * sizeof(uint32_t) + 31) & ~(size_t)31, b_pool0 = T.pool.size() * sizeof(Fr);
        const size_t b_fold0 = fold.size() * sizeof(Fr), b_sp0 = s.sp_ops.size() * sizeof(SpOp);
        img.resize(b_rows0 + b_var0 + b_pool0 + b_fold0 + b_sp0);
        if (b_sp0) memcpy(img.data() + b_rows0 + b_var0 + b_pool0 + b_fold0, s.sp_ops.data(), b_sp0);
        if (b_fold0) memcpy(img.data() + b_rows0 + b_var0 + b_pool0, fold.data(), b_fold0);
        if (b_rows0) memcpy(img.data(), s.rows.data(), b_rows0);
        if (!T.var_loc.empty()) memcpy(img.data() + b_rows0, T.var_loc.data(), T.var_loc.size() * sizeof(uint32_t));
        memcpy(img.data() + b_rows0 + b_var0, T.pool.data(), b_pool0);
        if (cache && n_operands == 1 && !view) {
            cache->resolved = true; cache->rkey = rk; cache->rows = s.rows; cache->sp_ops = s.sp_ops; cache->pool = s.t.pool; cache->img = img;
        }
        }
        const size_t b_rows = s.rows.size() * sizeof(DevRow), b_var = (T.var_loc.size() * sizeof(uint32_t) + 31) & ~(size_t)31, b_pool = T.pool.size() * sizeof(Fr);
        const size_t b_sp = s.sp_ops.size() * sizeof(SpOp);
        if (view && img.size() > view->image_bytes) return fail(PG_ERR_STATE, "segment view: image larger than its reserved memory");
        unsigned char* d_img = view ? view->image : (unsigned char*)dalloc(img.size());
        if (!d_img || !be.h2d(d_img, img.data(), img.size())) return fail(d_img ? PG_ERR_CUDA : PG_ERR_OOM, "template upload");
        s.d_rows = b_rows ? (DevRow*)d_img : nullptr;
        s.d_varloc = T.var_loc.empty() ? nullptr : (uint32_t*)(d_img + b_rows);
        s.d_pool = (uint32_t*)(d_img + b_rows + b_var);
        s.d_fold = (Fr*)(d_img + b_rows + b_var + b_pool);       // the fold table fills the image up to the program
        s.d_sp = b_sp ? (SpOp*)(d_img + img.size() - b_sp) : nullptr;
        s.d_image = d_img;
        // (pageable sources: cudaMemcpyAsync has consumed them when it returns; they stay alive in the Segment anyway)
        segs.push_back(std::move(s));
        Segment& S = segs.back();
        n_rows += n * S.t.rows.size(); n_vars += n * (uint64_t)S.t.n_vars;
        dsegs_dirty = true;                         // the device copy of the segment table is refreshed by the read-back calls
        return PG_OK;
    }
    DevSeg make_dseg(const Segment& s) const {
        DevSeg d; memset(&d, 0, sizeof(d));
        d.base_row = s.base_row; d.base_var = s.base_var; d.n_inst = s.n_inst;
        d.n_rows = (uint32_t)s.t.rows.size(); d.n_vars = s.t.n_vars;
        for (int k = 0; k < MAX_TABS; k++) d.tab[k] = s.tabs[k];
        d.rows = s.d_rows; d.varloc = s.d_varloc; d.pool = s.d_pool; d.param = s.param; d.param_stride = s.n_alloc;
        return d;
    }
    int sync_dsegs() {
        if (!dsegs_dirty) return PG_OK;
        dsegs_dirty = false;
        dsegs.resize(segs.size());
        for (size_t k = 0; k < segs.size(); k++) dsegs[k] = make_dseg(segs[k]);
        if (dsegs.size() > d_segs_cap) {
            if (d_segs) scratch.push_back(d_segs);       // may still be read by enqueued kernels
            d_segs_cap = dsegs.size() * 2 + 8;
            d_segs = (DevSeg*)dalloc(d_segs_cap * sizeof(DevSeg));
            if (!d_segs) return fail(PG_ERR_OOM, "segment table");
        }
        if (!be.h2d(d_segs, dsegs.data(), dsegs.size() * sizeof(DevSeg))) return fail(PG_ERR_CUDA, "segment table upload");
        return PG_OK;
    }
    // removes the last segment again (used when a call is rejected after its witness kernel ran)
    void pop_segment() {
        Segment& s = segs.back();
        n_rows -= s.n_inst * s.t.rows.size(); n_vars -= s.n_inst * (uint64_t)s.t.n_vars;
        if (s.owns_table) { scratch.push_back(s.fr); scratch.push_back(s.bits); scratch.push_back(s.param); scratch.push_back(s.d_image); }
        segs.pop_back();
        dsegs_dirty = true;
    }

    // host pointer -> device scratch copy (or pass-through for device pointers)
    const uint4* stage(const pg_fr* p, uint64_t count, int on_device, int* rc) {
        *rc = PG_OK;
        if (on_device) return reinterpret_cast<const uint4*>(p);
        void* d = dalloc(count * sizeof(pg_fr));
        if (!d) { *rc = fail(PG_ERR_OOM, "staging buffer"); return nullptr; }
        scratch.push_back(d);
        if (!be.h2d(d, p, count * sizeof(pg_fr))) { *rc = fail(PG_ERR_CUDA, "input copy"); return nullptr; }
        return reinterpret_cast<const uint4*>(d);
    }
    // Reads the counters back (synchronises).  Unreduced caller scalars seen by any ingest kernel since the composer was reset are
    // reported here: the composer then holds values the reference type cannot represent and must be reset.
    bool validation_pending = false;                 // an ingest check was enqueued since the counters were last read
    int read_counters(unsigned long long* out) {
        if (!be.d2h(out, d_counters, CNT_WORDS * sizeof(unsigned long long))) return fail(PG_ERR_CUDA, "counter read");
        validation_pending = false;
        if (out[CNT_BAD_INPUT]) {
            char msg[160];
            snprintf(msg, sizeof(msg), "%llu input scalar(s) not fully reduced (>= q), first at index %llu of its batch: reset the composer",
                     out[CNT_BAD_INPUT], out[CNT_FIRST_BAD_INPUT]);
            return fail(PG_ERR_ARG, msg);
        }
        return PG_OK;
    }
    // re-initialises the per-call words; `all`: also the sticky bad-input words (composer reset)
    int reset_counters(bool all = false) {
        static const unsigned long long init[CNT_WORDS] = {0, ~0ull, 0, 0, ~0ull, 0, ~0ull, 0, ~0ull, 0, 0, 0};
        if (!be.h2d(d_counters, init, (all ? (size_t)CNT_WORDS : (size_t)CNT_STICKY) * sizeof(unsigned long long))) return fail(PG_ERR_CUDA, "counter reset");
        return PG_OK;
    }
    // pg_sync: everything enqueued has finished, and no ingest check has failed
    int sync_checked() {
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        if (!validation_pending) return PG_OK;
        unsigned long long c[CNT_WORDS];
        return read_counters(c);
    }
    static bool host_reduced(const pg_fr& x) { return fr_is_reduced(fr_from_pg(x)); }

    // ------------------------------------------------------------------------------------------------ gadgets
    int add_input_batch(uint64_t n, const pg_fr* values, int on_device, pg_col* out) {
        if (!out || (n && !values)) return fail(PG_ERR_ARG, "add_input_batch: null argument");
        int rc = push_segment(make_add_input_template(), n, nullptr, 0);
        if (rc) return rc;
        Segment& s = segs.back();
        // a one-slot table of 32-byte scalars has exactly the caller's layout (BlsScalar[n]): the values are copied straight in
        // Large host batches arrive in INPUT_CHUNKS chunks on the backend's input stream; a range gadget called on the column next
        // starts on the first chunk while the others are still in flight (run_simple_chunked), anything else waits for all of them.
        const bool chunked = !on_device && n >= INPUT_CHUNK_MIN;
        const uint64_t chunk = (((n + INPUT_CHUNKS - 1) / INPUT_CHUNKS) + 1023) & ~1023ull;
        // every scalar is checked for full reduction on the device once it has arrived (chunked copies: chunk by chunk on the input stream)
        if (n && !(on_device ? be.d2d(s.fr, values, n * sizeof(pg_fr))
                   : chunked ? be.h2d_chunked(s.fr, values, n, sizeof(pg_fr), chunk, d_counters)
                             : be.h2d(s.fr, values, n * sizeof(pg_fr)))) return fail(PG_ERR_CUDA, "add_input copy");
        if (n && !chunked) {
            ValidateBody::Args va{s.fr, 0, n, d_counters};
            if (!be.template run_simple<ValidateBody>(va, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "input validation kernel");
        }
        if (n) validation_pending = true;
        *out = new_column((uint32_t)segs.size() - 1, 0, n);
        return PG_OK;
    }

    int range_batch(bool is_range_check, const pg_fr* mn, const pg_fr* mx, uint64_t n_bounds, int on_device, pg_col wit, pg_col* out, uint64_t* num_bits) {
        const Column* w = column(wit);
        if (!w || !out || !mx || (is_range_check && !mn)) return fail(PG_ERR_ARG, "range gadget: bad argument");
        const uint64_t n = w->n;
        if (n_bounds != 1 && n_bounds != n) return fail(PG_ERR_ARG, "range gadget: n_bounds must be 1 or the column length");
        const bool uniform = n_bounds == 1;
        // the first bound fixes num_bits (public data): k = num_bits_closest_power_of_two(max - 1), range.rs:87-90
        pg_fr mx0, mn0 = {{0, 0, 0, 0}};
        if (on_device) {
            if (!be.d2h(&mx0, mx, sizeof(pg_fr))) return fail(PG_ERR_CUDA, "bound read");
            if (is_range_check && !be.d2h(&mn0, mn, sizeof(pg_fr))) return fail(PG_ERR_CUDA, "bound read");
        } else { mx0 = mx[0]; if (is_range_check) mn0 = mn[0]; }
        if (!host_reduced(mx0) || !host_reduced(mn0)) return fail(PG_ERR_ARG, "range gadget: bound not fully reduced (>= q)");
        const Fr m0 = fr_sub(fr_from_pg(mx0), fr_one());
        const Fr negmin0 = fr_neg(fr_from_pg(mn0));
        const uint32_t k = num_bits_from_canonical(fr_from_mont(m0));
        int rc = PG_OK;
        const uint4 *d_mx = nullptr, *d_mn = nullptr;
        if (!uniform) {
            d_mx = stage(mx, n, on_device, &rc); if (!d_mx) return rc;
            if (is_range_check) { d_mn = stage(mn, n, on_device, &rc); if (!d_mn) return rc; }
            if ((rc = reset_counters())) return rc;
            validation_pending = true;
        }
        uint32_t result_local = 0;
        Column operand = *w;
        RangeTemplateKey tkey; memset(&tkey, 0, sizeof(tkey));
        tkey.range_check = is_range_check ? 1 : 0; tkey.k = k; tkey.uniform = uniform ? 1 : 0;
        if (uniform) { tkey.m = m0; tkey.negmin = negmin0; }          // (per-instance bounds: the template holds parameter slots, not values)
        CachedRange* cached = range_cache_get(tkey);
        result_local = cached->result_local;
        { Template tcopy = cached->t; rc = push_segment(std::move(tcopy), n, &operand, 1, nullptr, cached); }
        if (rc) return rc;
        Segment& s = segs.back();
        RangeArgs a; memset(&a, 0, sizeof(a));
        a.x_tab = s.tabs[1]; a.x_loc = loc_with_tab(loc_of(operand), 0);     // the body indexes its single operand table directly
        a.fr = s.fr; a.bits = s.bits; a.param = s.param; a.stride = s.n_alloc; a.n = n; a.k = k;
        a.uniform = uniform ? 1 : 0; a.m = m0; a.negmin = negmin0; a.max_aos = d_mx; a.min_aos = d_mn;
        a.param_m = s.t.param_m >= 0 ? (uint32_t)s.t.param_m : 0; a.param_negmin = s.t.param_negmin >= 0 ? (uint32_t)s.t.param_negmin : 0;
        a.d[0] = s.t.decomp[0]; a.d[1] = s.t.decomp[1]; a.slot_o = s.t.slot_o; a.counters = d_counters;
        if (n) {
            // witness generation: decomposition (everything up to u = acc - v) -> batch inversion z = u^-1|0 -> y (and y1*y2)
            BatchInvArgs inv; memset(&inv, 0, sizeof(inv));
            inv.fr = s.fr; inv.stride = s.n_alloc; inv.n = n; inv.n_pairs = is_range_check ? 2 : 1;
            for (uint32_t e = 0; e < inv.n_pairs; e++) { inv.in_slot[e] = a.d[e].u; inv.out_slot[e] = a.d[e].z; }
            // the operand's table, when the operand is a whole column of its segment (chunks of a pending input copy are instance ranges of it)
            const Segment& os = segs[operand.seg];
            const void* whole = (operand.inst_off == 0 && operand.n == os.n_inst) ? (const void*)os.fr : nullptr;
            // PG_F_FUSED_CHECK (structure-aware mode only): the same kernels also evaluate the rows they generate
            const bool fused = fused_mode();
            a.base_row = s.base_row; a.n_rows = (uint32_t)s.t.rows.size();
            // decomposition -> inversion -> results; with the fused check, behind a chunked input copy, the three run chunk by chunk, so
            // that an asynchronous read of the results (pg_col_read, dst_on_device = 2) starts on the first chunk while the later ones
            // are computed (without the fused check that copy runs under the gate-check kernel anyway)
            bool ok;
            if (fused)
                ok = is_range_check ? be.template run_range_pipeline<RangePre<true, true>, RangePost<true, true>>(a, inv, n, whole, s.fr, true)
                                    : be.template run_range_pipeline<RangePre<false, true>, RangePost<false, true>>(a, inv, n, whole, s.fr, true);
            else
                ok = is_range_check ? be.template run_range_pipeline<RangePre<true>, RangePost<true>>(a, inv, n, whole, s.fr, false)
                                    : be.template run_range_pipeline<RangePre<false>, RangePost<false>>(a, inv, n, whole, s.fr, false);
            if (!ok) return fail(PG_ERR_CUDA, "range witness kernels");
            if (fused) { s.fused_ok = true; be.count_check(PG_CK_FUSED, n * s.t.rows.size()); }
        }
        if (!uniform && n) {
            unsigned long long c[CNT_WORDS];
            if ((rc = read_counters(c))) return rc;
            if (c[CNT_MIXED_BITS]) { pop_segment(); return fail(PG_ERR_MIXED_BITS, "per-instance bounds give different num_bits"); }
        }
        if (num_bits) *num_bits = k;
        *out = new_column((uint32_t)segs.size() - 1, result_local, n);
        return PG_OK;
    }

    // PG_F_FUSED_CHECK (structure-aware mode): the gadget's own kernels evaluate its rows; marks the segment and counts the rows
    bool fused_mode() const { return (cfg.flags & PG_F_FUSED_CHECK) && cfg.check_mode == PG_CHECK_SPARSE; }
    FusedSite fused_site(const Segment& s) const { return fused_mode() ? FusedSite{d_counters, s.base_row} : FusedSite{nullptr, 0}; }
    void mark_fused(Segment& s) { if (fused_mode() && s.n_inst) { s.fused_ok = true; be.count_check(PG_CK_FUSED, s.n_inst * s.t.rows.size()); } }

    int maybe_equal_batch(pg_col ca, pg_col cb, pg_col* out) {
        const Column *a = column(ca), *b = column(cb);
        if (!a || !b || !out || a->n != b->n) return fail(PG_ERR_ARG, "maybe_equal_batch: bad columns");
        Column ops[2] = {*a, *b}; uint32_t result_local = 0;
        int rc = push_segment(make_maybe_equal_template(&result_local), ops[0].n, ops, 2);
        if (rc) return rc;
        Segment& s = segs.back();
        MaybeEqualArgs g{s.tabs[1], s.tabs[2], loc_with_tab(loc_of(ops[0]), 0), loc_with_tab(loc_of(ops[1]), 0), s.fr, s.n_alloc, ops[0].n, fused_site(s)};
        if (g.n) {
            BatchInvArgs inv; memset(&inv, 0, sizeof(inv));
            inv.fr = s.fr; inv.stride = s.n_alloc; inv.n = g.n; inv.n_pairs = 1; inv.in_slot[0] = 0; inv.out_slot[0] = 1;
            if (!be.template run_batch_inv_fused<MaybeEqualFused>(inv, g, CLS_WITNESS)) return fail(PG_ERR_CUDA, "maybe_equal kernel");
            mark_fused(s);
        }
        *out = new_column((uint32_t)segs.size() - 1, result_local, g.n);
        return PG_OK;
    }

    int is_non_zero_batch(pg_col cv, const pg_fr* assigned, int on_device, uint64_t* n_err, uint64_t* first_err) {
        const Column* v = column(cv);
        if (!v || (v->n && !assigned)) return fail(PG_ERR_ARG, "is_non_zero_batch: bad argument");
        const uint64_t n = v->n;
        int rc; const uint4* src = n ? stage(assigned, n, on_device, &rc) : nullptr;
        if (n && !src) return rc;
        if ((rc = reset_counters())) return rc;
        validation_pending = true;
        Column operand = *v;
        rc = push_segment(make_is_non_zero_template(false), n, &operand, 1);
        if (rc) return rc;
        {
            Segment& s = segs.back();
            IsNonZeroFused::Args g{src, s.fr, s.n_alloc, n, d_counters, nullptr, s.tabs[1], loc_with_tab(loc_of(operand), 0), FusedSite{nullptr, 0}};   // (`?` semantics may truncate the segment: not fused)
            BatchInvArgs inv; memset(&inv, 0, sizeof(inv));
            inv.fr = s.fr; inv.stride = s.n_alloc; inv.n = n; inv.n_pairs = 1; inv.in_slot[0] = 0; inv.out_slot[0] = 1;
            if (n && !be.template run_batch_inv_fused<IsNonZeroFused>(inv, g, CLS_WITNESS)) return fail(PG_ERR_CUDA, "is_non_zero kernel");
        }
        unsigned long long c[CNT_WORDS];
        if ((rc = read_counters(c))) return rc;
        if (n_err) *n_err = c[CNT_N_ERR];
        if (first_err) *first_err = c[CNT_N_ERR] ? c[CNT_FIRST_ERR] : ~0ull;
        if (!c[CNT_N_ERR]) return PG_OK;
        // Err(NonExistingInverse) at instance f: instances < f are complete; instance f has appended var_assigned and the
        // assert_equal row (scalar.rs:69-71) before returning at :79; nothing after it runs.
        const uint64_t f = c[CNT_FIRST_ERR];
        {
            Segment& s = segs.back();
            n_rows -= (n - f) * s.t.rows.size(); n_vars -= (n - f) * (uint64_t)s.t.n_vars;
            s.n_inst = f;
            dsegs_dirty = true;
        }
        Column part = *v; part.inst_off += f; part.n = 1;
        rc = push_segment(make_is_non_zero_template(true), 1, &part, 1);
        if (rc) return rc;
        Segment& p = segs.back();
        AddInputBody::Args g{src + 2 * f, p.fr, p.n_alloc, 1};
        if (!be.template run_simple<AddInputBody>(g, 1, CLS_OTHER)) return fail(PG_ERR_CUDA, "is_non_zero partial kernel");
        err = "is_non_zero: value_assigned is zero (NonExistingInverse)";
        return PG_ERR_NON_EXISTING_INVERSE;
    }

    // for i { results[i] = is_non_zero(composer, var_i, value_assigned_i); } -- every Result kept (scalar.rs:63-97 called without `?`):
    // a batch does not abort on one zero.  err_flags[i] = 1 where the call returned Err(NonExistingInverse).
    //   PG_NZ_UNIFORM  : every instance appends the full 3 variables + 3 rows (numbering first + 3i); an errored instance holds
    //                    var_assigned = 0, inv = 0 (invert().unwrap_or(zero), the convention of scalar.rs:122), one = 1, so its row
    //                    var*inv - 1 = 0 is unsatisfied: one segment, no host round trip besides the error count.
    //   PG_NZ_REFERENCE: the composer the reference loop leaves behind -- an errored call has appended var_assigned and the
    //                    assert_equal row only (scalar.rs:69-71, return at :79): 1 variable + 1 row.  The same device table is
    //                    re-described as 2*n_err + 1 segment views (runs of completed instances / single partial instances).
    static constexpr uint64_t NZ_MAX_VIEWS = 1ull << 20;
    int is_non_zero_flags(pg_col cv, const pg_fr* assigned, int on_device, uint8_t* err_flags, int layout, uint64_t* n_err_out) {
        const Column* v = column(cv);
        if (!v || (v->n && !assigned) || (layout != PG_NZ_UNIFORM && layout != PG_NZ_REFERENCE)) return fail(PG_ERR_ARG, "is_non_zero_batch_flags: bad argument");
        const uint64_t n = v->n;
        if (n_err_out) *n_err_out = 0;
        int rc; const uint4* src = n ? stage(assigned, n, on_device, &rc) : nullptr;
        if (n && !src) return rc;
        const bool need_flags = err_flags || layout == PG_NZ_REFERENCE;
        uint8_t* d_flags = nullptr;
        if (need_flags && n) {
            if (err_flags && on_device) d_flags = err_flags;
            else { d_flags = (uint8_t*)dalloc(n); if (!d_flags) return fail(PG_ERR_OOM, "error flags"); scratch.push_back(d_flags); }
        }
        if ((rc = reset_counters())) return rc;
        validation_pending = true;
        const Column operand = *v;
        rc = push_segment(make_is_non_zero_template(false), n, &operand, 1);
        if (rc) return rc;
        const size_t seg_index = segs.size() - 1;
        if (n) {
            Segment& s = segs.back();
            // the uniform layout keeps every instance's three rows where the kernel numbers them: its rows can be evaluated in the kernel
            const FusedSite site = layout == PG_NZ_UNIFORM ? fused_site(s) : FusedSite{nullptr, 0};
            IsNonZeroFused::Args g{src, s.fr, s.n_alloc, n, d_counters, d_flags, s.tabs[1], loc_with_tab(loc_of(operand), 0), site};
            BatchInvArgs inv; memset(&inv, 0, sizeof(inv));
            inv.fr = s.fr; inv.stride = s.n_alloc; inv.n = n; inv.n_pairs = 1; inv.in_slot[0] = 0; inv.out_slot[0] = 1;
            if (!be.template run_batch_inv_fused<IsNonZeroFused>(inv, g, CLS_WITNESS)) return fail(PG_ERR_CUDA, "is_non_zero kernel");
            if (layout == PG_NZ_UNIFORM) mark_fused(s);
        }
        unsigned long long c[CNT_WORDS];
        if ((rc = read_counters(c))) return rc;
        const uint64_t n_err = c[CNT_N_ERR];
        if (n_err_out) *n_err_out = n_err;
        std::vector<uint8_t> h_flags;
        if (layout == PG_NZ_REFERENCE && n_err) { h_flags.resize(n); if (!be.d2h(h_flags.data(), d_flags, n)) return fail(PG_ERR_CUDA, "error flag copy"); }
        if (err_flags && !on_device && n) {
            if (!h_flags.empty()) memcpy(err_flags, h_flags.data(), n);
            else if (!be.d2h(err_flags, d_flags, n)) return fail(PG_ERR_CUDA, "error flag copy");
        }
        if (layout == PG_NZ_UNIFORM || !n_err) return PG_OK;
        // ---- reference layout: runs of completed instances and single partial instances, as views of the table just filled
        if (2 * n_err + 1 > NZ_MAX_VIEWS) return fail(PG_ERR_ARG, "is_non_zero_batch_flags: too many errored instances for the reference layout (use PG_NZ_UNIFORM)");
        uint4* table; uint64_t stride;
        {
            Segment& s = segs[seg_index];
            table = s.fr; stride = s.n_alloc;
            uint64_t f = 0; while (!h_flags[f]) f++;                       // the owning segment keeps the instances before the first error
            n_rows -= (n - f) * s.t.rows.size(); n_vars -= (n - f) * (uint64_t)s.t.n_vars;
            s.n_inst = f;
            dsegs_dirty = true;
        }
        const Template full = make_is_non_zero_template(false), part = make_is_non_zero_template(true);
        const size_t b_full = image_bytes_bound(full), b_part = image_bytes_bound(part);
        unsigned char* arena = (unsigned char*)dalloc((n_err + 1) * b_full + n_err * b_part);
        if (!arena) return fail(PG_ERR_OOM, "segment view images");
        scratch.push_back(arena);
        uint64_t i = segs[seg_index].n_inst;
        while (i < n) {
            uint64_t j = i;
            const bool err_run = h_flags[i] != 0;
            if (err_run) j = i + 1; else while (j < n && !h_flags[j]) j++;
            Column sub = operand; sub.inst_off += i; sub.n = j - i;
            SegmentView view{table + 2 * i, stride, arena, err_run ? b_part : b_full};
            arena += view.image_bytes;
            Template t = err_run ? part : full;
            if ((rc = push_segment(std::move(t), j - i, &sub, 1, &view))) return rc;
            i = j;
        }
        return PG_OK;
    }

    int select_batch(bool one, pg_col cx, pg_col csel, pg_col* out) {
        const Column *x = column(cx), *s0 = column(csel);
        if (!x || !s0 || !out || x->n != s0->n) return fail(PG_ERR_ARG, "select: bad columns");
        Column ops[2] = {*x, *s0}; uint32_t result_local = 0;
        int rc = push_segment(make_select_template(one, &result_local), ops[0].n, ops, 2);
        if (rc) return rc;
        Segment& s = segs.back();
        const uint64_t n = ops[0].n;
        bool ok = true;
        if (one) { SelectOneBody::Args g{s.tabs[1], s.tabs[2], loc_with_tab(loc_of(ops[0]), 0), loc_with_tab(loc_of(ops[1]), 0), s.fr, s.n_alloc, n, fused_site(s)}; if (n) ok = be.template run_simple<SelectOneBody>(g, n, CLS_WITNESS); }
        else { SelectZeroBody::Args g{s.tabs[1], s.tabs[2], loc_with_tab(loc_of(ops[0]), 0), loc_with_tab(loc_of(ops[1]), 0), s.fr, s.n_alloc, n, fused_site(s)}; if (n) ok = be.template run_simple<SelectZeroBody>(g, n, CLS_WITNESS); }
        if (!ok) return fail(PG_ERR_CUDA, "select kernel");
        if (n) mark_fused(s);
        *out = new_column((uint32_t)segs.size() - 1, result_local, n);
        return PG_OK;
    }

    // for i { composer.range_gate(witness_i, num_bits) } -- dusk-plonk's native range gate (SURVEY.md 8f.4), see tmpl_range_gate
    int range_gate_batch(pg_col cw, uint32_t num_bits) {
        const Column* w = column(cw);
        if (!w) return fail(PG_ERR_ARG, "range_gate_batch: unknown column");
        if (num_bits % 2 != 0 || num_bits < 2 || num_bits > 256) return fail(PG_ERR_ARG, "range_gate_batch: num_bits must be even and in 2..256");
        Column operand = *w; const uint64_t n = operand.n;
        int rc = push_segment(make_range_gate_template(num_bits), n, &operand, 1);
        if (rc) return rc;
        Segment& s = segs.back();
        RangeGateBody::Args g{s.tabs[1], loc_with_tab(loc_of(operand), 0), s.fr, s.n_alloc, n, num_bits / 2};
        if (n && !be.template run_simple<RangeGateBody>(g, n, CLS_WITNESS)) return fail(PG_ERR_CUDA, "range_gate witness kernel");
        return PG_OK;
    }

    int constrain_batch(pg_col ca, const pg_fr* constant, uint64_t n_const, const pg_fr* pi, uint64_t n_pi, int on_device) {
        const Column* a = column(ca);
        if (!a || !constant) return fail(PG_ERR_ARG, "constrain_to_constant_batch: bad argument");
        const uint64_t n = a->n;
        if ((n_const != 1 && n_const != n) || (pi && n_pi != 1 && n_pi != n)) return fail(PG_ERR_ARG, "constrain_to_constant_batch: lengths must be 1 or n");
        const bool cu = n_const == 1, pu = pi && n_pi == 1;
        pg_fr c0 = {{0, 0, 0, 0}}, p0 = {{0, 0, 0, 0}};
        if (cu) { if (on_device) { if (!be.d2h(&c0, constant, sizeof(pg_fr))) return fail(PG_ERR_CUDA, "constant read"); } else c0 = constant[0]; }
        if (pu) { if (on_device) { if (!be.d2h(&p0, pi, sizeof(pg_fr))) return fail(PG_ERR_CUDA, "pi read"); } else p0 = pi[0]; }
        if (!host_reduced(c0) || !host_reduced(p0)) return fail(PG_ERR_ARG, "constrain_to_constant_batch: scalar not fully reduced (>= q)");
        int rc = PG_OK; const uint4 *d_c = nullptr, *d_p = nullptr;
        if (!cu) { d_c = stage(constant, n, on_device, &rc); if (!d_c) return rc; }
        if (pi && !pu) { d_p = stage(pi, n, on_device, &rc); if (!d_p) return rc; }
        Column operand = *a;
        rc = push_segment(make_constrain_template(cu, fr_neg(fr_from_pg(c0)), pi != nullptr, pu, fr_from_pg(p0)), n, &operand, 1);
        if (rc) return rc;
        Segment& s = segs.back();
        if (s.t.n_params && n) {
            ConstrainBody::Args g{d_c, d_p, s.param, s.n_alloc, n, s.t.param_qc, s.t.param_pi, d_counters};
            validation_pending = true;
            if (!be.template run_simple<ConstrainBody>(g, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "constrain kernel");
        }
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ verdict
    // Enqueues the gate check of every segment.  `mine` != nullptr (sharded composer, see shard.hpp): segment k + 1 is this rank's
    // part of call k of the whole circuit, and its rows are numbered from mine[k].row_base -- their indices in the SEQUENTIAL
    // composer -- so that the first bad row needs no translation before the all-reduce; the fresh composer's three rows exist on
    // every rank and are checked by rank 0 only.
    int enqueue_checks(const pg_op_shard* mine = nullptr, bool with_preamble = true, bool skip_fused = false) {
        for (size_t k = 0; k < segs.size(); k++) {
            const Segment& s = segs[k];
            if (!s.n_inst || s.t.rows.empty()) continue;
            if (mine && k == 0 && !with_preamble) continue;
            if (s.fused_ok && skip_fused) continue;  // verdict already in CNT_FUSED_* (pg_check adds it; a sharded check renumbers rows and evaluates them again)
            CheckArgs a; memset(&a, 0, sizeof(a));
            for (int j = 0; j < MAX_TABS; j++) a.tab[j] = s.tabs[j];
            a.param = s.param; a.param_stride = s.n_alloc; a.rows = s.d_rows; a.pool = s.d_pool; a.fold = s.d_fold;
            a.n_rows = (uint32_t)s.t.rows.size(); a.n_pool = (uint32_t)s.t.pool.size();
            a.n_inst = s.n_inst; a.base_row = (mine && k > 0) ? mine[k - 1].row_base : s.base_row; a.counters = d_counters; a.mode = cfg.check_mode;
            if (s.other_gates) {                     // rows of the range widget: per-row body, one thread per (row, instance)
                if (!be.run_check_gates(a)) return fail(PG_ERR_CUDA, "gate-check kernel (range rows)");
                continue;
            }
            const SparseProg prog{s.d_sp, (uint32_t)s.sp_ops.size()};
            if (!be.run_check(a, prog)) return fail(PG_ERR_CUDA, "gate-check kernel");
        }
        return PG_OK;
    }
    int check(uint64_t* n_unsat, uint64_t* first_bad) {
        int rc = reset_counters();
        if (rc) return rc;
        if ((rc = enqueue_checks(nullptr, true, true))) return rc;
        unsigned long long c[CNT_WORDS];
        if ((rc = read_counters(c))) return rc;
        bool any_fused = false;
        for (const Segment& s : segs) any_fused = any_fused || s.fused_ok;
        if (any_fused) { c[CNT_UNSAT] += c[CNT_FUSED_UNSAT]; if (c[CNT_FUSED_FIRST] < c[CNT_FIRST_BAD]) c[CNT_FIRST_BAD] = c[CNT_FUSED_FIRST]; }
        if (n_unsat) *n_unsat = c[CNT_UNSAT];
        if (first_bad) *first_bad = c[CNT_FIRST_BAD];
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ multi-GPU (SURVEY.md 8e)
    // One process (and one ctx) per GPU; the communicator spans the ranks of one box.  Without pg_comm_init the calls below act as
    // a world of one rank (no NCCL is loaded).
    int comm_init(const uint8_t* id, uint32_t rank, uint32_t world) {
        if (!id || !world || rank >= world) return fail(PG_ERR_ARG, "comm_init: bad rank / world / id");
        if (!be.comm_init(id, (int)rank, (int)world)) return fail(PG_ERR_CUDA, std::string("comm_init: ") + be.comm_error());
        return PG_OK;
    }
    // pg_check of a sharded composer + the all-reduce of the verdict: every rank returns the verdict of the whole circuit.
    // *n_err (in: this rank's NonExistingInverse count, out: the sum) may be null.
    int check_sharded(const pg_op_shard* mine, uint64_t n_ops, uint64_t* n_unsat, uint64_t* first_bad, uint64_t* n_err) {
        if (mine && n_ops + 1 != segs.size()) return fail(PG_ERR_STATE, "check_sharded: the composer must hold exactly one segment per planned call");
        if (mine) for (uint64_t k = 0; k < n_ops; k++)
            if (mine[k].inst_hi - mine[k].inst_lo != segs[k + 1].n_inst) return fail(PG_ERR_ARG, "check_sharded: a call's instance count differs from its planned range");
        int rc = reset_counters();
        if (rc) return rc;
        if ((rc = enqueue_checks(mine, be.comm_rank() == 0, true))) return rc;
        // segments whose rows were evaluated inside witness generation: their recorded verdict joins in, renumbered like the launched checks
        std::vector<FusedSpan> spans;
        for (size_t k = 0; k < segs.size(); k++) {
            const Segment& s = segs[k];
            if (!s.fused_ok || !s.n_inst) continue;
            spans.push_back(FusedSpan{s.base_row, s.base_row + s.n_inst * s.t.rows.size(), (mine && k > 0) ? mine[k - 1].row_base : s.base_row});
        }
        const FusedSpan* d_spans = nullptr;
        if (!spans.empty()) {
            void* d = dalloc(spans.size() * sizeof(FusedSpan));
            if (!d) return fail(PG_ERR_OOM, "fused span table");
            scratch.push_back(d);
            if (!be.h2d(d, spans.data(), spans.size() * sizeof(FusedSpan))) return fail(PG_ERR_CUDA, "fused span upload");
            d_spans = (const FusedSpan*)d;
        }
        unsigned long long v[4];
        if (!be.comm_verdict(d_counters, n_err ? *n_err : 0ull, v, d_spans, (uint32_t)spans.size())) return fail(PG_ERR_CUDA, std::string("verdict all-reduce: ") + be.comm_error());
        validation_pending = false;
        if (v[3]) return fail(PG_ERR_ARG, "input scalar(s) not fully reduced (>= q) on some rank: reset the composers");
        if (n_unsat) *n_unsat = v[0];
        if (n_err) *n_err = v[1];
        if (first_bad) *first_bad = v[2];
        return PG_OK;
    }
    // shards of a ragged all-gather, 32-byte units: `d_send` (mine units) -> dst (all ranks' shards in rank order)
    int gather_units(const uint4* d_send, uint64_t mine, pg_fr* dst, uint64_t capacity, int dst_on_device, uint64_t* counts_out, uint64_t* total_out) {
        const uint32_t world = (uint32_t)be.comm_world();
        std::vector<unsigned long long> counts(world);
        if (!be.comm_counts(mine, counts.data())) return fail(PG_ERR_CUDA, std::string("gather (counts): ") + be.comm_error());
        uint64_t total = 0;
        for (uint32_t g = 0; g < world; g++) { total += counts[g]; if (counts_out) counts_out[g] = counts[g]; }
        if (total_out) *total_out = total;
        if (total > capacity) return fail(PG_ERR_ARG, "gather: destination too small for the shards of all ranks");
        if (!total) return PG_OK;
        if (!dst) return fail(PG_ERR_ARG, "gather: null destination");
        const size_t mark = scratch.size();
        uint4* recv = dst_on_device ? reinterpret_cast<uint4*>(dst) : (uint4*)dalloc(total * sizeof(pg_fr));
        if (!recv) return fail(PG_ERR_OOM, "gather buffer");
        if (!dst_on_device) scratch.push_back(recv);
        if (!be.comm_gather(d_send, recv, counts.data())) return fail(PG_ERR_CUDA, std::string("gather: ") + be.comm_error());
        if (dst_on_device) return PG_OK;
        const int rc = deliver(dst, recv, total * sizeof(pg_fr), 0);
        release_scratch_from(mark);
        return rc;
    }
    // all-gather of a column (the per-instance results of a call): every rank receives the shards of all ranks, in rank order
    int gather_column(pg_col c, pg_fr* dst, uint64_t capacity, int dst_on_device, uint64_t* counts_out, uint64_t* total_out) {
        const Column* col = column(c);
        if (!col) return fail(PG_ERR_ARG, "gather_column: unknown column");
        const uint64_t n = col->n;
        const size_t mark = scratch.size();
        uint4* send = (uint4*)dalloc((n ? n : 1) * sizeof(pg_fr));
        if (!send) return fail(PG_ERR_OOM, "gather send buffer");
        scratch.push_back(send);
        if (n) {
            ColReadBody::Args a{view_of(*col), loc_with_tab(loc_of(*col), 0), send, n};
            if (!be.template run_simple<ColReadBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "col_read kernel");
        }
        const int rc = gather_units(send, n, dst, capacity, dst_on_device, counts_out, total_out);
        release_scratch_from(mark);                  // only touched by work on the engine's stream: stream order makes its reuse safe
        return rc;
    }
    // gather of witness shards: the Variables call `call` (0-based since the reset) appended on every rank, in the sequential
    // composer's Variable order (instance-major; ranks hold consecutive instance ranges, so rank order is instance order)
    int gather_variables(uint64_t call, pg_fr* dst, uint64_t capacity, int dst_on_device, uint64_t* total_out) {
        if (call + 1 >= segs.size()) return fail(PG_ERR_ARG, "gather_variables: no such call");
        const Segment& s = segs[call + 1];
        const uint64_t cnt = s.n_inst * (uint64_t)s.t.n_vars;
        if (cnt) { const int rcs = sync_dsegs(); if (rcs) return rcs; }      // (may park the old segment table in `scratch`: before the mark)
        const size_t mark = scratch.size();
        uint4* send = (uint4*)dalloc((cnt ? cnt : 1) * sizeof(pg_fr));
        if (!send) return fail(PG_ERR_OOM, "gather send buffer");
        scratch.push_back(send);
        if (cnt) {
            ReadVarsBody::Args a{d_segs, (uint32_t)dsegs.size(), s.base_var, cnt, send};
            if (!be.template run_simple<ReadVarsBody>(a, cnt, CLS_OTHER)) return fail(PG_ERR_CUDA, "read_variables kernel");
        }
        const int rc = gather_units(send, cnt, dst, capacity, dst_on_device, nullptr, total_out);
        release_scratch_from(mark);
        return rc;
    }
    int check_rows(uint64_t n, const pg_fr* w, const pg_fr* sel, const pg_fr* pi, int on_device, uint64_t* n_unsat, uint64_t* first_bad,
                   const pg_fr* q_arith = nullptr, const pg_fr* q_range = nullptr) {
        if (n && (!w || !sel)) return fail(PG_ERR_ARG, "check_rows: null argument");
        int rc = reset_counters();
        if (rc) return rc;
        if (n) {
            const uint4* dw = stage(w, 4 * n, on_device, &rc); if (!dw) return rc;
            const uint4* ds = stage(sel, 6 * n, on_device, &rc); if (!ds) return rc;
            const uint4* dp = nullptr;
            if (pi) { dp = stage(pi, n, on_device, &rc); if (!dp) return rc; }
            const uint4 *da = nullptr, *dr = nullptr;
            if (q_arith) { da = stage(q_arith, n, on_device, &rc); if (!da) return rc; }
            if (q_range) { dr = stage(q_range, n, on_device, &rc); if (!dr) return rc; }
            CheckRowsBody::Args a{dw, ds, dp, n, d_counters, da, dr};
            if (!be.run_check_rows(a)) return fail(PG_ERR_CUDA, "row-check kernel");
        }
        unsigned long long c[CNT_WORDS];
        if ((rc = read_counters(c))) return rc;
        if (n_unsat) *n_unsat = c[CNT_UNSAT];
        if (first_bad) *first_bad = c[CNT_FIRST_BAD];
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ read-back
    template <class T>
    int deliver(T* dst, const void* dev, size_t bytes, int dst_on_device) {   // dev -> caller memory
        if (dst_on_device) { if (!be.d2d(dst, dev, bytes)) return fail(PG_ERR_CUDA, "device copy"); }
        else if (!be.d2h(dst, dev, bytes)) return fail(PG_ERR_CUDA, "result copy");
        return PG_OK;
    }
    int read_variables(uint64_t var0, uint64_t cnt, pg_fr* dst, int dst_on_device) {
        if (var0 + cnt > n_vars || (cnt && !dst)) return fail(PG_ERR_ARG, "read_variables: range");
        if (!cnt) return PG_OK;
        const size_t mark = scratch.size();
        uint4* out = dst_on_device ? reinterpret_cast<uint4*>(dst) : (uint4*)dalloc(cnt * sizeof(pg_fr));
        if (!out) return fail(PG_ERR_OOM, "read buffer");
        if (!dst_on_device) scratch.push_back(out);
        { const int rcs = sync_dsegs(); if (rcs) return rcs; }
        ReadVarsBody::Args a{d_segs, (uint32_t)dsegs.size(), var0, cnt, out};
        if (!be.template run_simple<ReadVarsBody>(a, cnt, CLS_OTHER)) return fail(PG_ERR_CUDA, "read_variables kernel");
        if (dst_on_device) return PG_OK;
        const int rc = deliver(dst, out, cnt * sizeof(pg_fr), 0);
        release_scratch_from(mark);
        return rc;
    }
    // Fault injection (tests, diagnostics): overwrite the stored value of one Variable.  Packed bit variables cannot be poked.
    int poke_variable(uint64_t var, const pg_fr* value) {
        if (var >= n_vars || !value) return fail(PG_ERR_ARG, "poke_variable: unknown Variable or null value");
        if (!host_reduced(*value)) return fail(PG_ERR_ARG, "poke_variable: value not fully reduced (>= q)");
        for (size_t k = segs.size(); k-- > 0;) {
            Segment& s = segs[k];
            if (!s.n_inst || !s.t.n_vars || var < s.base_var) continue;
            const uint64_t off = var - s.base_var, i = off / s.t.n_vars; const uint32_t j = (uint32_t)(off % s.t.n_vars);
            if (i >= s.n_inst) return fail(PG_ERR_ARG, "poke_variable: Variable outside its segment");
            const uint32_t loc = s.t.var_loc[j];
            if (loc_kind(loc) != LOC_FR) return fail(PG_ERR_ARG, "poke_variable: packed bit variables cannot be overwritten");
            if (!be.h2d(s.fr + 2 * ((uint64_t)loc_payload(loc) * s.n_alloc + i), value, sizeof(pg_fr)) || !be.sync()) return fail(PG_ERR_CUDA, "poke copy");
            // the stored witness no longer is what generation verified: this segment and every segment that reads the Variable through an
            // operand column (segments are appended in call order: all later ones may) go back to the ordinary check.  The verdict
            // recorded at generation is ONE pair of sticky words for the whole composer, so the unsatisfied rows an invalidated segment
            // had recorded (is_non_zero instances that errored or mismatched) cannot be taken out of it again: the whole composer goes
            // back to the check kernels and the recorded verdict is dropped -- calls made after this start a fresh record.
            bool had_fused = false;
            for (Segment& t : segs) { had_fused = had_fused || t.fused_ok; t.fused_ok = false; }
            if (had_fused) {
                static const unsigned long long fresh[2] = {0, ~0ull};
                static_assert(CNT_FUSED_FIRST == CNT_FUSED_UNSAT + 1, "the two words are reset with one copy");
                if (!be.h2d(d_counters + CNT_FUSED_UNSAT, fresh, sizeof(fresh)) || !be.sync()) return fail(PG_ERR_CUDA, "poke: verdict record reset");
            }
            return PG_OK;
        }
        return fail(PG_ERR_ARG, "poke_variable: Variable not found");
    }
    int col_read(pg_col c, uint64_t i0, uint64_t cnt, pg_fr* dst, int dst_on_device) {
        const Column* col = column(c);
        if (!col || i0 + cnt > col->n || (cnt && !dst)) return fail(PG_ERR_ARG, "col_read: range");
        if (!cnt) return PG_OK;
        // a column is a strided set of variables: gather it with the add_input body run "in reverse" (SoA -> AoS)
        const size_t mark = scratch.size();
        const bool to_device = dst_on_device == 1;
        uint4* out = to_device ? reinterpret_cast<uint4*>(dst) : (uint4*)dalloc(cnt * sizeof(pg_fr));
        if (!out) return fail(PG_ERR_OOM, "read buffer");
        if (!to_device) scratch.push_back(out);
        Column sub = *col; sub.inst_off += i0; sub.n = cnt;
        ColReadBody::Args a{view_of(sub), loc_with_tab(loc_of(sub), 0), out, cnt};
        // results of a range call that ran chunk by chunk, read asynchronously and whole: gather and copy each chunk on the copy stream
        // as soon as that chunk's results exist (the kernels of the later chunks are still running on the main stream)
        if (dst_on_device == 2 && sub.inst_off == 0 && cnt == segs[sub.seg].n_inst && be.result_chunks_of(segs[sub.seg].fr)) {
            if (!be.col_read_chunked(a, dst, segs[sub.seg].fr)) return fail(PG_ERR_CUDA, "chunked asynchronous result copy");
            return PG_OK;
        }
        if (!be.template run_simple<ColReadBody>(a, cnt, CLS_OTHER)) return fail(PG_ERR_CUDA, "col_read kernel");
        if (to_device) return PG_OK;
        if (dst_on_device == 2) {                 // pinned host, asynchronous: the staging buffer lives until the next reset
            if (!be.d2h_async(dst, out, cnt * sizeof(pg_fr))) return fail(PG_ERR_CUDA, "asynchronous result copy");
            return PG_OK;
        }
        const int rc = deliver(dst, out, cnt * sizeof(pg_fr), 0);
        release_scratch_from(mark);
        return rc;
    }
    // device side of materialize: rows [row0, row0 + cnt) into column-major device buffers of `stride` rows per column
    int materialize_dev(uint64_t row0, uint64_t cnt, uint64_t stride, unsigned long long* d_idx, uint4* d_val, uint4* d_sel, uint4* d_pi) {
        { const int rcs = sync_dsegs(); if (rcs) return rcs; }
        // per segment: whole instances go through the tiled kernel (wire values + the 5 instance-independent selector columns),
        // the simple body adds w_idx / q_c / PI for them and does everything for the ragged ends of the requested range
        auto simple = [&](uint64_t r0, uint64_t n, uint32_t what) -> bool {
            if (!n || !what) return true;
            MaterializeBody::Args a{d_segs, (uint32_t)dsegs.size(), what, r0, n, stride, r0 - row0, d_idx, d_val, d_sel, d_pi};
            return be.template run_simple<MaterializeBody>(a, n, CLS_OTHER);
        };
        const uint64_t row_end = row0 + cnt;
        for (size_t k = 0; k < segs.size(); k++) {
            const Segment& sg = segs[k];
            const uint64_t nr = sg.t.rows.size();
            if (!nr || !sg.n_inst) continue;
            const uint64_t s_lo = std::max(row0, sg.base_row), s_hi = std::min(row_end, sg.base_row + sg.n_inst * nr);
            if (s_lo >= s_hi) continue;
            const uint64_t iA = (s_lo - sg.base_row + nr - 1) / nr, iB = (s_hi - sg.base_row) / nr;      // whole instances [iA, iB)
            const bool tiled = (d_val || d_sel) && iB > iA && iB - iA >= 32 && nr >= 8;
            if (!tiled) { if (!simple(s_lo, s_hi - s_lo, MAT_ALL)) return fail(PG_ERR_CUDA, "materialize kernel"); continue; }
            const uint64_t t_lo = sg.base_row + iA * nr, t_hi = sg.base_row + iB * nr;
            MatTileArgs ta; memset(&ta, 0, sizeof(ta));
            ta.seg = dsegs[k]; ta.inst0 = iA; ta.n_inst = iB - iA; ta.stride = stride; ta.out_off = t_lo - row0; ta.w_val = d_val; ta.sel = d_sel;
            if (!be.run_mat_tiled(ta)) return fail(PG_ERR_CUDA, "tiled materialize kernel");
            if (!simple(s_lo, t_lo - s_lo, MAT_ALL) || !simple(t_hi, s_hi - t_hi, MAT_ALL) ||
                !simple(t_lo, t_hi - t_lo, MAT_W_IDX | MAT_QC | MAT_PI)) return fail(PG_ERR_CUDA, "materialize kernel");
        }
        return PG_OK;
    }
    int materialize(uint64_t row0, uint64_t cnt, uint64_t* w_idx, pg_fr* w_val, pg_fr* sel, pg_fr* pi, int dst_on_device) {
        if (row0 + cnt > n_rows) return fail(PG_ERR_ARG, "materialize_rows: range");
        if (!cnt) return PG_OK;
        const size_t mark = scratch.size();
        unsigned long long* d_idx = nullptr; uint4 *d_val = nullptr, *d_sel = nullptr, *d_pi = nullptr;
        auto buf = [&](void* user, size_t bytes) -> void* {
            if (!user) return nullptr;
            if (dst_on_device) return user;
            void* p = dalloc(bytes); if (p) scratch.push_back(p); return p;
        };
        d_idx = (unsigned long long*)buf(w_idx, 4 * cnt * sizeof(uint64_t));
        d_val = (uint4*)buf(w_val, 4 * cnt * sizeof(pg_fr));
        d_sel = (uint4*)buf(sel, 6 * cnt * sizeof(pg_fr));
        d_pi = (uint4*)buf(pi, cnt * sizeof(pg_fr));
        if ((w_idx && !d_idx) || (w_val && !d_val) || (sel && !d_sel) || (pi && !d_pi)) return fail(PG_ERR_OOM, "materialize buffers");
        int rc = materialize_dev(row0, cnt, cnt, d_idx, d_val, d_sel, d_pi);
        if (rc) return rc;
        if (dst_on_device) return PG_OK;
        if (w_idx && (rc = deliver(w_idx, d_idx, 4 * cnt * sizeof(uint64_t), 0))) return rc;
        if (w_val && (rc = deliver(w_val, d_val, 4 * cnt * sizeof(pg_fr), 0))) return rc;
        if (sel && (rc = deliver(sel, d_sel, 6 * cnt * sizeof(pg_fr), 0))) return rc;
        if (pi && (rc = deliver(pi, d_pi, cnt * sizeof(pg_fr), 0))) return rc;
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        release_scratch_from(mark);
        return PG_OK;
    }

    // q_arith / q_range columns of rows [row0, row0 + cnt) (either may be null)
    int gate_selectors(uint64_t row0, uint64_t cnt, pg_fr* q_arith, pg_fr* q_range, int dst_on_device) {
        if (row0 + cnt > n_rows) return fail(PG_ERR_ARG, "materialize_gate_selectors: range");
        if (!cnt || (!q_arith && !q_range)) return PG_OK;
        const size_t mark = scratch.size();
        auto buf = [&](void* user) -> uint4* {
            if (!user) return nullptr;
            if (dst_on_device) return (uint4*)user;
            void* p = dalloc(cnt * sizeof(pg_fr)); if (p) scratch.push_back(p); return (uint4*)p;
        };
        uint4 *d_a = buf(q_arith), *d_r = buf(q_range);
        if ((q_arith && !d_a) || (q_range && !d_r)) return fail(PG_ERR_OOM, "gate selector buffers");
        { const int rcs = sync_dsegs(); if (rcs) return rcs; }
        GateSelBody::Args a{d_segs, (uint32_t)dsegs.size(), row0, cnt, d_a, d_r};
        if (!be.template run_simple<GateSelBody>(a, cnt, CLS_OTHER)) return fail(PG_ERR_CUDA, "gate selector kernel");
        if (dst_on_device) return PG_OK;
        int rc;
        if (q_arith && (rc = deliver(q_arith, d_a, cnt * sizeof(pg_fr), 0))) return rc;
        if (q_range && (rc = deliver(q_range, d_r, cnt * sizeof(pg_fr), 0))) return rc;
        release_scratch_from(mark);
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ evaluation domain
    // SURVEY.md 8f.2 (first half): EvaluationDomain::fft / ifft and the wire polynomials of Prover::prove; see ntt.cuh.
    uint4* ntt_tw = nullptr; uint32_t ntt_tw_log_n = 0;
    uint4* fb_table_gen = nullptr;                   // window multiples of the G1 generator (g1_fixed_base_mul_dev), kept for the life of the ctx
    int ntt_twiddles(uint32_t log_n) {
        if (ntt_tw && ntt_tw_log_n == log_n) return PG_OK;
        if (ntt_tw) { be.sync(); dfree(ntt_tw); ntt_tw = nullptr; }
        const uint64_t n_entries = (1ull << (log_n - 1)) + 1;             // w^0 .. w^(n/2) (= -1: the inverse transform's entry for i = 0)
        ntt_tw = (uint4*)dalloc(n_entries * sizeof(pg_fr));
        if (!ntt_tw) return fail(PG_ERR_OOM, "twiddle table");
        ntt_tw_log_n = log_n;
        NttTwiddleBody::Args a;
        a.tw = ntt_tw; a.n_entries = n_entries; a.n = (n_entries + 15) / 16; a.log_n = log_n;
        Fr w = fr_root_of_unity();                                       // EvaluationDomain::new: group_gen
        for (uint32_t i = log_n; i < NTT_TWO_ADICITY; i++) w = fr_sqr(w);
        a.pw2[0] = w;
        for (uint32_t b = 1; b < NTT_TWO_ADICITY; b++) a.pw2[b] = fr_sqr(a.pw2[b - 1]);
        if (!be.template run_simple<NttTwiddleBody>(a, a.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "twiddle kernel");
        return PG_OK;
    }
    // Transform of `data` in place.  Transforms of more than 2^11 points go through a scratch vector of the same size (first
    // pass data -> scratch with the bit reversal folded into its loads, last pass scratch -> data); it is only touched by
    // kernels on the engine's stream, so it goes back to the pool as soon as they are enqueued.
    int ntt_inplace(uint4* data, uint32_t log_n, bool inverse) { return ntt_transform(data, data, log_n, inverse, nullptr); }
    // The same from src to dst (the same buffer, or two that do not overlap).  shift_tab != nullptr (forward only): the coset
    // transform of EvaluationDomain::coset_fft, source element m multiplied by h^m from pow_table_host's two-level table of h.
    int ntt_transform(const uint4* src, uint4* data, uint32_t log_n, bool inverse, const uint4* shift_tab) {
        if (shift_tab && inverse) return fail(PG_ERR_ARG, "ntt: a coset shift applies to the forward transform only");
        if (log_n == 0)                                                  // one element: the transform is the identity (h^0 = 1)
            return src == data || be.d2d(data, src, sizeof(pg_fr)) ? PG_OK : fail(PG_ERR_CUDA, "device copy");
        int rc = ntt_twiddles(log_n);
        if (rc) return rc;
        const uint64_t n = 1ull << log_n;
        Fr factor = fr_one();
        if (inverse) { Fr raw = fr_zero(); raw.v[0] = (uint32_t)n; raw.v[1] = (uint32_t)(n >> 32); factor = fr_inv_fermat(fr_to_mont(raw)); }   // size_inv
        const NttPlan plan = ntt_plan(log_n);
        uint4* work = nullptr;
        if (plan.n_pass > 1 && !(work = (uint4*)dalloc(sizeof(pg_fr) << log_n))) return fail(PG_ERR_OOM, "NTT scratch vector");
        for (uint32_t p = 0; p < plan.n_pass; p++) {
            NttPassArgs a; memset(&a, 0, sizeof(a));
            const bool first = p == 0, last = p + 1 == plan.n_pass;
            a.src = first ? src : work;                                  // first pass: gather through the bit reversal, scale / shift
            a.dst = last ? data : work;                                  // last pass: back to the caller's buffer
            a.tw = ntt_tw; a.log_n = log_n; a.t0 = plan.t0[p]; a.s = plan.s[p]; a.log_c = plan.log_c[p];
            a.inverse = inverse ? 1 : 0; a.bitrev = first ? 1 : 0; a.scale = first && inverse ? 1 : 0; a.factor = factor;
            if (first && shift_tab) { a.shift = 1; a.shift_tab = shift_tab; a.shift_log_lo = pow_table_log_lo(log_n); }
            if (!be.run_ntt_pass(a, n >> (plan.s[p] + plan.log_c[p]))) { dfree(work); return fail(PG_ERR_CUDA, "NTT pass kernel"); }
        }
        dfree(work);
        return PG_OK;
    }
    int fft(uint32_t log_n, int inverse, const pg_fr* src, pg_fr* dst, int on_device) {
        if (log_n > NTT_TWO_ADICITY || !src || !dst) return fail(PG_ERR_ARG, "fft: domain larger than 2^32 or null buffer");
        const uint64_t n = 1ull << log_n; const size_t bytes = n * sizeof(pg_fr);
        const size_t mark = scratch.size();
        uint4* buf;
        if (on_device) { buf = reinterpret_cast<uint4*>(dst); if (src != dst && !be.d2d(dst, src, bytes)) return fail(PG_ERR_CUDA, "device copy"); }
        else {
            buf = (uint4*)dalloc(bytes);
            if (!buf) return fail(PG_ERR_OOM, "fft buffer");
            scratch.push_back(buf);
            if (!be.h2d(buf, src, bytes)) return fail(PG_ERR_CUDA, "input copy");
        }
        int rc = ntt_inplace(buf, log_n, inverse != 0);
        if (rc || on_device) return rc;
        rc = deliver(dst, buf, bytes, 0);
        release_scratch_from(mark);
        return rc;
    }
    // to_scalars(w_l..w_4) of the composer's rows, padded with zeros up to the domain size n: 4 columns of n scalars in buf
    int wire_values(uint64_t n, uint4* buf) {
        int rc = materialize_dev(0, n_rows, n, nullptr, buf, nullptr, nullptr);
        if (rc) return rc;
        for (int w = 0; w < 4 && n > n_rows; w++) {
            NttZeroBody::Args z{buf + 2 * (uint64_t)w * n, n_rows, n - n_rows};
            if (!be.template run_simple<NttZeroBody>(z, z.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "padding kernel");
        }
        return PG_OK;
    }
    // dst: 4 columns (w_l, w_r, w_o, w_4) of 2^log_n coefficients each
    int wire_polynomials(uint32_t log_n, pg_fr* dst, int dst_on_device) {
        if (log_n > NTT_TWO_ADICITY || (1ull << log_n) < n_rows || !dst) return fail(PG_ERR_ARG, "wire_polynomials: domain smaller than the circuit, larger than 2^32, or null buffer");
        const uint64_t n = 1ull << log_n; const size_t bytes = 4 * n * sizeof(pg_fr);
        const size_t mark = scratch.size();
        uint4* buf = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { buf = (uint4*)dalloc(bytes); if (!buf) return fail(PG_ERR_OOM, "wire polynomial buffer"); scratch.push_back(buf); }
        int rc = wire_values(n, buf);
        if (rc) return rc;
        for (int w = 0; w < 4; w++)
            if ((rc = ntt_inplace(buf + 2 * (uint64_t)w * n, log_n, true))) return rc;   // domain.ifft
        if (dst_on_device) return PG_OK;
        rc = deliver(dst, buf, bytes, 0);
        release_scratch_from(mark);
        return rc;
    }

    // ------------------------------------------------------------------------------------------------ permutation map
    // sigma[w][t] = cycle successor (row*4 + wire) of wire position (row0 + t, w); see PermBody.
    int permutation(uint64_t row0, uint64_t cnt, uint64_t* sigma, int dst_on_device) {
        if (row0 + cnt > n_rows || (cnt && !sigma)) return fail(PG_ERR_ARG, "permutation: range");
        if (!cnt) return PG_OK;
        const size_t mark = scratch.size();
        { const int rcs = sync_dsegs(); if (rcs) return rcs; }
        const size_t S = segs.size();
        std::vector<PermSeg> ps(S);
        std::vector<PermCons> cons;
        std::vector<std::vector<uint32_t>> next_in(S), ref(S), first_local(S), cons_head(S);
        for (size_t k = 0; k < S; k++) cons_head[k].assign(segs[k].t.n_vars, 0);
        uint32_t prev_zero_seg = PERM_NONE, first_zero_seg = PERM_NONE;
        for (size_t k = 0; k < S; k++) {
            const Segment& sg = segs[k]; const Template& T = sg.t;
            PermSeg& p = ps[k]; memset(&p, 0, sizeof(p));
            p.base_row = sg.base_row; p.n_inst = sg.n_inst; p.n_rows = (uint32_t)T.rows.size();
            p.first_zero = PERM_NONE; p.next_zero_seg = PERM_NONE;
            for (int e = 0; e < 4; e++) p.first_op[e] = PERM_NONE;
            // canonical operand index: operands bound to the same column are one variable
            uint32_t canon[4] = {0, 1, 2, 3};
            for (size_t e = 0; e < sg.operands.size(); e++)
                for (size_t f = 0; f < e; f++)
                    if (sg.operands[f].seg == sg.operands[e].seg && sg.operands[f].local == sg.operands[e].local && sg.operands[f].inst_off == sg.operands[e].inst_off) { canon[e] = (uint32_t)f; break; }
            const size_t NW = T.rows.size() * 4;
            ref[k].assign(NW, 0); next_in[k].assign(NW, PERM_NONE); first_local[k].assign(T.n_vars, PERM_NONE);
            std::vector<uint32_t> last_local(T.n_vars, PERM_NONE); uint32_t last_op[4] = {PERM_NONE, PERM_NONE, PERM_NONE, PERM_NONE}, last_zero = PERM_NONE;
            for (size_t r = 0; r < T.rows.size(); r++)
                for (uint32_t ow = 0; ow < 4; ow++) {
                    // order in which the row's wires entered perm.variable_map (templates.hpp PERM_*): a, b, c, d for the arithmetic
                    // gate methods; fourth, output, right, left for range_gate, whose closing gate enters its fourth wire only
                    const uint8_t pm = T.rows[r].perm;
                    const uint32_t w = pm == PERM_LROF ? ow : 3u - ow;
                    const WireRef& wr = T.rows[r].w[w]; const uint32_t pos = (uint32_t)(r * 4 + w);
                    if (pm == PERM_F_ONLY && w != 3u) { ref[k][pos] = PERM_REF_UNMAPPED; continue; }
                    uint32_t* last; uint32_t* first;
                    if (wr.src == 0 || (T.kind == G_PREAMBLE && wr.src == 1 && wr.idx == 0)) { ref[k][pos] = 0; last = &last_zero; first = &p.first_zero; }
                    else if (wr.src == 1) { ref[k][pos] = 1 + wr.idx; last = &last_local[wr.idx]; first = &first_local[k][wr.idx]; }
                    else { const uint32_t e = canon[wr.src - 2]; ref[k][pos] = 0x80000000u | e; last = &last_op[e]; first = &p.first_op[e]; }
                    if (*last != PERM_NONE) next_in[k][*last] = pos; else *first = pos;
                    *last = pos;
                }
            if (sg.n_inst && p.first_zero != PERM_NONE) {
                if (prev_zero_seg != PERM_NONE) ps[prev_zero_seg].next_zero_seg = (uint32_t)k; else first_zero_seg = (uint32_t)k;
                prev_zero_seg = (uint32_t)k;
            }
            // register this segment as a consumer of its operand columns (call order = list order)
            for (size_t e = 0; e < sg.operands.size(); e++) {
                p.op_src_seg[e] = sg.operands[e].seg; p.op_src_local[e] = sg.operands[e].local; p.op_inst_off[e] = sg.operands[e].inst_off;
                if (canon[e] != e) { p.op_cons_idx[e] = p.op_cons_idx[canon[e]]; continue; }
                if (p.first_op[e] == PERM_NONE || !sg.n_inst) { p.op_cons_idx[e] = 0; continue; }     // operand never appears on a wire / no instances
                PermCons c; memset(&c, 0, sizeof(c));
                c.seg = (uint32_t)k; c.op = (uint32_t)e; c.inst_off = sg.operands[e].inst_off; c.n = sg.n_inst; c.next = 0;
                cons.push_back(c);
                const uint32_t me = (uint32_t)cons.size();                                              // index + 1
                uint32_t* head = &cons_head[sg.operands[e].seg][sg.operands[e].local];
                if (!*head) *head = me;
                else { uint32_t t = *head; while (cons[t - 1].next) t = cons[t - 1].next; cons[t - 1].next = me; }
                p.op_cons_idx[e] = me - 1;
            }
        }
        // upload
        auto up = [&](const void* src, size_t bytes) -> void* {
            void* d = dalloc(bytes ? bytes : 16); if (!d) return nullptr;
            scratch.push_back(d);
            if (bytes && !be.h2d(d, src, bytes)) return nullptr;
            return d;
        };
        for (size_t k = 0; k < S; k++) {
            ps[k].next_in_inst = (const uint32_t*)up(next_in[k].data(), next_in[k].size() * 4);
            ps[k].ref = (const uint32_t*)up(ref[k].data(), ref[k].size() * 4);
            ps[k].first_local = (const uint32_t*)up(first_local[k].data(), first_local[k].size() * 4);
            ps[k].cons_head = (const uint32_t*)up(cons_head[k].data(), cons_head[k].size() * 4);
            if (!ps[k].next_in_inst || !ps[k].ref || !ps[k].first_local || !ps[k].cons_head) return fail(PG_ERR_OOM, "permutation tables");
        }
        if (cons.empty()) { PermCons c; memset(&c, 0, sizeof(c)); cons.push_back(c); }
        const PermSeg* d_ps = (const PermSeg*)up(ps.data(), ps.size() * sizeof(PermSeg));
        const PermCons* d_cons = (const PermCons*)up(cons.data(), cons.size() * sizeof(PermCons));
        if (!d_ps || !d_cons) return fail(PG_ERR_OOM, "permutation tables");
        unsigned long long* out = dst_on_device ? reinterpret_cast<unsigned long long*>(sigma) : (unsigned long long*)dalloc(4 * cnt * sizeof(uint64_t));
        if (!out) return fail(PG_ERR_OOM, "permutation buffer");
        if (!dst_on_device) scratch.push_back(out);
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");            // the host vectors above are the sources of the copies
        PermBody::Args a{d_segs, d_ps, d_cons, (uint32_t)dsegs.size(), first_zero_seg, row0, cnt, out};
        if (!be.template run_simple<PermBody>(a, cnt, CLS_OTHER)) return fail(PG_ERR_CUDA, "permutation kernel");
        if (dst_on_device) return PG_OK;                             // tables stay parked until the next composer reset
        const int rc = deliver(sigma, out, 4 * cnt * sizeof(uint64_t), 0);
        release_scratch_from(mark);
        return rc;
    }

    // ------------------------------------------------------------------------------------------------ permutation argument
    // Preprocessing's sigma polynomials and prover round 2's z(X) [DEP dusk-plonk 0.8 permutation.rs]; bodies.cuh PermSigmaBody /
    // PermRatioHook, scan.cuh.  Coset constants k = (1, K1, K2, K3) = (1, 7, 13, 17) (permutation/constants.rs, recalled).
    static Fr perm_coset(uint32_t w) { static const uint32_t k[4] = {1, 7, 13, 17}; Fr raw = fr_zero(); raw.v[0] = k[w]; return fr_to_mont(raw); }
    int perm_domain(const char* who, uint32_t log_n, uint64_t rows, int form) {
        if (log_n > NTT_TWO_ADICITY || (1ull << log_n) < rows) return fail(PG_ERR_ARG, std::string(who) + ": domain smaller than the circuit or larger than 2^32");
        if (form != PG_FORM_EVALUATIONS && form != PG_FORM_COEFFICIENTS) return fail(PG_ERR_ARG, std::string(who) + ": form must be PG_FORM_EVALUATIONS or PG_FORM_COEFFICIENTS");
        return PG_OK;
    }
    // a sharded composer holds one rank's rows: the grand product would need the other ranks' carries (not built)
    int perm_unsharded(const char* who) {
        return be.comm_world() > 1 ? fail(PG_ERR_STATE, std::string(who) + ": the composer is sharded over a communicator; a sharded permutation argument is not built") : PG_OK;
    }
    // the composer's copy-constraint map (rows 0 .. n_rows) on the device, parked in `scratch`
    unsigned long long* perm_map_dev(int* rc) {
        unsigned long long* d = (unsigned long long*)dalloc(4 * (n_rows ? n_rows : 1) * sizeof(uint64_t));
        if (!d) { *rc = fail(PG_ERR_OOM, "permutation buffer"); return nullptr; }
        scratch.push_back(d);
        *rc = permutation(0, n_rows, reinterpret_cast<uint64_t*>(d), 1);
        return *rc ? nullptr : d;
    }
    int sigma_polynomials(uint32_t log_n, int form, pg_fr* dst, int dst_on_device) {
        int rc;
        if ((rc = perm_unsharded("sigma_polynomials")) || (rc = perm_domain("sigma_polynomials", log_n, n_rows, form))) return rc;
        if (!dst) return fail(PG_ERR_ARG, "sigma_polynomials: null buffer");
        const uint64_t n = 1ull << log_n; const size_t bytes = 4 * n * sizeof(pg_fr);
        const size_t mark = scratch.size();
        uint4* buf = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { buf = (uint4*)dalloc(bytes); if (!buf) return fail(PG_ERR_OOM, "sigma buffer"); scratch.push_back(buf); }
        const unsigned long long* sig = perm_map_dev(&rc); if (!sig) return rc;
        if (log_n && (rc = ntt_twiddles(log_n))) return rc;
        PermSigmaBody::Args a; memset(&a, 0, sizeof(a));
        a.sigma = sig; a.n_sig = n_rows; a.n = n; a.tw = log_n ? ntt_tw : nullptr; a.log_n = log_n; a.out = buf;
        for (uint32_t w = 0; w < 4; w++) a.k[w] = perm_coset(w);
        if (!be.template run_simple<PermSigmaBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "sigma kernel");   // compute_permutation_lagrange
        for (int w = 0; w < 4 && form == PG_FORM_COEFFICIENTS; w++)
            if ((rc = ntt_inplace(buf + 2 * (uint64_t)w * n, log_n, true))) return rc;      // compute_sigma_polynomials: domain.ifft
        if (!dst_on_device) { if ((rc = deliver(dst, buf, bytes, 0))) return rc; }
        else if (!be.sync()) return fail(PG_ERR_CUDA, "sync");                            // the map's tables go back to the pool
        release_scratch_from(mark);
        return PG_OK;
    }
    int permutation_z(uint32_t log_n, const pg_fr* beta, const pg_fr* gamma, int form, pg_fr* dst, int dst_on_device, pg_fr* closing) {
        int rc;
        if ((rc = perm_unsharded("permutation_z")) || (rc = perm_domain("permutation_z", log_n, n_rows, form))) return rc;
        if ((rc = perm_scalars("permutation_z", beta, gamma, dst))) return rc;
        const uint64_t n = 1ull << log_n;
        const size_t mark = scratch.size();
        uint4* w = (uint4*)dalloc(4 * n * sizeof(pg_fr)); if (!w) return fail(PG_ERR_OOM, "wire value buffer");
        scratch.push_back(w);
        if ((rc = wire_values(n, w))) return rc;
        const unsigned long long* sig = perm_map_dev(&rc); if (!sig) return rc;
        return permutation_z_dev(log_n, w, sig, n_rows, false, beta, gamma, form, dst, dst_on_device, closing, mark);
    }
    // the same over caller-supplied rows: w_val 4 x n_in, sigma 4 x n_in (row*4 + wire), rows n_in .. 2^log_n padding
    int permutation_z_rows(uint32_t log_n, uint64_t n_in, const pg_fr* w_val, const uint64_t* sigma, int on_device, const pg_fr* beta,
                           const pg_fr* gamma, int form, pg_fr* dst, int dst_on_device, pg_fr* closing) {
        int rc;
        if ((rc = perm_domain("permutation_z_rows", log_n, n_in, form))) return rc;
        if ((rc = perm_scalars("permutation_z_rows", beta, gamma, dst))) return rc;
        if (n_in && (!w_val || !sigma)) return fail(PG_ERR_ARG, "permutation_z_rows: null rows");
        const uint64_t n = 1ull << log_n;
        const size_t mark = scratch.size();
        uint4* w = (uint4*)dalloc(4 * n * sizeof(pg_fr)); if (!w) return fail(PG_ERR_OOM, "wire value buffer");
        scratch.push_back(w);
        for (uint64_t c = 0; c < 4; c++) {                                                  // stride n_in -> stride n, zero padding
            uint4* col = w + 2 * c * n;
            if (n_in && !(on_device ? be.d2d(col, w_val + c * n_in, n_in * sizeof(pg_fr)) : be.h2d(col, w_val + c * n_in, n_in * sizeof(pg_fr))))
                return fail(PG_ERR_CUDA, "row copy");
            NttZeroBody::Args z{col, n_in, n - n_in};
            if (n > n_in && !be.template run_simple<NttZeroBody>(z, z.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "padding kernel");
        }
        const unsigned long long* sig = reinterpret_cast<const unsigned long long*>(sigma);
        if (!on_device && n_in) {
            void* d = dalloc(4 * n_in * sizeof(uint64_t)); if (!d) return fail(PG_ERR_OOM, "sigma staging buffer");
            scratch.push_back(d);
            if (!be.h2d(d, sigma, 4 * n_in * sizeof(uint64_t))) return fail(PG_ERR_CUDA, "sigma copy");
            sig = (const unsigned long long*)d;
        }
        return permutation_z_dev(log_n, w, sig, n_in, true, beta, gamma, form, dst, dst_on_device, closing, mark);
    }
    int perm_scalars(const char* who, const pg_fr* beta, const pg_fr* gamma, const pg_fr* dst) {
        if (!beta || !gamma || !dst) return fail(PG_ERR_ARG, std::string(who) + ": null argument");
        if (!host_reduced(*beta) || !host_reduced(*gamma)) return fail(PG_ERR_ARG, std::string(who) + ": beta / gamma not fully reduced (>= q)");
        return PG_OK;
    }
    // exclusive prefix product of n scalars, *total = their product: the backend's device-wide scan (CudaBackend::run_fr_scan, scan.cuh;
    // engine.cu asserts that it has one), else FrScanSerialBody as one unit of work
    bool fr_scan(const uint4* in, uint4* out, uint64_t n, uint4* total, uint4* scratch) {
        if constexpr (has_fr_scan<BE>::value) return be.run_fr_scan(in, out, n, total, scratch);
        else { (void)scratch; const FrScanSerialBody::Args a{in, out, n, total}; return be.template run_simple<FrScanSerialBody>(a, 1, CLS_OTHER); }
    }
    // ratios fused into the batch inversion (k_batch_inv<PermRatioHook>), exclusive prefix product (z and the closing product),
    // optionally domain.ifft; synchronises to read the zero-denominator / bad-row counters
    int permutation_z_dev(uint32_t log_n, const uint4* w, const unsigned long long* sig, uint64_t n_sig, bool check_rows, const pg_fr* beta,
                          const pg_fr* gamma, int form, pg_fr* dst, int dst_on_device, pg_fr* closing, size_t mark) {
        const uint64_t n = 1ull << log_n;
        int rc;
        uint4* z = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { z = (uint4*)dalloc(n * sizeof(pg_fr)); if (!z) return fail(PG_ERR_OOM, "z buffer"); scratch.push_back(z); }
        uint4* tab = (uint4*)dalloc(2 * n * sizeof(pg_fr)); if (!tab) return fail(PG_ERR_OOM, "inversion table");
        scratch.push_back(tab);
        uint4* tot = (uint4*)dalloc((1 + fr_scan_scratch(n)) * sizeof(pg_fr)); if (!tot) return fail(PG_ERR_OOM, "scan scratch");
        scratch.push_back(tot);
        if (log_n && (rc = ntt_twiddles(log_n))) return rc;
        if ((rc = reset_counters())) return rc;
        const Fr b = fr_from_pg(*beta);
        PermRatioHook::Args h; memset(&h, 0, sizeof(h));
        h.w = w; h.n = n; h.sigma = sig; h.n_sig = n_sig; h.tw = log_n ? ntt_tw : nullptr; h.log_n = log_n;
        for (uint32_t k = 0; k < 4; k++) h.bk[k] = fr_mul(b, perm_coset(k));
        h.gamma = fr_from_pg(*gamma); h.den = tab; h.ratio = z; h.counters = d_counters; h.check = check_rows ? 1 : 0;
        BatchInvArgs inv; memset(&inv, 0, sizeof(inv));
        inv.fr = tab; inv.stride = n; inv.n = n; inv.n_pairs = 1; inv.in_slot[0] = 0; inv.out_slot[0] = 1;
        if (!be.template run_batch_inv_fused<PermRatioHook>(inv, h, CLS_OTHER)) return fail(PG_ERR_CUDA, "permutation ratio kernel");
        if (!fr_scan(z, z, n, tot, tot + 2)) return fail(PG_ERR_CUDA, "grand-product scan");
        if (form == PG_FORM_COEFFICIENTS && (rc = ntt_inplace(z, log_n, true))) return rc;      // compute_permutation_poly: domain.ifft(z)
        unsigned long long c[CNT_WORDS];
        if ((rc = read_counters(c))) return rc;
        if (c[CNT_UNSAT]) {
            char msg[200];
            snprintf(msg, sizeof(msg), "permutation_z_rows: %llu row(s) with a sigma entry >= 4 * 2^%u or an unreduced wire value, first at row %llu",
                     c[CNT_UNSAT], log_n, c[CNT_FIRST_BAD]);
            return fail(PG_ERR_ARG, msg);
        }
        if (c[CNT_N_ERR]) {
            char msg[200];
            snprintf(msg, sizeof(msg), "permutation_z: %llu zero denominator(s) v + beta*sigma + gamma, first at row %llu", c[CNT_N_ERR], c[CNT_FIRST_ERR]);
            return fail(PG_ERR_ARG, msg);
        }
        if (closing && (rc = deliver(closing, tot, sizeof(pg_fr), 0))) return rc;
        if (!dst_on_device && (rc = deliver(dst, z, n * sizeof(pg_fr), 0))) return rc;
        release_scratch_from(mark);
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ quotient polynomial
    // Preprocessing's selector and public-input polynomials and prover round 3's t(X) [DEP dusk-plonk 0.8 quotient_poly.rs, recalled];
    // bodies.cuh QuotientBody / QuotientSplitBody, ntt.cuh k_ntt_coset_pass.
    // the eight selector columns q_m q_l q_r q_o q_4 q_c q_arith q_range (padding rows 0) in 8 columns of 2^log_n, optionally ifft'd
    int selector_polynomials(uint32_t log_n, int form, pg_fr* dst, int dst_on_device) {
        int rc;
        if ((rc = perm_unsharded("selector_polynomials")) || (rc = perm_domain("selector_polynomials", log_n, n_rows, form))) return rc;
        if (!dst) return fail(PG_ERR_ARG, "selector_polynomials: null buffer");
        const uint64_t n = 1ull << log_n; const size_t bytes = 8 * n * sizeof(pg_fr);
        const size_t mark = scratch.size();
        uint4* buf = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { buf = (uint4*)dalloc(bytes); if (!buf) return fail(PG_ERR_OOM, "selector buffer"); scratch.push_back(buf); }
        if ((rc = materialize_dev(0, n_rows, n, nullptr, nullptr, buf, nullptr))) return rc;          // q_m .. q_c
        GateSelBody::Args g{d_segs, (uint32_t)dsegs.size(), 0, n_rows, buf + 2 * 6 * n, buf + 2 * 7 * n};  // q_arith, q_range
        if (!be.template run_simple<GateSelBody>(g, n_rows, CLS_OTHER)) return fail(PG_ERR_CUDA, "gate selector kernel");
        for (uint64_t c = 0; c < 8; c++) {
            uint4* col = buf + 2 * c * n;
            NttZeroBody::Args z{col, n_rows, n - n_rows};
            if (n > n_rows && !be.template run_simple<NttZeroBody>(z, z.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "padding kernel");
            if (form == PG_FORM_COEFFICIENTS && (rc = ntt_inplace(col, log_n, true))) return rc;
        }
        if (dst_on_device) return PG_OK;
        rc = deliver(dst, buf, bytes, 0);
        release_scratch_from(mark);
        return rc;
    }
    // construct_dense_pi_vec padded with zeros to 2^log_n, optionally ifft'd
    int public_input_polynomial(uint32_t log_n, int form, pg_fr* dst, int dst_on_device) {
        int rc;
        if ((rc = perm_unsharded("public_input_polynomial")) || (rc = perm_domain("public_input_polynomial", log_n, n_rows, form))) return rc;
        if (!dst) return fail(PG_ERR_ARG, "public_input_polynomial: null buffer");
        const uint64_t n = 1ull << log_n; const size_t bytes = n * sizeof(pg_fr);
        const size_t mark = scratch.size();
        uint4* buf = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { buf = (uint4*)dalloc(bytes); if (!buf) return fail(PG_ERR_OOM, "public input buffer"); scratch.push_back(buf); }
        if ((rc = materialize_dev(0, n_rows, n, nullptr, nullptr, nullptr, buf))) return rc;
        NttZeroBody::Args z{buf, n_rows, n - n_rows};
        if (n > n_rows && !be.template run_simple<NttZeroBody>(z, z.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "padding kernel");
        if (form == PG_FORM_COEFFICIENTS && (rc = ntt_inplace(buf, log_n, true))) return rc;
        if (dst_on_device) return PG_OK;
        rc = deliver(dst, buf, bytes, 0);
        release_scratch_from(mark);
        return rc;
    }
    // The coefficient vectors of rounds 3 to 5, 2^log_n each in QV_* order: wires, z (for beta, gamma), sigma, the eight selectors and,
    // with_pi, PI (coef holds QV_COEF vectors then, else QV_PI)
    int component_polynomials(uint32_t log_n, const pg_fr* beta, const pg_fr* gamma, bool with_pi, uint4* coef) {
        const uint64_t n = 1ull << log_n;
        auto col = [n, coef](uint32_t v) { return (pg_fr*)(coef + 2 * (uint64_t)v * n); };
        int rc;
        if ((rc = wire_polynomials(log_n, col(QV_W), 1))) return rc;
        if ((rc = permutation_z(log_n, beta, gamma, PG_FORM_COEFFICIENTS, col(QV_Z), 1, nullptr))) return rc;
        if ((rc = sigma_polynomials(log_n, PG_FORM_COEFFICIENTS, col(QV_S), 1))) return rc;
        if ((rc = selector_polynomials(log_n, PG_FORM_COEFFICIENTS, col(QV_QM), 1))) return rc;
        if (with_pi && (rc = public_input_polynomial(log_n, PG_FORM_COEFFICIENTS, col(QV_PI), 1))) return rc;
        return PG_OK;
    }
    static Fr fr_small(uint64_t v) { Fr raw = fr_zero(); raw.v[0] = (uint32_t)v; raw.v[1] = (uint32_t)(v >> 32); return fr_to_mont(raw); }
    static Fr fr_pow2k(Fr x, uint32_t k) { for (uint32_t i = 0; i < k; i++) x = fr_sqr(x); return x; }     // x^(2^k)
    // Round 3: t_1 .. t_4 (4 columns of N = 2^log_n coefficients).  Coefficient vectors of the wires, z, sigma, the selectors and PI
    // (QV_* order), then per sub-coset j: coset FFTs of each (shift h_j = g zeta^j) and of alpha^2 / N (= alpha^2 L_1), the
    // numerator / Z_H pointwise; then an inverse size-N transform per sub-coset and the split.
    int quotient(uint32_t log_n, const pg_fr* alpha, const pg_fr* beta, const pg_fr* gamma, const pg_fr* rho, pg_fr* dst, int dst_on_device) {
        int rc;
        if ((rc = perm_unsharded("quotient"))) return rc;
        if (log_n > NTT_TWO_ADICITY - 2 || (1ull << log_n) < n_rows)
            return fail(PG_ERR_ARG, "quotient: domain smaller than the circuit, or larger than 2^30 (the 4N coset needs 2-adicity log_n + 2 <= 32)");
        if (!alpha || !beta || !gamma || !rho || !dst) return fail(PG_ERR_ARG, "quotient: null argument");
        if (!host_reduced(*alpha) || !host_reduced(*beta) || !host_reduced(*gamma) || !host_reduced(*rho))
            return fail(PG_ERR_ARG, "quotient: alpha / beta / gamma / range_challenge not fully reduced (>= q)");
        // polynomials that are zero by the composer's structure: no row template has a public input / a range-widget row
        bool has_pi = false, has_range = false;
        for (const Segment& s : segs) {
            if (!s.n_inst) continue;
            for (const RowT& r : s.t.rows) { has_range = has_range || r.gate == GATE_RANGE; has_pi = has_pi || r.pi_param >= 0 || r.pi_sel != POOL_ZERO; }
        }
        const uint64_t n = 1ull << log_n;
        const size_t mark = scratch.size();
        auto col = [n](uint4* base, uint32_t v) { return base + 2 * (uint64_t)v * n; };
        uint4* coef = (uint4*)dalloc(QV_COEF * n * sizeof(pg_fr)); if (!coef) return fail(PG_ERR_OOM, "quotient coefficient vectors");
        scratch.push_back(coef);
        if ((rc = component_polynomials(log_n, beta, gamma, has_pi, coef))) return rc;
        uint4* ev = (uint4*)dalloc(QV_EV * n * sizeof(pg_fr)); if (!ev) return fail(PG_ERR_OOM, "quotient evaluation vectors");
        scratch.push_back(ev);
        uint4* out = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { out = (uint4*)dalloc(4 * n * sizeof(pg_fr)); if (!out) return fail(PG_ERR_OOM, "quotient buffer"); scratch.push_back(out); }
        // constants: zeta generates the 4N-th roots (zeta^4 = w), iota = zeta^N, g = 7 (dusk-bls12_381 GENERATOR), h_j = g zeta^j
        const Fr zeta = fr_pow2k(fr_root_of_unity(), NTT_TWO_ADICITY - log_n - 2), iota = fr_pow2k(zeta, log_n);
        const Fr g = fr_small(7), g_n = fr_pow2k(g, log_n), n_inv = fr_inv_fermat(fr_small(n));
        const Fr al = fr_from_pg(*alpha), be_ = fr_from_pg(*beta), ga = fr_from_pg(*gamma), rh = fr_from_pg(*rho);
        Fr h[4], iota_j[4];
        h[0] = g; iota_j[0] = fr_one();
        for (int j = 1; j < 4; j++) { h[j] = fr_mul(h[j - 1], zeta); iota_j[j] = fr_mul(iota_j[j - 1], iota); }
        // two-level power tables of h_j (coset FFTs) and h_j^-1 (split): table j at tabs + 2 * j * entries, j = 0..7
        const uint64_t entries = pow_table_entries(log_n);
        std::vector<Fr> host_tabs(8 * entries);
        for (int j = 0; j < 4; j++) {
            pow_table_host(h[j], log_n, host_tabs.data() + j * entries);
            pow_table_host(fr_inv_fermat(h[j]), log_n, host_tabs.data() + (4 + j) * entries);
        }
        uint4* tabs = (uint4*)dalloc(host_tabs.size() * sizeof(pg_fr)); if (!tabs) return fail(PG_ERR_OOM, "coset power tables");
        scratch.push_back(tabs);
        if (!be.h2d(tabs, host_tabs.data(), host_tabs.size() * sizeof(pg_fr))) return fail(PG_ERR_CUDA, "coset power table copy");
        if ((rc = ntt_twiddles(log_n))) return rc;
        QuotientBody::Args q; memset(&q, 0, sizeof(q));
        q.ev = ev; q.n = n; q.tw = ntt_tw; q.log_n = log_n; q.has_pi = has_pi; q.has_range = has_range;
        q.beta = be_; q.gamma = ga; q.alpha = al; q.rho = rh; q.kappa = fr_sqr(rh); q.two = fr_small(2); q.three = fr_small(3);
        const Fr l1_coef = fr_mul(fr_sqr(al), n_inv);                         // alpha^2 L_1(X) = alpha^2 / N * sum_{i<N} X^i
        for (uint32_t j = 0; j < 4; j++) {
            const uint4* tab = tabs + 2 * (uint64_t)j * entries;
            for (uint32_t v = 0; v < QV_COEF; v++) {
                if ((v == QV_PI && !has_pi) || (v == QV_QRANGE && !has_range)) continue;
                if ((rc = ntt_transform(col(coef, v), col(ev, v), log_n, false, tab))) return rc;
            }
            FillBody::Args f{col(ev, QV_L1), l1_coef, n};
            if (!be.template run_simple<FillBody>(f, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "fill kernel");
            if ((rc = ntt_transform(col(ev, QV_L1), col(ev, QV_L1), log_n, false, tab))) return rc;
            for (uint32_t w = 0; w < 4; w++) q.bkh[w] = fr_mul(fr_mul(be_, perm_coset(w)), h[j]);
            q.zh_inv = fr_inv_fermat(fr_sub(fr_mul(g_n, iota_j[j]), fr_one()));    // x^N - 1 = g^N iota^j - 1 on all of sub-coset j
            q.out = col(out, j);
            if (!be.template run_simple<QuotientBody>(q, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "quotient kernel");
        }
        for (uint32_t j = 0; j < 4; j++)
            if ((rc = ntt_inplace(col(out, j), log_n, true))) return rc;
        QuotientSplitBody::Args s; memset(&s, 0, sizeof(s));
        s.t = out; s.n = n; s.log_lo = pow_table_log_lo(log_n); s.iota_inv = fr_inv_fermat(iota);
        const Fr g_n_inv = fr_inv_fermat(g_n);
        s.scale[0] = fr_inv_fermat(fr_small(4));                                          // (1/4) g^-rN
        for (int r = 1; r < 4; r++) s.scale[r] = fr_mul(s.scale[r - 1], g_n_inv);
        for (int j = 0; j < 4; j++) s.inv_tab[j] = tabs + 2 * (uint64_t)(4 + j) * entries;
        if (!be.template run_simple<QuotientSplitBody>(s, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "quotient split kernel");
        if (!dst_on_device) { if ((rc = deliver(dst, out, 4 * n * sizeof(pg_fr), 0))) return rc; }
        else if (!be.sync()) return fail(PG_ERR_CUDA, "sync");                            // the coefficient and evaluation vectors go back to the pool
        release_scratch_from(mark);
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ openings (rounds 4 and 5)
    // [DEP dusk-plonk 0.8 Prover::prove, linearisation_poly::compute, compute_quotient_opening_poly / compute_aggregate_witness,
    // Polynomial::ruffini, recalled]; bodies.cuh OpenEvalBody / OpenSumBody / OpenCombineBody, scan.cuh (Ruffini division).
    // out[i] = s_(i+1) of s_i = f_i + p s_(i+1) and *rem = f(p) (in place allowed): the backend's device-wide scan (CudaBackend::
    // run_fr_ruffini; engine.cu asserts that it has one), else FrRuffiniSerialBody as one unit of work
    int fr_ruffini(const uint4* in, uint4* out, uint64_t n, const Fr& p, uint4* rem) {
        if constexpr (has_fr_ruffini<BE>::value) {
            const uint32_t levels = fr_ruffini_levels(n);
            std::vector<Fr> host(levels * RUF_TAB);
            Fr x = p;                                                       // level l: powers of p^(SCAN_TILE^l)
            for (uint32_t l = 0; l < levels; l++) {
                Fr y = fr_one();
                for (uint64_t k = 0; k < RUF_TAB; k++) { host[l * RUF_TAB + k] = y; y = fr_mul(y, x); }
                x = host[l * RUF_TAB + SCAN_TILE];
            }
            uint4* pw = (uint4*)dalloc((host.size() + fr_scan_scratch(n)) * sizeof(pg_fr)); if (!pw) return fail(PG_ERR_OOM, "ruffini tables");
            scratch.push_back(pw);
            if (!be.h2d(pw, host.data(), host.size() * sizeof(pg_fr))) return fail(PG_ERR_CUDA, "ruffini table copy");
            if (!be.run_fr_ruffini(in, out, n, pw, rem, pw + 2 * host.size())) return fail(PG_ERR_CUDA, "ruffini scan");
        } else {
            const FrRuffiniSerialBody::Args a{in, out, n, p, rem};
            if (!be.template run_simple<FrRuffiniSerialBody>(a, 1, CLS_OTHER)) return fail(PG_ERR_CUDA, "ruffini loop");
        }
        return PG_OK;
    }
    // Rounds 4 and 5 for the caller's challenges (alpha beta gamma rho zeta v v') and t = pg_quotient's t_1 .. t_4: the 17 evaluations
    // (pg_proof_evaluations), and dst = [W_zeta, W_zeta_w, r] (3 x 2^log_n coefficients).  Coefficient vectors as for the quotient,
    // one evaluation pass over them (25 pairs), the weights on the host, one combination pass, two in-place Ruffini divisions whose
    // remainders must equal the aggregates' values computed from the evaluations.
    int prover_openings(uint32_t log_n, const pg_fr* challenges, const pg_fr* t_in, int t_on_device, pg_proof_evaluations* evals, pg_fr* dst,
                        int dst_on_device) {
        int rc;
        if ((rc = perm_unsharded("prover_openings"))) return rc;
        if (log_n > NTT_TWO_ADICITY - 2 || (1ull << log_n) < n_rows)
            return fail(PG_ERR_ARG, "prover_openings: domain smaller than the circuit, or larger than 2^30 (pg_quotient's bound)");
        if (!challenges || !t_in || !evals || !dst) return fail(PG_ERR_ARG, "prover_openings: null argument");
        for (int k = 0; k < 7; k++)
            if (!host_reduced(challenges[k])) return fail(PG_ERR_ARG, "prover_openings: a challenge (alpha beta gamma rho zeta v v') not fully reduced (>= q)");
        const uint64_t n = 1ull << log_n;
        const Fr al = fr_from_pg(challenges[0]), bt = fr_from_pg(challenges[1]), ga = fr_from_pg(challenges[2]), rh = fr_from_pg(challenges[3]);
        const Fr zt = fr_from_pg(challenges[4]), v = fr_from_pg(challenges[5]), vs = fr_from_pg(challenges[6]);
        const Fr one = fr_one(), zt_n = fr_pow2k(zt, log_n);
        if (fr_eq(zt_n, one)) return fail(PG_ERR_ARG, "prover_openings: zeta^N = 1 (zeta in the domain: L_1(zeta) and the verifier's 1 / Z_H(zeta) do not exist)");
        const Fr omega = fr_pow2k(fr_root_of_unity(), NTT_TWO_ADICITY - log_n), zw = fr_mul(zt, omega);
        const size_t mark = scratch.size();
        const uint4* t = stage(t_in, 4 * n, t_on_device, &rc); if (!t) return rc;
        uint4* coef = (uint4*)dalloc(QV_PI * n * sizeof(pg_fr)); if (!coef) return fail(PG_ERR_OOM, "opening coefficient vectors");
        scratch.push_back(coef);
        if ((rc = component_polynomials(log_n, &challenges[1], &challenges[2], false, coef))) return rc;
        // evaluation pass: s strided Horner chains per vector, partial sums of 2^7 then the rest
        const uint32_t log_s = std::min<uint32_t>(log_n, 14), log_g = std::min<uint32_t>(log_s, 7);
        const uint64_t s = 1ull << log_s, g = 1ull << log_g;
        const uint64_t entries = pow_table_entries(log_s);
        std::vector<Fr> host_tabs(2 * entries);
        pow_table_host(zt, log_s, host_tabs.data());
        pow_table_host(zw, log_s, host_tabs.data() + entries);
        uint4* buf = (uint4*)dalloc((host_tabs.size() + OV_PAIRS * s + OV_PAIRS * (s / g) + 2) * sizeof(pg_fr));
        if (!buf) return fail(PG_ERR_OOM, "evaluation buffers");
        scratch.push_back(buf);
        uint4* partial = buf + 2 * host_tabs.size(); uint4* partial2 = partial + 2 * OV_PAIRS * s; uint4* rem = partial2 + 2 * OV_PAIRS * (s / g);
        if (!be.h2d(buf, host_tabs.data(), host_tabs.size() * sizeof(pg_fr))) return fail(PG_ERR_CUDA, "power table copy");
        if ((rc = reset_counters())) return rc;
        OpenEvalBody::Args ea; memset(&ea, 0, sizeof(ea));
        ea.coef = coef; ea.t = t; ea.len = n; ea.s = s; ea.n = OV_VEC * s; ea.log_lo = pow_table_log_lo(log_s); ea.tab[0] = buf; ea.tab[1] = buf + 2 * entries;
        ea.step[0] = fr_pow2k(zt, log_s); ea.step[1] = fr_pow2k(zw, log_s); ea.partial = partial; ea.counters = d_counters;
        if (!be.template run_simple<OpenEvalBody>(ea, OV_VEC * s, CLS_OTHER)) return fail(PG_ERR_CUDA, "evaluation kernel");
        OpenSumBody::Args s1{partial, partial2, g, OV_PAIRS * (s / g)}, s2{partial2, partial, s / g, OV_PAIRS};
        if (!be.template run_simple<OpenSumBody>(s1, OV_PAIRS * (s / g), CLS_OTHER) || !be.template run_simple<OpenSumBody>(s2, OV_PAIRS, CLS_OTHER))
            return fail(PG_ERR_CUDA, "evaluation sum kernel");
        unsigned long long c[CNT_WORDS];
        if ((rc = read_counters(c))) return rc;
        if (c[CNT_UNSAT]) {
            char msg[200];
            snprintf(msg, sizeof(msg), "prover_openings: %llu coefficient(s) of t not fully reduced (>= q), first at index %llu", c[CNT_UNSAT], c[CNT_FIRST_BAD]);
            return fail(PG_ERR_ARG, msg);
        }
        pg_fr ev_pg[OV_PAIRS];
        if ((rc = deliver(ev_pg, partial, sizeof(ev_pg), 0))) return rc;
        Fr e[OV_PAIRS];
        for (uint32_t k = 0; k < OV_PAIRS; k++) e[k] = fr_from_pg(ev_pg[k]);
        const Fr a_ = e[QV_W], b_ = e[QV_W + 1], c_ = e[QV_W + 2], d_ = e[QV_W + 3], aw = e[OV_SHIFTED], bw = e[OV_SHIFTED + 1], dw = e[OV_SHIFTED + 2];
        const Fr zw_ = e[OV_SHIFTED + 3];
        const Fr zt_2n = fr_mul(zt_n, zt_n), zt_3n = fr_mul(zt_2n, zt_n);
        const Fr t_bar = fr_add(fr_add(e[OV_T], fr_mul(zt_n, e[OV_T + 1])), fr_add(fr_mul(zt_2n, e[OV_T + 2]), fr_mul(zt_3n, e[OV_T + 3])));
        // linearisation weights: r = rw . (q_m q_l q_r q_o q_4 q_c q_range z sigma_4)
        const Fr qa = e[QV_QARITH], two = fr_small(2), three = fr_small(3), kappa = fr_sqr(rh);
        Fr rw[9];
        rw[0] = fr_mul(qa, fr_mul(a_, b_)); rw[1] = fr_mul(qa, a_); rw[2] = fr_mul(qa, b_); rw[3] = fr_mul(qa, c_); rw[4] = fr_mul(qa, d_); rw[5] = qa;
        Fr rng = quot_delta(fr_sub(dw, quot_times4(a_)), two, three);
        rng = fr_add(fr_mul(rng, kappa), quot_delta(fr_sub(a_, quot_times4(b_)), two, three));
        rng = fr_add(fr_mul(rng, kappa), quot_delta(fr_sub(b_, quot_times4(c_)), two, three));
        rng = fr_add(fr_mul(rng, kappa), quot_delta(fr_sub(c_, quot_times4(d_)), two, three));
        rw[6] = fr_mul(rh, rng);
        const Fr wv[4] = {a_, b_, c_, d_};
        Fr prod_id = one, prod_sig = one;                                   // prod_w (v_w + beta k_w zeta + gamma), prod_(w<3) (v_w + beta sigma_w + gamma)
        for (uint32_t w = 0; w < 4; w++) {
            prod_id = fr_mul(prod_id, fr_add(fr_add(wv[w], fr_mul(fr_mul(bt, perm_coset(w)), zt)), ga));
            if (w < 3) prod_sig = fr_mul(prod_sig, fr_add(fr_add(wv[w], fr_mul(bt, e[QV_S + w])), ga));
        }
        const Fr alpha2 = fr_sqr(al);
        const Fr l1 = fr_mul(fr_sub(zt_n, one), fr_inv_fermat(fr_mul(fr_small(n), fr_sub(zt, one))));       // (zeta^N - 1) / (N (zeta - 1))
        rw[7] = fr_add(fr_mul(al, prod_id), fr_mul(alpha2, l1));
        rw[8] = fr_neg(fr_mul(fr_mul(fr_mul(al, bt), zw_), prod_sig));
        const uint32_t r_terms[9] = {QV_QM, QV_QL, QV_QR, QV_QO, QV_Q4, QV_QC, QV_QRANGE, QV_Z, QV_S + 3};
        Fr r_bar = fr_zero();
        for (int k = 0; k < 9; k++) r_bar = fr_add(r_bar, fr_mul(rw[k], e[r_terms[k]]));
        const Fr out_ev[17] = {a_, b_, c_, d_, aw, bw, dw, qa, e[QV_QC], e[QV_QL], e[QV_QR], e[QV_S], e[QV_S + 1], e[QV_S + 2], r_bar, zw_, t_bar};
        // combination pass
        uint4* out = reinterpret_cast<uint4*>(dst);
        if (!dst_on_device) { out = (uint4*)dalloc(3 * n * sizeof(pg_fr)); if (!out) return fail(PG_ERR_OOM, "opening buffer"); scratch.push_back(out); }
        OpenCombineBody::Args ca; memset(&ca, 0, sizeof(ca));
        ca.coef = coef; ca.t = t; ca.n = n; ca.out = out;
        for (int k = 0; k < 9; k++) ca.rw[k] = rw[k];
        ca.zn[0] = zt_n; ca.zn[1] = zt_2n; ca.zn[2] = zt_3n;
        ca.v[0] = v; for (int k = 1; k < 8; k++) ca.v[k] = fr_mul(ca.v[k - 1], v);
        ca.vs[0] = vs; ca.vs[1] = fr_mul(vs, vs); ca.vs[2] = fr_mul(ca.vs[1], vs);
        if (!be.template run_simple<OpenCombineBody>(ca, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "combination kernel");
        // the aggregates' values at their points, from the evaluations
        const Fr agg_at[2] = {
            [&] { Fr x = t_bar; const Fr p[8] = {r_bar, a_, b_, c_, d_, e[QV_S], e[QV_S + 1], e[QV_S + 2]};
                  for (int k = 0; k < 8; k++) x = fr_add(x, fr_mul(ca.v[k], p[k])); return x; }(),
            fr_add(fr_add(zw_, fr_mul(ca.vs[0], aw)), fr_add(fr_mul(ca.vs[1], bw), fr_mul(ca.vs[2], dw)))};
        const Fr pts[2] = {zt, zw};
        for (int k = 0; k < 2; k++)
            if ((rc = fr_ruffini(out + 2 * (uint64_t)k * n, out + 2 * (uint64_t)k * n, n, pts[k], rem + 2 * k))) return rc;
        pg_fr rem_pg[2];
        if ((rc = deliver(rem_pg, rem, sizeof(rem_pg), 0))) return rc;
        for (int k = 0; k < 2; k++)
            if (!fr_eq(fr_from_pg(rem_pg[k]), agg_at[k]))
                return fail(PG_ERR_CUDA, k ? "prover_openings: the division's remainder differs from the zeta*w aggregate's evaluation"
                                           : "prover_openings: the division's remainder differs from the zeta aggregate's evaluation");
        for (int k = 0; k < 17; k++) reinterpret_cast<pg_fr*>(evals)[k] = fr_to_pg(out_ev[k]);      // the struct's 17 fields, in order
        if (!dst_on_device && (rc = deliver(dst, out, 3 * n * sizeof(pg_fr), 0))) return rc;
        release_scratch_from(mark);
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ export (SURVEY.md 8f.1)
    // Everything a host needs to rebuild this composer inside a real dusk-plonk StandardComposer (the import adapter replays it:
    // bindings/rust/.../import.rs), written to one little-endian file in chunks so that the expanded form never has to fit anywhere:
    //   header   : "PGB2EXP1", u32 version = 1, u32 flags (bit 0: sigma present), u64 n_rows, n_vars, n_calls, chunk_rows, 2 x u64 0
    //   calls    : n_calls x 64 bytes {u32 kind (GadgetKind), u32 num_bits, u64 n_inst, base_row, base_var, u32 rows/inst, u32 vars/inst,
    //              u64 first Variable of operand 0 (instance 0), u64 its stride, u64 0} -- range_gate calls are replayed natively
    //   variables: n_vars x 32 bytes, BlsScalar::to_bytes (canonical little endian)
    //   row chunks until n_rows: u64 row0, u64 cnt, w_idx[4][cnt] u64 (w_l, w_r, w_o, w_4), sel[8][cnt] x 32 bytes canonical
    //              (q_m q_l q_r q_o q_4 q_c q_arith q_range), pi[cnt] x 32 bytes canonical (dense), then sigma[4][cnt] u64 if flagged
    int export_composer(const char* path, uint64_t chunk_rows, uint32_t flags) {
        if (!path) return fail(PG_ERR_ARG, "export_composer: null path");
        if (!chunk_rows) chunk_rows = 1ull << 20;
        FILE* f = fopen(path, "wb");
        if (!f) return fail(PG_ERR_ARG, std::string("export_composer: cannot open ") + path);
        struct Closer { FILE* f; ~Closer() { if (f) fclose(f); } } closer{f};
        auto put = [&](const void* p, size_t bytes) { return fwrite(p, 1, bytes, f) == bytes; };
        const uint64_t n_calls = segs.size();
        { char magic[8] = {'P', 'G', 'B', '2', 'E', 'X', 'P', '1'}; uint32_t ver = 1, fl = flags & 1u;
          uint64_t h[6] = {n_rows, n_vars, n_calls, chunk_rows, 0, 0};
          if (!put(magic, 8) || !put(&ver, 4) || !put(&fl, 4) || !put(h, sizeof(h))) return fail(PG_ERR_STATE, "export_composer: write failed"); }
        for (const Segment& sg : segs) {
            uint64_t e[8] = {0, sg.n_inst, sg.base_row, sg.base_var, 0, 0, 0, 0};
            e[0] = (uint64_t)(uint32_t)sg.t.kind | ((uint64_t)sg.t.k << 32);
            e[4] = (uint64_t)(uint32_t)sg.t.rows.size() | ((uint64_t)sg.t.n_vars << 32);
            if (!sg.operands.empty()) { const Column& c = sg.operands[0]; const Segment& os = segs[c.seg]; e[5] = os.base_var + c.inst_off * os.t.n_vars + c.local; e[6] = os.t.n_vars; }
            if (!put(e, sizeof(e))) return fail(PG_ERR_STATE, "export_composer: write failed");
        }
        std::vector<pg_fr> host(chunk_rows * 8);
        std::vector<uint64_t> idx(chunk_rows * 4);
        const size_t mark = scratch.size();
        uint4* d_a = (uint4*)dalloc(chunk_rows * 8 * sizeof(pg_fr)); uint4* d_b = (uint4*)dalloc(chunk_rows * 8 * sizeof(pg_fr));
        if (!d_a || !d_b) return fail(PG_ERR_OOM, "export buffers");
        scratch.push_back(d_a); scratch.push_back(d_b);
        int rc;
        for (uint64_t v0 = 0; v0 < n_vars; v0 += chunk_rows * 8) {          // variables, canonical bytes
            const uint64_t cnt = std::min<uint64_t>(chunk_rows * 8, n_vars - v0);
            if ((rc = read_variables(v0, cnt, reinterpret_cast<pg_fr*>(d_a), 1))) return rc;
            if ((rc = convert(true, cnt, reinterpret_cast<const pg_fr*>(d_a), reinterpret_cast<pg_fr*>(d_b), 1, nullptr, nullptr))) return rc;
            if ((rc = deliver(host.data(), d_b, cnt * sizeof(pg_fr), 0))) return rc;
            if (!put(host.data(), cnt * sizeof(pg_fr))) return fail(PG_ERR_STATE, "export_composer: write failed");
        }
        for (uint64_t r0 = 0; r0 < n_rows; r0 += chunk_rows) {
            const uint64_t cnt = std::min<uint64_t>(chunk_rows, n_rows - r0);
            const uint64_t hdr[2] = {r0, cnt};
            if (!put(hdr, sizeof(hdr))) return fail(PG_ERR_STATE, "export_composer: write failed");
            if ((rc = materialize(r0, cnt, idx.data(), nullptr, nullptr, nullptr, 0))) return rc;
            if (!put(idx.data(), 4 * cnt * sizeof(uint64_t))) return fail(PG_ERR_STATE, "export_composer: write failed");
            // selectors: 6 columns + q_arith + q_range, then PI, all to canonical bytes on the device
            if ((rc = materialize(r0, cnt, nullptr, nullptr, reinterpret_cast<pg_fr*>(d_a), nullptr, 1))) return rc;
            if ((rc = gate_selectors(r0, cnt, reinterpret_cast<pg_fr*>(d_a + 2 * 6 * cnt), reinterpret_cast<pg_fr*>(d_a + 2 * 7 * cnt), 1))) return rc;
            if ((rc = convert(true, 8 * cnt, reinterpret_cast<const pg_fr*>(d_a), reinterpret_cast<pg_fr*>(d_b), 1, nullptr, nullptr))) return rc;
            if ((rc = deliver(host.data(), d_b, 8 * cnt * sizeof(pg_fr), 0))) return rc;
            if (!put(host.data(), 8 * cnt * sizeof(pg_fr))) return fail(PG_ERR_STATE, "export_composer: write failed");
            if ((rc = materialize(r0, cnt, nullptr, nullptr, nullptr, reinterpret_cast<pg_fr*>(d_a), 1))) return rc;
            if ((rc = convert(true, cnt, reinterpret_cast<const pg_fr*>(d_a), reinterpret_cast<pg_fr*>(d_b), 1, nullptr, nullptr))) return rc;
            if ((rc = deliver(host.data(), d_b, cnt * sizeof(pg_fr), 0))) return rc;
            if (!put(host.data(), cnt * sizeof(pg_fr))) return fail(PG_ERR_STATE, "export_composer: write failed");
            if (flags & 1u) {
                if ((rc = permutation(r0, cnt, idx.data(), 0))) return rc;
                if (!put(idx.data(), 4 * cnt * sizeof(uint64_t))) return fail(PG_ERR_STATE, "export_composer: write failed");
            }
        }
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        release_scratch_from(mark);
        return PG_OK;
    }

    // ------------------------------------------------------------------------------------------------ helpers
    int synth(uint64_t seed, uint64_t stream, uint64_t n, int kind, uint32_t bits, pg_fr* dst) {
        if (n && !dst) return fail(PG_ERR_ARG, "synth: null destination");
        if (kind < 0 || kind > 3 || (kind != 0 && bits > 254)) return fail(PG_ERR_ARG, "synth: kind/bits");
        SynthBody::Args a{seed ^ (stream * 0xD1342543DE82EF95ull), n, kind, bits, reinterpret_cast<uint4*>(dst)};
        if (n && !be.template run_simple<SynthBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "synth kernel");
        return PG_OK;
    }
    // canonical little-endian bytes <-> Montgomery limbs, n scalars; src/dst both host or both device
    int convert(bool to_bytes, uint64_t n, const pg_fr* src, pg_fr* dst, int on_device, uint64_t* n_invalid, uint64_t* first_invalid) {
        if (n_invalid) *n_invalid = 0;
        if (first_invalid) *first_invalid = ~0ull;
        if (!n) return PG_OK;
        if (!src || !dst) return fail(PG_ERR_ARG, "convert: null argument");
        const size_t mark = scratch.size();
        int rc; const uint4* ds = stage(src, n, on_device, &rc); if (!ds) return rc;
        uint4* dd = on_device ? reinterpret_cast<uint4*>(dst) : (uint4*)dalloc(n * sizeof(pg_fr));
        if (!dd) return fail(PG_ERR_OOM, "convert buffer");
        if (!on_device) scratch.push_back(dd);
        if (to_bytes) {
            ToBytesBody::Args a{ds, dd, n};
            if (!be.template run_simple<ToBytesBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "to_bytes kernel");
        } else {
            if ((rc = reset_counters())) return rc;
            FromBytesBody::Args a{ds, dd, n, d_counters};
            if (!be.template run_simple<FromBytesBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "from_bytes kernel");
            unsigned long long c[CNT_WORDS];
            if ((rc = read_counters(c))) return rc;
            if (n_invalid) *n_invalid = c[CNT_N_ERR];
            if (first_invalid) *first_invalid = c[CNT_N_ERR] ? c[CNT_FIRST_ERR] : ~0ull;
        }
        if (on_device) return PG_OK;
        rc = deliver(dst, dd, n * sizeof(pg_fr), 0);
        release_scratch_from(mark);
        return rc;
    }
    int fr_op(int op, uint64_t n, const pg_fr* a, const pg_fr* b, pg_fr* out) {
        if (!n) return PG_OK;
        if (!a || !out) return fail(PG_ERR_ARG, "fr_op: null argument");
        const size_t mark = scratch.size();
        int rc; const uint4* da = stage(a, n, 0, &rc); if (!da) return rc;
        if (op == 8 && !b) return fail(PG_ERR_ARG, "fr_op 8: null b");
        const uint4* db = nullptr; if (b && op != 8) { db = stage(b, n, 0, &rc); if (!db) return rc; }
        uint4* dout = (uint4*)dalloc(n * sizeof(pg_fr)); if (!dout) return fail(PG_ERR_OOM, "fr_op buffer");
        scratch.push_back(dout);
        bool ok;
        if (op == 4) {   // invert-or-zero through the batch-inversion kernel: a 2-slot scratch table (slot 0 in, slot 1 out)
            uint4* tab = (uint4*)dalloc(n * 4 * sizeof(uint4)); if (!tab) return fail(PG_ERR_OOM, "fr_op table");
            scratch.push_back(tab);
            AddInputBody::Args in{da, tab, n, n};
            BatchInvArgs inv; memset(&inv, 0, sizeof(inv));
            inv.fr = tab; inv.stride = n; inv.n = n; inv.n_pairs = 1; inv.in_slot[0] = 0; inv.out_slot[0] = 1;
            DevTab view; memset(&view, 0, sizeof(view)); view.fr = tab; view.stride = n;
            ColReadBody::Args rd{view, loc_make(LOC_FR, 0, 1), dout, n};
            ok = be.template run_simple<AddInputBody>(in, n, CLS_OTHER) && be.run_batch_inv(inv, CLS_OTHER) && be.template run_simple<ColReadBody>(rd, n, CLS_OTHER);
        }
        else if (op == 8) {  // Ruffini division by (X - b[0]) in place on the staged copy of a, the remainder a(b[0]) into out[n-1]
            if (!host_reduced(*b)) return fail(PG_ERR_ARG, "fr_op 8: b[0] not fully reduced (>= q)");
            uint4* rem = (uint4*)dalloc(sizeof(pg_fr)); if (!rem) return fail(PG_ERR_OOM, "fr_op remainder");
            scratch.push_back(rem);
            uint4* d = const_cast<uint4*>(da);
            if ((rc = fr_ruffini(d, d, n, fr_from_pg(*b), rem))) return rc;
            ok = be.d2d(d + 2 * (n - 1), rem, sizeof(pg_fr));
            dout = d;
        }
        else if (op == 7) {  // exclusive prefix product through the grand-product scan (scan.cuh)
            uint4* tot = (uint4*)dalloc((1 + fr_scan_scratch(n)) * sizeof(pg_fr)); if (!tot) return fail(PG_ERR_OOM, "fr_op scan scratch");
            scratch.push_back(tot);
            ok = fr_scan(da, dout, n, tot, tot + 2);
        }
        else { FrOpBody::Args g{op, da, db, dout, n}; ok = be.template run_simple<FrOpBody>(g, n, CLS_OTHER); }
        if (!ok) return fail(PG_ERR_CUDA, "fr_op kernel");
        rc = deliver(out, dout, n * sizeof(pg_fr), 0);
        release_scratch_from(mark);
        return rc;
    }
    // ------------------------------------------------------------------------------------------------ commitments (SURVEY 8f.2)
    // msm_variable_base / CommitKey::commit / PublicParameters::setup powers; see msm.cuh.  Points are 96-byte affine pairs.
    const uint4* stage_bytes(const void* p, size_t bytes, int on_device, int* rc) {
        return stage(reinterpret_cast<const pg_fr*>(p), (bytes + sizeof(pg_fr) - 1) / sizeof(pg_fr), on_device, rc);   // whole 32-byte units
    }
    // device-side MSM: d_points (n affine), d_scalars (n Montgomery scalars) -> d_out (one affine point, 96 bytes)
    // `defer` != nullptr: the window sums (n_windows XYZZ points) are parked there instead of being combined; msm_finish combines the
    // window sums of several MSMs of the same size in one launch.
    int msm_dev(uint64_t n, const uint4* d_points, const uint4* d_scalars, uint4* d_out, uint4* defer = nullptr) {
        const size_t mark = scratch.size();
        auto tmp = [&](size_t bytes) -> void* { void* q = dalloc(bytes); if (q) scratch.push_back(q); return q; };
        const MsmPlan plan = msm_plan(n);
        const uint64_t count = (uint64_t)plan.n_windows * n, n_buckets = (uint64_t)plan.n_windows << plan.c;
        uint32_t key_bits = plan.c; while ((1u << (key_bits - plan.c)) < plan.n_windows) key_bits++;
        uint32_t* keys = (uint32_t*)tmp(count * 4); uint32_t* vals = (uint32_t*)tmp(count * 4);
        uint32_t* keys2 = (uint32_t*)tmp(count * 4); uint32_t* vals2 = (uint32_t*)tmp(count * 4);
        uint4* buckets = (uint4*)tmp(n_buckets * sizeof(G1X));
        const uint64_t n_chunks = n_buckets / plan.chunk;
        uint4* ping = (uint4*)tmp(n_chunks * sizeof(G1X)); uint4* pong = (uint4*)tmp(((n_chunks + 15) / 16 + plan.n_windows) * sizeof(G1X));
        if (!keys || !vals || !keys2 || !vals2 || !buckets || !ping || !pong) return fail(PG_ERR_OOM, "msm buffers");
        MsmDigitsBody::Args dg{d_scalars, keys, vals, n, plan.c, plan.n_windows};
        if (!be.template run_simple<MsmDigitsBody>(dg, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm digits kernel");
        if (!be.sort_pairs(keys, vals, keys2, vals2, count, key_bits)) return fail(PG_ERR_CUDA, "msm sort");
        unsigned long long* start = (unsigned long long*)tmp(n_buckets * 8);
        uint32_t* size_key = (uint32_t*)tmp(n_buckets * 4); uint32_t* ids = (uint32_t*)tmp(n_buckets * 4);
        uint32_t* size_key2 = (uint32_t*)tmp(n_buckets * 4); uint32_t* ids2 = (uint32_t*)tmp(n_buckets * 4);
        if (!start || !size_key || !ids || !size_key2 || !ids2) return fail(PG_ERR_OOM, "msm buffers");
        MsmBoundsBody::Args bd{keys2, start, size_key, ids, count, n_buckets, plan.c};
        if (!be.template run_simple<MsmBoundsBody>(bd, n_buckets, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm bounds kernel");
        if (!be.sort_pairs(size_key, ids, size_key2, ids2, n_buckets, 32)) return fail(PG_ERR_CUDA, "msm bucket-order sort");
        // bucket sums in three levels (parts of <= 512 entries, groups of <= 64 parts, one thread per bucket): see msm.cuh
        const uint64_t max_parts = count / MSM_PART + n_buckets, max_groups = max_parts / MSM_GROUP + n_buckets;
        uint32_t* parts = (uint32_t*)tmp(n_buckets * 4); uint32_t* groups = (uint32_t*)tmp(n_buckets * 4);
        uint32_t* off1 = (uint32_t*)tmp(n_buckets * 4); uint32_t* off2 = (uint32_t*)tmp(n_buckets * 4);
        uint32_t* part_owner = (uint32_t*)tmp(max_parts * 4); uint32_t* group_owner = (uint32_t*)tmp(max_groups * 4);
        uint4* p1 = (uint4*)tmp(max_parts * sizeof(G1X)); uint4* p2 = (uint4*)tmp(max_groups * sizeof(G1X));
        if (!parts || !groups || !off1 || !off2 || !part_owner || !group_owner || !p1 || !p2) return fail(PG_ERR_OOM, "msm buffers");
        if (max_parts >= (1ull << 32)) return fail(PG_ERR_ARG, "msm: too many terms for 32-bit part numbers");
        MsmPartsBody::Args pb{size_key2, parts, groups, n_buckets};
        if (!be.template run_simple<MsmPartsBody>(pb, n_buckets, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm parts kernel");
        if (!be.exclusive_sum(parts, off1, n_buckets) || !be.exclusive_sum(groups, off2, n_buckets)) return fail(PG_ERR_CUDA, "msm scan");
        MsmExpandBody::Args ex{parts, groups, off1, off2, part_owner, group_owner, n_buckets};
        if (!be.template run_simple<MsmExpandBody>(ex, n_buckets, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm expand kernel");
        MsmBucketBody::Args bk{ids2, size_key2, start, vals2, d_points, parts, off1, part_owner, p1, max_parts, n_buckets};
        if (!be.run_msm_buckets(bk)) return fail(PG_ERR_CUDA, "msm bucket kernel");
        MsmGroupSumBody::Args gs{parts, groups, off1, off2, group_owner, p1, p2, max_groups, n_buckets};
        if (!be.template run_simple<MsmGroupSumBody>(gs, max_groups, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm group kernel");
        MsmBucketFinishBody::Args bf{ids2, groups, off2, p2, buckets, n_buckets};
        if (!be.template run_simple<MsmBucketFinishBody>(bf, n_buckets, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm bucket finish kernel");
        MsmChunkBody::Args ck{buckets, ping, n_chunks, plan.c, plan.chunk};
        if (!be.template run_simple<MsmChunkBody>(ck, n_chunks, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm chunk kernel");
        uint32_t seg = (1u << plan.c) / plan.chunk;                    // partial sums per window
        uint4 *src = ping, *dst = pong;
        while (seg > 1) {
            const uint32_t seg_out = (seg + 15) / 16;
            MsmSumBody::Args sm{src, dst, (uint64_t)plan.n_windows * seg_out, seg, seg_out, 16};
            if (!be.template run_simple<MsmSumBody>(sm, sm.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm sum kernel");
            std::swap(src, dst); seg = seg_out;
        }
        if (defer) { if (!be.d2d(defer, src, (size_t)plan.n_windows * sizeof(G1X))) return fail(PG_ERR_CUDA, "msm window sums"); }
        else {
            MsmFinalBody::Args fin{src, d_out, 1, plan.c, plan.n_windows};
            if (!be.template run_simple<MsmFinalBody>(fin, 1, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm final kernel");
        }
        release_scratch_from(mark);      // work buffers are only touched by kernels on the engine's stream: stream order makes their reuse safe
        return PG_OK;
    }
    // d_out[t] = the MSM whose window sums were parked at windows + t * n_windows (count MSMs of n terms each)
    int msm_finish(uint64_t n, const uint4* windows, uint64_t count, uint4* d_out) {
        const MsmPlan plan = msm_plan(n);
        MsmFinalBody::Args fin{windows, d_out, count, plan.c, plan.n_windows};
        if (!be.template run_simple<MsmFinalBody>(fin, count, CLS_OTHER)) return fail(PG_ERR_CUDA, "msm final kernel");
        return PG_OK;
    }
    static constexpr size_t MSM_MAX_WINDOWS = 256;     // c >= 1
    int msm(uint64_t n, const pg_g1_affine* points, const pg_fr* scalars, pg_g1_affine* out, int on_device) {
        if (!out || (n && (!points || !scalars))) return fail(PG_ERR_ARG, "msm: null argument");
        if (n >= (1ull << 32)) return fail(PG_ERR_ARG, "msm: more than 2^32 - 1 terms");
        if (!n) { memset(out, 0, sizeof(*out)); return PG_OK; }          // empty sum: the point at infinity
        const size_t mark = scratch.size();
        int rc; const uint4* dp = stage_bytes(points, n * sizeof(pg_g1_affine), on_device, &rc); if (!dp) return rc;
        const uint4* ds = stage(scalars, n, on_device, &rc); if (!ds) return rc;
        uint4* d_out = (uint4*)dalloc(sizeof(pg_g1_affine)); if (!d_out) return fail(PG_ERR_OOM, "msm result"); scratch.push_back(d_out);
        if ((rc = msm_dev(n, dp, ds, d_out))) return rc;
        rc = deliver(out, d_out, sizeof(pg_g1_affine), 0);
        release_scratch_from(mark);
        return rc;
    }
    // out[i] = scalars[i] * base (base == nullptr: the G1 generator)
    int g1_fixed_base_mul(uint64_t n, const pg_g1_affine* base, const pg_fr* scalars, pg_g1_affine* out, int on_device) {
        if (n && (!scalars || !out)) return fail(PG_ERR_ARG, "g1_fixed_base_mul: null argument");
        if (!n) return PG_OK;
        const size_t mark = scratch.size();
        int rc; const uint4* ds = stage(scalars, n, on_device, &rc); if (!ds) return rc;
        rc = g1_fixed_base_mul_dev(n, base, ds, out, on_device);
        if (!on_device) release_scratch_from(mark);      // (host results: g1_fixed_base_mul_dev has synchronised)
        return rc;
    }
    // the same with the scalars already in device memory and the result in host or device memory
    int g1_fixed_base_mul_dev(uint64_t n, const pg_g1_affine* base, const uint4* d_scalars, pg_g1_affine* out, int out_on_device) {
        const size_t mark = scratch.size();
        uint4* d_out = reinterpret_cast<uint4*>(out);
        if (!out_on_device) { d_out = (uint4*)dalloc(n * sizeof(pg_g1_affine)); if (!d_out) return fail(PG_ERR_OOM, "point buffer"); scratch.push_back(d_out); }
        G1Affine b;
        if (base) memcpy(&b, base, sizeof(G1Affine)); else b = g1_generator();
        // The table costs a few milliseconds to build (its critical path is 248 dependent doublings and one inversion on a thread):
        // worth it from FB_MIN_POINTS scalars on, or from FB_MIN_POINTS_CACHED when it exists already -- the generator's table is kept
        // for the life of the ctx (PublicParameters::setup and the Lagrange-basis SRS both multiply the generator).
        const char* fb_env = getenv("PG_FB_MIN");                                                                  // tests
        const uint64_t min_env = fb_env ? strtoull(fb_env, nullptr, 10) : 0;
        const bool have_table = !base && fb_table_gen;
        if (n >= (min_env ? min_env : have_table ? FB_MIN_POINTS_CACHED : FB_MIN_POINTS)) {
            // windowed table of multiples of the base, then tiles of FB_TILE scalars: <= 32 mixed additions each, batch normalisation
            const uint64_t n_table = (uint64_t)FB_WINDOWS * FB_ENTRIES, tile = std::min<uint64_t>(n, FB_TILE);
            uint4* table = have_table ? fb_table_gen : (uint4*)dalloc(n_table * sizeof(pg_g1_affine));
            uint4* xyzz = (uint4*)dalloc(tile * sizeof(G1X)); uint4* prefix = (uint4*)dalloc(tile * sizeof(Fp));
            if (!table || !xyzz || !prefix) return fail(PG_ERR_OOM, "fixed-base buffers");
            if (!have_table && base) scratch.push_back(table);
            scratch.push_back(xyzz); scratch.push_back(prefix);
            if (!have_table) {
                G1WindowTableBody::Args ta; ta.table = table; ta.n = n_table; ta.base = b;
                if (!be.template run_simple<G1WindowTableBody>(ta, n_table, CLS_OTHER)) return fail(PG_ERR_CUDA, "fixed-base table kernel");
                if (!base) fb_table_gen = table;
            }
            for (uint64_t i0 = 0; i0 < n; i0 += tile) {
                const uint64_t cnt = std::min<uint64_t>(tile, n - i0), threads = (cnt + FB_CHUNK - 1) / FB_CHUNK;
                G1FixedBaseWindowedBody::Args wa{d_scalars + 2 * i0, table, xyzz, cnt};
                G1BatchAffineBody::Args na{xyzz, prefix, d_out + 6 * i0, threads, cnt};
                if (!be.template run_simple<G1FixedBaseWindowedBody>(wa, cnt, CLS_OTHER) || !be.template run_simple<G1BatchAffineBody>(na, threads, CLS_OTHER))
                    return fail(PG_ERR_CUDA, "fixed-base kernels");
            }
        } else {
            G1FixedBaseMulBody::Args a; a.scalars = d_scalars; a.out = d_out; a.n = n; a.base = b;
            if (!be.template run_simple<G1FixedBaseMulBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "fixed-base kernel");
        }
        if (out_on_device) { release_scratch_from(mark); return PG_OK; }      // work buffers are only touched on the engine's stream
        const int rc = deliver(out, d_out, n * sizeof(pg_g1_affine), 0);
        release_scratch_from(mark);
        return rc;
    }
    // powers_of_g[i] = beta^i * base, i < n  (PublicParameters::setup)
    int srs_powers(const pg_fr* beta, const pg_g1_affine* base, uint64_t n, pg_g1_affine* out, int out_on_device) {
        if (!beta || (n && !out)) return fail(PG_ERR_ARG, "srs_powers: null argument");
        if (!n) return PG_OK;
        const size_t mark = scratch.size();
        uint4* pw = (uint4*)dalloc(n * sizeof(pg_fr));                     // util::powers_of(beta, n), on the device
        if (!pw) return fail(PG_ERR_OOM, "powers of beta");
        scratch.push_back(pw);
        FrPowersBody::Args pa; memcpy(&pa.beta, beta, sizeof(Fr)); pa.out = pw; pa.n = (n + FRPOW_CHUNK - 1) / FRPOW_CHUNK; pa.n_points = n;
        if (!host_reduced(*beta)) return fail(PG_ERR_ARG, "srs_powers: beta not fully reduced (>= q)");
        if (!be.template run_simple<FrPowersBody>(pa, pa.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "powers kernel");
        const int rc = g1_fixed_base_mul_dev(n, base, pw, out, out_on_device);
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        release_scratch_from(mark);
        return rc;
    }
    // the four wire-polynomial commitments of Prover::prove: out[w] = commit(w-th wire polynomial) against powers_of_g[0 .. 2^log_n)
    int commit_wire_polynomials(uint32_t log_n, const pg_g1_affine* powers, uint64_t n_powers, int powers_on_device, pg_g1_affine* out) {
        if (!powers || !out) return fail(PG_ERR_ARG, "commit_wire_polynomials: null argument");
        if (log_n <= NTT_TWO_ADICITY && n_powers < (1ull << log_n)) return fail(PG_ERR_ARG, "commit_wire_polynomials: the SRS holds fewer powers than the domain size (polynomial degree too large)");
        if (log_n > NTT_TWO_ADICITY || (1ull << log_n) < n_rows) return fail(PG_ERR_ARG, "commit_wire_polynomials: domain smaller than the circuit or larger than 2^32");
        const uint64_t n = 1ull << log_n;
        const size_t mark = scratch.size();
        int rc; const uint4* dp = stage_bytes(powers, n * sizeof(pg_g1_affine), powers_on_device, &rc); if (!dp) return rc;
        uint4* polys = (uint4*)dalloc(4 * n * sizeof(pg_fr)); if (!polys) return fail(PG_ERR_OOM, "wire polynomial buffer"); scratch.push_back(polys);
        uint4* d_out = (uint4*)dalloc(4 * sizeof(pg_g1_affine)); if (!d_out) return fail(PG_ERR_OOM, "commitments"); scratch.push_back(d_out);
        uint4* win = (uint4*)dalloc(4 * MSM_MAX_WINDOWS * sizeof(G1X)); if (!win) return fail(PG_ERR_OOM, "window sums"); scratch.push_back(win);
        if ((rc = wire_polynomials(log_n, reinterpret_cast<pg_fr*>(polys), 1))) return rc;
        for (int w = 0; w < 4; w++)
            if ((rc = msm_dev(n, dp, polys + 2 * (uint64_t)w * n, nullptr, win + (size_t)w * msm_plan(n).n_windows * (sizeof(G1X) / sizeof(uint4))))) return rc;
        if ((rc = msm_finish(n, win, 4, d_out))) return rc;                 // the four Horner chains side by side
        rc = deliver(out, d_out, 4 * sizeof(pg_g1_affine), 0);
        release_scratch_from(mark);
        return rc;
    }
    // out[i] = L_i(beta) * base, i < 2^log_n: the Lagrange-basis form of the SRS for that domain (test / local setups that know
    // beta, like PublicParameters::setup; srs_lagrange_from_powers derives the same points from the monomial powers alone)
    int srs_lagrange(const pg_fr* beta, const pg_g1_affine* base, uint32_t log_n, pg_g1_affine* out, int out_on_device) {
        if (!beta || !out || log_n > NTT_TWO_ADICITY) return fail(PG_ERR_ARG, "srs_lagrange: null argument or domain larger than 2^32");
        const uint64_t n = 1ull << log_n;
        int rc = log_n ? ntt_twiddles(log_n) : PG_OK;
        if (rc) return rc;
        const size_t mark = scratch.size();
        uint4* sc = (uint4*)dalloc(n * sizeof(pg_fr)); if (!sc) return fail(PG_ERR_OOM, "lagrange scalars"); scratch.push_back(sc);
        LagrangeScalarsBody::Args a; a.tw = ntt_tw; a.out = sc; a.n = n; a.log_n = log_n;
        memcpy(&a.beta, beta, sizeof(Fr));
        Fr bn = a.beta;                                                  // beta^n by log_n squarings
        for (uint32_t k = 0; k < log_n; k++) bn = fr_sqr(bn);
        const Fr z = fr_sub(bn, fr_one());                               // Z_H(beta) = beta^n - 1
        if (fr_is_zero(z)) return fail(PG_ERR_ARG, "srs_lagrange: beta lies on the evaluation domain");
        Fr raw = fr_zero(); raw.v[0] = (uint32_t)n; raw.v[1] = (uint32_t)(n >> 32);
        a.c = fr_mul(z, fr_inv_fermat(fr_to_mont(raw)));
        if (!be.template run_simple<LagrangeScalarsBody>(a, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "lagrange scalar kernel");
        if ((rc = g1_fixed_base_mul_dev(n, base, sc, out, out_on_device))) return rc;
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        release_scratch_from(mark);
        return PG_OK;
    }
    // out[i] = (1/n) sum_j w^(-ij) powers[j], i < n = 2^log_n: the Lagrange-basis SRS from the first n monomial powers, by the group
    // inverse FFT of g1fft.cuh.  For powers[j] = beta^j * base it is srs_lagrange(beta, base, log_n), point for point.
    int srs_lagrange_from_powers(uint32_t log_n, const pg_g1_affine* powers, uint64_t n_powers, int powers_on_device, pg_g1_affine* out, int out_on_device) {
        if (!powers || !out || log_n > NTT_TWO_ADICITY) return fail(PG_ERR_ARG, "srs_lagrange_from_powers: null argument or domain larger than 2^32");
        const uint64_t n = 1ull << log_n;
        if (n_powers < n) return fail(PG_ERR_ARG, "srs_lagrange_from_powers: the SRS holds fewer powers than the domain size");
        const size_t mark = scratch.size();
        auto tmp = [&](size_t bytes) -> uint4* { void* q = dalloc(bytes); if (q) scratch.push_back(q); return (uint4*)q; };
        int rc; const uint4* dp = stage_bytes(powers, n * sizeof(pg_g1_affine), powers_on_device, &rc); if (!dp) return rc;
        if (log_n == 0) rc = deliver(out, dp, sizeof(pg_g1_affine), out_on_device);          // L_0 = 1
        else {
            if ((rc = ntt_twiddles(log_n))) return rc;
            uint4* data = tmp(n * sizeof(G1X));
            uint4* d_out = out_on_device ? reinterpret_cast<uint4*>(out) : tmp(n * sizeof(pg_g1_affine));
            const uint64_t tile = std::min<uint64_t>(n, FB_TILE);
            uint4* prefix = tmp(tile * sizeof(Fp));
            if (!data || !d_out || !prefix) return fail(PG_ERR_OOM, "group FFT buffers");
            Fr raw = fr_zero(); raw.v[0] = (uint32_t)n; raw.v[1] = (uint32_t)(n >> 32);
            G1FftIngestBody::Args ia{dp, data, n, log_n, fr_from_mont(fr_inv_fermat(fr_to_mont(raw)))};
            if (!be.template run_simple<G1FftIngestBody>(ia, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "group FFT ingest kernel");
            for (uint32_t s = 0; s < log_n; s++) {
                G1FftStageBody::Args sa{data, ntt_tw, n >> 1, log_n, s};
                if (!be.template run_simple<G1FftStageBody>(sa, sa.n, CLS_OTHER)) return fail(PG_ERR_CUDA, "group FFT stage kernel");
            }
            for (uint64_t i0 = 0; i0 < n; i0 += tile) {
                const uint64_t cnt = std::min<uint64_t>(tile, n - i0), threads = (cnt + FB_CHUNK - 1) / FB_CHUNK;
                G1BatchAffineBody::Args na{data + 12 * i0, prefix, d_out + 6 * i0, threads, cnt};
                if (!be.template run_simple<G1BatchAffineBody>(na, threads, CLS_OTHER)) return fail(PG_ERR_CUDA, "group FFT normalisation kernel");
            }
            if (!out_on_device) rc = deliver(out, d_out, n * sizeof(pg_g1_affine), 0);
        }
        if (rc) return rc;
        if (!be.sync()) return fail(PG_ERR_CUDA, "sync");
        release_scratch_from(mark);
        return PG_OK;
    }
    // The four wire commitments from the wire VALUES (evaluation form) against a Lagrange-basis SRS: same group elements as
    // commit_wire_polynomials against the monomial powers of the same beta, without any FFT and with mostly-empty windows.
    int commit_wire_evaluations(uint32_t log_n, const pg_g1_affine* lagrange, uint64_t n_points, int points_on_device, pg_g1_affine* out) {
        if (!lagrange || !out) return fail(PG_ERR_ARG, "commit_wire_evaluations: null argument");
        if (log_n > NTT_TWO_ADICITY || (1ull << log_n) < n_rows) return fail(PG_ERR_ARG, "commit_wire_evaluations: domain smaller than the circuit or larger than 2^32");
        const uint64_t n = 1ull << log_n;
        if (n_points != n) return fail(PG_ERR_ARG, "commit_wire_evaluations: a Lagrange-basis SRS belongs to exactly one domain size");
        const size_t mark = scratch.size();
        int rc; const uint4* dp = stage_bytes(lagrange, n * sizeof(pg_g1_affine), points_on_device, &rc); if (!dp) return rc;
        uint4* vals = (uint4*)dalloc(4 * n * sizeof(pg_fr)); if (!vals) return fail(PG_ERR_OOM, "wire value buffer"); scratch.push_back(vals);
        uint4* d_out = (uint4*)dalloc(4 * sizeof(pg_g1_affine)); if (!d_out) return fail(PG_ERR_OOM, "commitments"); scratch.push_back(d_out);
        uint4* win = (uint4*)dalloc(4 * MSM_MAX_WINDOWS * sizeof(G1X)); if (!win) return fail(PG_ERR_OOM, "window sums"); scratch.push_back(win);
        if ((rc = wire_values(n, vals))) return rc;
        for (int w = 0; w < 4; w++) {
            uint4* col = vals + 2 * (uint64_t)w * n;
            if ((rc = msm_dev(n, dp, col, nullptr, win + (size_t)w * msm_plan(n).n_windows * (sizeof(G1X) / sizeof(uint4))))) return rc;
        }
        if ((rc = msm_finish(n, win, 4, d_out))) return rc;
        rc = deliver(out, d_out, 4 * sizeof(pg_g1_affine), 0);
        release_scratch_from(mark);
        return rc;
    }
    int g1_op(int op, uint64_t n, const pg_g1_affine* a, const pg_g1_affine* b, pg_g1_affine* out) {
        if (!n) return PG_OK;
        if (!a || !out || (op == 0 && !b)) return fail(PG_ERR_ARG, "g1_op: null argument");
        const size_t mark = scratch.size();
        int rc; const uint4* da = stage_bytes(a, n * sizeof(pg_g1_affine), 0, &rc); if (!da) return rc;
        const uint4* db = nullptr; if (b) { db = stage_bytes(b, n * sizeof(pg_g1_affine), 0, &rc); if (!db) return rc; }
        uint4* d_out = (uint4*)dalloc(n * sizeof(pg_g1_affine)); if (!d_out) return fail(PG_ERR_OOM, "g1_op buffer"); scratch.push_back(d_out);
        G1OpBody::Args g{da, db, d_out, n, op};
        if (!be.template run_simple<G1OpBody>(g, n, CLS_OTHER)) return fail(PG_ERR_CUDA, "g1_op kernel");
        rc = deliver(out, d_out, n * sizeof(pg_g1_affine), 0);
        release_scratch_from(mark);
        return rc;
    }
};

}  // namespace pg
