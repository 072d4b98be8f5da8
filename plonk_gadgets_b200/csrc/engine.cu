// engine.cu -- CUDA backend (sm_100a) and the extern "C" ABI of include/pg_b200.h.
//
// This translation unit is the whole shipped library: Engine<CudaBackend>.  There is no CPU path in it -- when no B200 is
// present pg_ctx_create fails with PG_ERR_NO_DEVICE and nothing else can be called.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <new>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include "engine.hpp"
#include "kernels.cuh"
#include "comm.cuh"

namespace pg {

Fr h_pow2[256];

#define PG_CUDA(call)                                                                     \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) { snprintf(errbuf, sizeof(errbuf), "%s: %s", #call, cudaGetErrorString(e_)); return false; } \
    } while (0)

class CudaBackend {
public:
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;      // device -> pinned-host result copies that overlap with later kernels
    cudaEvent_t copy_ready = nullptr;
    cudaStream_t in_stream = nullptr;        // chunked host -> device input copies that overlap with the kernels consuming earlier chunks
    struct PendingCopy { const void* table; const void* table_end; uint64_t lo, hi; cudaEvent_t ev; };   // elements [lo, hi) of `table` arrive with `ev`
    std::vector<PendingCopy> pending;
    std::vector<cudaEvent_t> sync_ev_free;   // events without timing, for stream ordering only
    bool own_stream = false;
    bool nodev = false;
    bool timing_on = false;
    char errbuf[512] = {0};
    int sm_count = 0;
    int check_shape = 0;
    struct Ev { cudaEvent_t a, b; int cls; uint64_t rows; };
    std::vector<Ev> events;
    std::vector<cudaEvent_t> ev_free;
    pg_timing acc{};

    const char* error() const { return errbuf; }
    bool no_device() const { return nodev; }
    int device = 0;
    void activate() { cudaSetDevice(device); }

    bool init(const pg_cfg& cfg) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) { nodev = true; snprintf(errbuf, sizeof(errbuf), "no CUDA device: %s", cudaGetErrorString(e)); return false; }
        if (cfg.device < 0 || cfg.device >= count) { nodev = true; snprintf(errbuf, sizeof(errbuf), "device %d out of range (%d devices)", cfg.device, count); return false; }
        PG_CUDA(cudaSetDevice(cfg.device));
        device = cfg.device;
        cudaDeviceProp prop;
        PG_CUDA(cudaGetDeviceProperties(&prop, cfg.device));
        if (prop.major != 10) { nodev = true; snprintf(errbuf, sizeof(errbuf), "device %d is sm_%d%d; this library is built for sm_100a only", cfg.device, prop.major, prop.minor); return false; }
        sm_count = prop.multiProcessorCount;
        if (cfg.stream) { stream = (cudaStream_t)cfg.stream; own_stream = false; }
        else { PG_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)); own_stream = true; }
        PG_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        PG_CUDA(cudaStreamCreateWithFlags(&in_stream, cudaStreamNonBlocking));
        PG_CUDA(cudaEventCreateWithFlags(&copy_ready, cudaEventDisableTiming));
        timing_on = (cfg.flags & PG_F_TIMING) != 0;
        check_shape = cfg.check_shape < (uint32_t)CHECK_SHAPES ? (int)cfg.check_shape : 0;
        PG_CUDA(cudaFuncSetAttribute(k_ntt_pass<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 << NTT_MAX_LOG_TILE));
        PG_CUDA(cudaFuncSetAttribute(k_ntt_pass<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 << NTT_MAX_LOG_TILE));
        PG_CUDA(cudaFuncSetAttribute(k_ntt_coset_pass, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 << NTT_MAX_LOG_TILE));
        PG_CUDA(cudaFuncSetAttribute(k_check_rowpar<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        PG_CUDA(cudaFuncSetAttribute(k_check_rowpar<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        if (!set_check_attrs<0>() || !set_check_attrs<1>() || !set_check_attrs<2>() || !set_check_attrs<3>() || !set_check_attrs<4>()) return false;
        return true;
    }
    template <int SHAPE>
    bool set_check_attrs() {
        if constexpr (SHAPE == 0) PG_CUDA(cudaFuncSetAttribute(k_check_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        else PG_CUDA(cudaFuncSetAttribute(k_check<0, SHAPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        PG_CUDA(cudaFuncSetAttribute(k_check<1, SHAPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        PG_CUDA(cudaFuncSetAttribute(k_check_prog<SHAPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        return true;
    }
    template <int SHAPE>
    void launch_check(const CheckArgs& a, const SparseProg& prog, size_t smem) {
        constexpr int T = CheckShape<SHAPE>::BLOCK_T;
        const unsigned grid = (unsigned)((a.n_inst + T - 1) / T);
        if (a.mode == PG_CHECK_SPARSE && prog.ops) { const CheckProgArgs pa{a, prog}; k_check_prog<SHAPE><<<grid, T, smem, stream>>>(pa); }   // compiled row program
        else if (a.mode == PG_CHECK_SPARSE) k_check<1, SHAPE><<<grid, T, smem, stream>>>(a);
        else if constexpr (SHAPE == 0) k_check_tc<<<grid, T, smem, stream>>>(a);   // generic mode, default shape: tensor-core selector products
        else k_check<0, SHAPE><<<grid, T, smem, stream>>>(a);
    }
    void shutdown() {
        for (auto& ev : events) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
        for (auto& ev : ev_free) cudaEventDestroy(ev);
        events.clear(); ev_free.clear();
        if (sort_tmp) { cudaFree(sort_tmp); sort_tmp = nullptr; sort_tmp_bytes = 0; }
        comm.destroy();
        if (d_verdict) { cudaFree(d_verdict); d_verdict = nullptr; }
        for (auto& pc : pending) cudaEventDestroy(pc.ev);
        for (auto& r : results) cudaEventDestroy(r.ev);
        results.clear();
        for (auto& ev : sync_ev_free) cudaEventDestroy(ev);
        pending.clear(); sync_ev_free.clear();
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (in_stream) cudaStreamDestroy(in_stream);
        if (copy_ready) cudaEventDestroy(copy_ready);
        copy_stream = nullptr; in_stream = nullptr; copy_ready = nullptr;
        if (own_stream && stream) cudaStreamDestroy(stream);
        stream = nullptr;
    }
    void* alloc(size_t bytes) {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { snprintf(errbuf, sizeof(errbuf), "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return nullptr; }
        return p;
    }
    void release(void* p) { cudaFree(p); }
    bool h2d(void* dst, const void* src, size_t bytes) {
        for (auto& pc : pending)                    // a write INTO a table that is still arriving (pg_poke_variable) must land after it
            if (dst >= pc.table && dst < pc.table_end) { join_copies(); break; }
        PG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
        return true;
    }
    // ---- input copies that overlap with compute ----------------------------------------------------------------------
    // h2d_chunked copies `n` elements in chunks on in_stream, one event per chunk.  Until the main stream has waited on those
    // events the destination is "pending": join_copies() makes it wait on all of them and runs at the head of EVERY operation
    // that could read device memory (tic() -- i.e. every kernel launch --, d2h, d2d, d2h_async, sync, scans and sorts); the one
    // consumer that knows about chunks, run_simple_chunked, waits chunk by chunk instead and so overlaps with the copies.
    // Plain h2d joins only when its destination lies inside a pending table (template uploads and counter resets between
    // add_input and the range gadget write buffers of their own and must not serialise the pipeline).
    cudaEvent_t get_sync_event() {
        if (!sync_ev_free.empty()) { cudaEvent_t e = sync_ev_free.back(); sync_ev_free.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); return e;
    }
    void join_copies() {
        for (auto& pc : pending) { cudaStreamWaitEvent(stream, pc.ev, 0); sync_ev_free.push_back(pc.ev); }
        pending.clear();
    }
    bool h2d_chunked(void* dst, const void* src, uint64_t n, size_t elem, uint64_t chunk, unsigned long long* counters) {
        cudaEvent_t head = get_sync_event();         // the destination may come from the pool: order behind what is queued
        PG_CUDA(cudaEventRecord(head, stream));
        PG_CUDA(cudaStreamWaitEvent(in_stream, head, 0));
        sync_ev_free.push_back(head);
        for (uint64_t lo = 0; lo < n; lo += chunk) {
            const uint64_t hi = lo + chunk < n ? lo + chunk : n;
            PG_CUDA(cudaMemcpyAsync((char*)dst + lo * elem, (const char*)src + lo * elem, (hi - lo) * elem, cudaMemcpyHostToDevice, in_stream));
            if (counters) {                          // ingest check of the chunk (scalars must be < q), behind its copy on the same stream
                const ValidateBody::Args va{reinterpret_cast<const uint4*>(dst), lo, hi - lo, counters};
                k_simple<ValidateBody><<<grid_for(hi - lo), BLOCK, 0, in_stream>>>(va);
            }
            cudaEvent_t ev = get_sync_event();
            PG_CUDA(cudaEventRecord(ev, in_stream));
            pending.push_back(PendingCopy{dst, (const char*)dst + n * elem, lo, hi, ev});
        }
        return true;
    }
    // Body over [0, n) whose operand table may still be arriving: if every pending copy targets `table`, one launch per chunk
    // behind that chunk's event (Body::Args carries the chunk as i0 / n); otherwise the ordinary launch (which joins).
    template <class Body>
    bool run_simple_chunked(const typename Body::Args& a_in, uint64_t n, int cls, const void* table) {
        bool mine = !pending.empty();
        uint64_t covered = 0;
        for (auto& pc : pending) { mine = mine && pc.table == table && pc.lo == covered; covered = pc.hi; }
        if (!mine || covered != n) return run_simple<Body>(a_in, n, cls);
        std::vector<PendingCopy> chunks; chunks.swap(pending);          // tic() must not join what is waited on below
        tic(cls, 0);
        for (auto& pc : chunks) {
            typename Body::Args a = a_in;
            a.i0 = pc.lo; a.n = pc.hi - pc.lo;
            cudaStreamWaitEvent(stream, pc.ev, 0);
            sync_ev_free.push_back(pc.ev);
            k_simple<Body><<<grid_for(a.n), BLOCK, 0, stream>>>(a);
        }
        toc();
        return launched("k_simple (chunked)");
    }
    // ---- the range gadgets' three kernels, chunk by chunk behind a chunked input copy --------------------------------------------
    // For every chunk of the pending input copy: wait for it, decomposition (Pre), batch inversion and results (Post) of that instance
    // range, then an event: `results` lists, per variable table, which instance ranges are final behind which event, so that an
    // asynchronous whole-column read can be issued per chunk on the copy stream (col_read_chunked) and its device -> host copy runs
    // under the kernels of the later chunks.  Without a pending chunked copy of the operand: three launches over all instances.
    std::vector<PendingCopy> results;
    void drop_result_chunks() { for (auto& r : results) sync_ev_free.push_back(r.ev); results.clear(); }
    bool result_chunks_of(const void* table) const { for (auto& r : results) if (r.table == table) return true; return false; }
    template <class Pre, class Post>
    bool run_range_pipeline(const typename Pre::Args& a_in, const BatchInvArgs& inv_in, uint64_t n, const void* operand_table, const void* own_table,
                            bool chunk_results) {
        bool mine = !pending.empty();
        uint64_t covered = 0;
        for (auto& pc : pending) { mine = mine && pc.table == operand_table && pc.lo == covered; covered = pc.hi; }
        // Whole pipeline per chunk only when nothing long follows that would hide the result copy anyway (fused check): with a check
        // kernel behind it the copy runs under that kernel, and starting it earlier only makes it compete with the input copy for the
        // host's memory (measured: 278.0 -> 281.2 ms end to end in the generic mode, 29.9 -> 32.7 ms structure-aware; run r04l).
        if (!chunk_results || !mine || covered != n)
            return run_simple_chunked<Pre>(a_in, n, CLS_WITNESS, operand_table) && run_batch_inv(inv_in, CLS_WITNESS) && run_simple<Post>(a_in, n, CLS_WITNESS);
        std::vector<PendingCopy> chunks; chunks.swap(pending);          // tic() must not join what is waited on below
        for (auto& pc : chunks) {
            typename Pre::Args a = a_in;
            a.i0 = pc.lo; a.n = pc.hi - pc.lo;
            BatchInvArgs inv = inv_in;
            inv.fr = inv_in.fr + 2 * pc.lo; inv.n = a.n;
            cudaStreamWaitEvent(stream, pc.ev, 0);
            sync_ev_free.push_back(pc.ev);
            tic(CLS_WITNESS, 0);
            k_simple<Pre><<<grid_for(a.n), BLOCK, 0, stream>>>(a);
            toc();
            if (!launched("k_simple<RangePre> (chunk)") || !run_batch_inv(inv, CLS_WITNESS)) return false;
            tic(CLS_WITNESS, 0);
            k_simple<Post><<<grid_for(a.n), BLOCK, 0, stream>>>(a);
            toc();
            if (!launched("k_simple<RangePost> (chunk)")) return false;
            cudaEvent_t done = get_sync_event();
            PG_CUDA(cudaEventRecord(done, stream));
            results.push_back(PendingCopy{own_table, nullptr, pc.lo, pc.hi, done});
        }
        return true;
    }
    // whole-column asynchronous read of such a table: per chunk, on the copy stream, behind the chunk's event
    bool col_read_chunked(const ColReadBody::Args& whole, void* dst_host, const void* table) {
        for (auto& r : results) {
            if (r.table != table) continue;
            ColReadBody::Args a = whole;
            a.tab.fr = whole.tab.fr ? whole.tab.fr + 2 * r.lo : nullptr;
            a.tab.bits = whole.tab.bits ? whole.tab.bits + r.lo : nullptr;
            a.dst = whole.dst + 2 * r.lo; a.n = r.hi - r.lo;
            PG_CUDA(cudaStreamWaitEvent(copy_stream, r.ev, 0));
            k_simple<ColReadBody><<<grid_for(a.n), BLOCK, 0, copy_stream>>>(a);
            if (!launched("k_simple<ColReadBody> (chunk)")) return false;
            PG_CUDA(cudaMemcpyAsync((char*)dst_host + r.lo * sizeof(pg_fr), a.dst, a.n * sizeof(pg_fr), cudaMemcpyDeviceToHost, copy_stream));
        }
        return true;
    }
    bool d2h(void* dst, const void* src, size_t bytes) {
        join_copies();
        PG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream));
        PG_CUDA(cudaStreamSynchronize(stream));
        return true;
    }
    bool d2d(void* dst, const void* src, size_t bytes) { join_copies(); PG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, stream)); return true; }
    bool sync() { join_copies(); PG_CUDA(cudaStreamSynchronize(stream)); PG_CUDA(cudaStreamSynchronize(copy_stream)); return true; }
    // copy to (pinned) host memory on the copy stream, ordered after everything enqueued so far; complete after sync()
    bool d2h_async(void* dst, const void* src, size_t bytes) {
        join_copies();
        PG_CUDA(cudaEventRecord(copy_ready, stream));
        PG_CUDA(cudaStreamWaitEvent(copy_stream, copy_ready, 0));
        PG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, copy_stream));
        return true;
    }
    bool upload_pow2(const Fr* table) {
        PG_CUDA(cudaMemcpyToSymbolAsync(c_pow2, table, 256 * sizeof(Fr), 0, cudaMemcpyHostToDevice, stream));
        PG_CUDA(cudaStreamSynchronize(stream));
        return true;
    }

    // ---- timing --------------------------------------------------------------------------------------------------
    cudaEvent_t get_event() {
        if (!ev_free.empty()) { cudaEvent_t e = ev_free.back(); ev_free.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    void fold_events() {                         // resolve recorded event pairs into the accumulators (synchronises)
        cudaStreamSynchronize(stream);
        for (auto& ev : events) {
            float ms = 0.f; cudaEventElapsedTime(&ms, ev.a, ev.b);
            if (ev.cls == CLS_CHECK) { acc.check_ms += ms; acc.check_launches++; acc.check_rows += ev.rows; }
            else if (ev.cls == CLS_WITNESS) { acc.witness_ms += ms; acc.witness_launches++; }
            else { acc.other_ms += ms; acc.other_launches++; }
            ev_free.push_back(ev.a); ev_free.push_back(ev.b);
        }
        events.clear();
    }
    void tic(int cls, uint64_t rows) {
        join_copies();
        if (!timing_on) return;
        if (events.size() >= 4096) fold_events();    // bounded bookkeeping when nobody collects the timings
        Ev ev{get_event(), get_event(), cls, rows};
        cudaEventRecord(ev.a, stream);
        events.push_back(ev);
    }
    void toc() { if (timing_on) cudaEventRecord(events.back().b, stream); }
    bool timing(pg_timing* out, bool reset) {
        join_copies();
        PG_CUDA(cudaStreamSynchronize(stream));
        fold_events();
        *out = acc;
        if (reset) acc = pg_timing{};
        return true;
    }
    bool launched(const char* what) {
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { snprintf(errbuf, sizeof(errbuf), "%s launch: %s", what, cudaGetErrorString(e)); return false; }
        return true;
    }
    static unsigned grid_for(uint64_t n) { return (unsigned)((n + BLOCK - 1) / BLOCK); }

    // ---- launches ------------------------------------------------------------------------------------------------
    template <class Body>
    bool run_simple(const typename Body::Args& a, uint64_t n, int cls) {
        tic(cls, 0);
        k_simple<Body><<<grid_for(n), BLOCK, 0, stream>>>(a);
        toc();
        return launched("k_simple");
    }
    // bucket sums of the MSM: 128 threads x 3 blocks/SM (168 registers, no spills that matter) measured best; PG_MSM_SHAPE selects
    // the alternatives for tuning runs (profiles/README.md)
    int msm_shape = -1;
    bool run_msm_buckets(const MsmBucketBody::Args& a) {
        if (msm_shape < 0) { const char* e = getenv("PG_MSM_SHAPE"); msm_shape = e ? atoi(e) : 1; }
        tic(CLS_OTHER, 0);
        switch (msm_shape) {
            case 1: k_simple_shaped<MsmBucketBody, 128, 3><<<(unsigned)((a.n + 127) / 128), 128, 0, stream>>>(a); break;    // <=168 regs, 12 warps/SM
            case 2: k_simple_shaped<MsmBucketBody, 128, 4><<<(unsigned)((a.n + 127) / 128), 128, 0, stream>>>(a); break;    // <=128 regs, 16 warps/SM
            case 3: k_simple_shaped<MsmBucketBody, 128, 5><<<(unsigned)((a.n + 127) / 128), 128, 0, stream>>>(a); break;    // <=96 regs, 20 warps/SM
            default: k_simple<MsmBucketBody><<<grid_for(a.n), BLOCK, 0, stream>>>(a); break;
        }
        toc();
        return launched("k_simple<MsmBucketBody>");
    }
    // One wave: the elements are divided over the blocks that are resident together (sm_count x 2 blocks/SM), so every block
    // streams its share twice and inverts once (3 and 4 blocks/SM measured within 3 %: profiles/r03c_batch_inv_shapes.log).
    template <class Hook>
    bool run_batch_inv_fused(const BatchInvArgs& a_in, const typename Hook::Args& h, int cls) {
        BatchInvArgs a = a_in;
        const uint64_t total = (uint64_t)a.n_pairs * a.n;
        if (!total) return true;
        const uint64_t resident = (uint64_t)sm_count * 2 * BLOCK;
        const uint64_t e = (total + resident - 1) / resident;
        a.elems_per_thread = (uint32_t)(e < 8 ? 8 : e);
        const uint64_t per_block = (uint64_t)BLOCK * a.elems_per_thread;
        tic(cls, 0);
        k_batch_inv<Hook><<<(unsigned)((total + per_block - 1) / per_block), BLOCK, 0, stream>>>(a, h);
        toc();
        return launched("k_batch_inv");
    }
    bool run_batch_inv(const BatchInvArgs& a, int cls) { return run_batch_inv_fused<InvPlain>(a, InvPlain::Args{}, cls); }
    // which kernel evaluated how many rows (pg_get_check_stats): the tests use it to prove that a verdict came from the kernel they mean
    pg_check_stats ck{};
    void count_check(int kind, uint64_t rows) { ck.launches[kind]++; ck.rows[kind] += rows; }
    bool run_check(const CheckArgs& a, const SparseProg& prog) {
        const size_t smem = (size_t)a.n_pool * sizeof(Fr);
        if (smem > 64 * 1024) { snprintf(errbuf, sizeof(errbuf), "selector pool of %u entries exceeds the shared-memory budget", a.n_pool); return false; }
        tic(CLS_CHECK, a.n_inst * a.n_rows);
        if (a.n_inst < (uint64_t)sm_count * 320 && a.n_rows > 1) {      // fewer instances than half the resident threads: one thread per row
            const uint64_t total = a.n_inst * a.n_rows;
            const unsigned grid = (unsigned)((total + 127) / 128);
            if (a.mode == PG_CHECK_SPARSE) k_check_rowpar<1><<<grid, 128, smem, stream>>>(a); else k_check_rowpar<0><<<grid, 128, smem, stream>>>(a);
            toc();
            count_check(PG_CK_ROWPAR, total);
            return launched("k_check_rowpar");
        }
        // the structure-aware check streams the table (HBM-bound): 20 warps/SM with three 32-byte loads in flight per thread (no register
        // spill, no local memory) and 24 warps/SM with four measure the same, 12.95 / 12.98 ms (profiles/README.md, run r04n)
        switch (check_shape) {
            case 1: launch_check<1>(a, prog, smem); break; case 2: launch_check<2>(a, prog, smem); break;
            case 3: launch_check<3>(a, prog, smem); break; case 4: launch_check<4>(a, prog, smem); break;
            default: launch_check<0>(a, prog, smem); break;
        }
        toc();
        count_check(a.mode != PG_CHECK_SPARSE ? PG_CK_INSTANCE_GENERIC : prog.ops ? PG_CK_PROGRAM : PG_CK_INSTANCE_TERMS, a.n_inst * a.n_rows);
        return launched("k_check");
    }
    bool run_check_gates(const CheckArgs& a) {
        const size_t smem = (size_t)a.n_pool * sizeof(Fr);
        if (smem > 48 * 1024) { snprintf(errbuf, sizeof(errbuf), "selector pool of %u entries exceeds the shared-memory budget", a.n_pool); return false; }
        const uint64_t total = a.n_inst * a.n_rows;
        tic(CLS_CHECK, total);
        // Large segments in the structure-aware mode: one thread per instance walking the rows (every accumulator loaded once; 7.2 vs
        // 8.1 ms at 2^24 x 64 bits).  In the generic mode the (row, instance) mapping stays: the walk measured 18.8 vs 18.1 ms -- the range
        // rows are bound by their multiplications either way (profiles/README.md, run r04k).  PG_GATES_WALK=0/1 overrides (tuning runs).
        static const int walk_env = getenv("PG_GATES_WALK") ? atoi(getenv("PG_GATES_WALK")) : -1;
        const bool walk = walk_env >= 0 ? walk_env != 0 : a.mode == PG_CHECK_SPARSE;
        if (walk && a.n_inst >= (uint64_t)sm_count * 320) {
            k_check_gates_walk<<<(unsigned)((a.n_inst + 127) / 128), 128, smem, stream>>>(a);
            toc();
            count_check(PG_CK_GATES, total);
            return launched("k_check_gates_walk");
        }
        const unsigned grid = (unsigned)((total + 127) / 128);
        switch (check_shape) {                                   // 20 / 24 / 28 warps per SM measure the same (18.16 / 18.05 / 18.26 ms, run r04j)
            case 2: k_check_gates<6><<<grid, 128, smem, stream>>>(a); break;
            case 3: k_check_gates<7><<<grid, 128, smem, stream>>>(a); break;
            default: k_check_gates<5><<<grid, 128, smem, stream>>>(a); break;
        }
        toc();
        count_check(PG_CK_GATES, total);
        return launched("k_check_gates");
    }
    bool run_mat_tiled(const MatTileArgs& a) {
        const uint64_t tiles = ((a.n_inst + MT_I - 1) / MT_I) * ((a.seg.n_rows + MT_R - 1) / MT_R);
        tic(CLS_OTHER, 0);
        k_materialize_tiled<<<(unsigned)tiles, BLOCK, 0, stream>>>(a);
        toc();
        return launched("k_materialize_tiled");
    }
    bool exclusive_sum(const uint32_t* in, uint32_t* out, uint64_t n) {
        size_t need = 0;
        PG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, need, in, out, (long long)n, stream));
        if (need > sort_tmp_bytes) {
            if (sort_tmp) { PG_CUDA(cudaStreamSynchronize(stream)); cudaFree(sort_tmp); sort_tmp = nullptr; sort_tmp_bytes = 0; }
            PG_CUDA(cudaMalloc(&sort_tmp, need));
            sort_tmp_bytes = need;
        }
        tic(CLS_OTHER, 0);
        PG_CUDA(cub::DeviceScan::ExclusiveSum(sort_tmp, need, in, out, (long long)n, stream));
        toc();
        return launched("cub::DeviceScan::ExclusiveSum");
    }
    // radix sort of (key, value) pairs by the low key_bits of the key (CUB; temporary storage kept for the context's lifetime)
    void* sort_tmp = nullptr; size_t sort_tmp_bytes = 0;
    bool sort_pairs(const uint32_t* keys, const uint32_t* vals, uint32_t* keys_out, uint32_t* vals_out, uint64_t n, uint32_t key_bits) {
        size_t need = 0;
        PG_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, keys, keys_out, vals, vals_out, (long long)n, 0, (int)key_bits, stream));
        if (need > sort_tmp_bytes) {
            if (sort_tmp) { PG_CUDA(cudaStreamSynchronize(stream)); cudaFree(sort_tmp); sort_tmp = nullptr; sort_tmp_bytes = 0; }
            PG_CUDA(cudaMalloc(&sort_tmp, need));
            sort_tmp_bytes = need;
        }
        tic(CLS_OTHER, 0);
        PG_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp, need, keys, keys_out, vals, vals_out, (long long)n, 0, (int)key_bits, stream));
        toc();
        return launched("cub::DeviceRadixSort::SortPairs");
    }
    bool run_ntt_pass(const NttPassArgs& a, uint64_t n_blocks) {
        const size_t smem = (size_t)32 << (a.s + a.log_c);
        tic(CLS_OTHER, 0);
        if (a.shift) k_ntt_coset_pass<<<(unsigned)n_blocks, NTT_THREADS, smem, stream>>>(a);
        else if (a.inverse) k_ntt_pass<true><<<(unsigned)n_blocks, NTT_THREADS, smem, stream>>>(a);
        else k_ntt_pass<false><<<(unsigned)n_blocks, NTT_THREADS, smem, stream>>>(a);
        toc();
        return launched(a.shift ? "k_ntt_coset_pass" : "k_ntt_pass");
    }
    // exclusive prefix product (scan.cuh) of n scalars; *total = product of all; scratch: fr_scan_scratch(n) scalars
    bool run_fr_scan(const uint4* in, uint4* out, uint64_t n, uint4* total, uint4* scratch) {
        if (!n) return true;
        tic(CLS_OTHER, 0);
        const bool ok = fr_scan_level(in, out, n, total, scratch);
        toc();
        return ok;
    }
    bool fr_scan_level(const uint4* in, uint4* out, uint64_t n, uint4* total, uint4* scratch) {
        if (n <= SCAN_TILE) {
            k_fr_scan_apply<<<1, SCAN_THREADS, 0, stream>>>(in, out, n, nullptr, total);
            return launched("k_fr_scan_apply");
        }
        const uint64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
        k_fr_scan_reduce<<<(unsigned)tiles, SCAN_THREADS, 0, stream>>>(in, n, scratch);
        if (!launched("k_fr_scan_reduce")) return false;
        if (!fr_scan_level(scratch, scratch, tiles, total, scratch + 2 * tiles)) return false;      // tile totals -> their exclusive prefixes
        k_fr_scan_apply<<<(unsigned)tiles, SCAN_THREADS, 0, stream>>>(in, out, n, scratch, nullptr);
        return launched("k_fr_scan_apply");
    }
    // Ruffini division (scan.cuh) of n scalars by (X - p): out[i] = s_(i+1), *rem = f(p); pw: fr_ruffini_levels(n) tables of RUF_TAB
    // powers (level l: of p^(SCAN_TILE^l)); scratch: fr_scan_scratch(n) scalars
    bool run_fr_ruffini(const uint4* in, uint4* out, uint64_t n, const uint4* pw, uint4* rem, uint4* scratch) {
        if (!n) return true;
        tic(CLS_OTHER, 0);
        const bool ok = fr_ruffini_level(in, out, n, pw, rem, scratch);
        toc();
        return ok;
    }
    bool fr_ruffini_level(const uint4* in, uint4* out, uint64_t n, const uint4* pw, uint4* rem, uint4* scratch) {
        if (n <= SCAN_TILE) {
            k_fr_ruffini_apply<<<1, SCAN_THREADS, 0, stream>>>(in, out, n, pw, nullptr, rem);
            return launched("k_fr_ruffini_apply");
        }
        const uint64_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
        k_fr_ruffini_reduce<<<(unsigned)tiles, SCAN_THREADS, 0, stream>>>(in, n, pw, scratch);
        if (!launched("k_fr_ruffini_reduce")) return false;
        if (!fr_ruffini_level(scratch, scratch, tiles, pw + 2 * RUF_TAB, rem, scratch + 2 * tiles)) return false;   // tile values -> their carries
        k_fr_ruffini_apply<<<(unsigned)tiles, SCAN_THREADS, 0, stream>>>(in, out, n, pw, scratch, nullptr);
        return launched("k_fr_ruffini_apply");
    }
    bool run_check_rows(const CheckRowsBody::Args& a) {
        tic(CLS_CHECK, a.n);
        k_check_rows<<<grid_for(a.n), BLOCK, 0, stream>>>(a);
        toc();
        return launched("k_check_rows");
    }
    // ---- collectives (comm.cuh); without a communicator: a world of one rank, no NCCL ----------------------------------------------
    Comm comm;
    unsigned long long* d_verdict = nullptr;
    const char* comm_error() const { return comm.err[0] ? comm.err : errbuf; }
    int comm_rank() const { return comm.rank; }
    int comm_world() const { return comm.world; }
    static bool comm_unique_id(uint8_t* id) {
        NcclApi& api = nccl_api();
        if (const char* e = api.load()) { fprintf(stderr, "pg_comm_unique_id: %s\n", e); return false; }
        ncclUniqueId uid;
        if (api.GetUniqueId(&uid) != ncclSuccess) return false;
        memcpy(id, &uid, sizeof(uid));
        return true;
    }
    bool comm_init(const uint8_t* id, int rank, int world) { join_copies(); if (comm.active()) comm.destroy(); return comm.init(id, rank, world); }
    void comm_destroy() { comm.destroy(); }
    bool comm_verdict(const unsigned long long* d_counters, unsigned long long n_err, unsigned long long out[4], const FusedSpan* d_map, uint32_t n_map) {
        join_copies();
        if (comm.active()) return comm.allreduce_verdict(d_counters, n_err, out, d_map, n_map, stream);
        if (!d_verdict) PG_CUDA(cudaMalloc(&d_verdict, 4 * sizeof(unsigned long long)));
        k_verdict_pack<<<1, 1, 0, stream>>>(d_counters, n_err, d_verdict, d_map, n_map);
        PG_CUDA(cudaMemcpyAsync(out, d_verdict, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
        PG_CUDA(cudaStreamSynchronize(stream));
        return true;
    }
    bool comm_counts(unsigned long long mine, unsigned long long* counts) {
        join_copies();
        if (comm.active()) return comm.allgather_u64(mine, counts, stream);
        counts[0] = mine;
        return true;
    }
    bool comm_gather(const void* send, void* recv, const unsigned long long* counts) {
        tic(CLS_OTHER, 0);
        bool ok = true;
        if (comm.active()) ok = comm.allgather_ragged(send, recv, counts, stream);
        else if (cudaMemcpyAsync(recv, send, (size_t)counts[0] * 32, cudaMemcpyDeviceToDevice, stream) != cudaSuccess) { snprintf(errbuf, sizeof(errbuf), "gather copy"); ok = false; }
        toc();
        return ok;
    }
    template <int MODE>
    void ubench_launch(uint32_t* buf, int blocks, int iters, int rep) { k_ubench<MODE><<<blocks, BLOCK, 0, stream>>>(buf, 12345u + rep, 0x9e3779b1u, iters); }
    // operations per second of one micro-benchmark mode (best of 3 after a warm-up launch)
    bool ubench(int mode, double* ops_per_s) {
        if (mode < 0 || mode >= UB_MODES) { snprintf(errbuf, sizeof(errbuf), "unknown micro-benchmark mode %d", mode); return false; }
        const int blocks = sm_count * 8, iters = (mode >= UB_FR_MUL && mode <= UB_FR_ADD) ? 512 : 4096;
        uint32_t* buf = nullptr;
        PG_CUDA(cudaMalloc(&buf, (size_t)blocks * BLOCK * sizeof(uint32_t)));
        cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
        double best = 0;
        for (int rep = 0; rep < 4; rep++) {
            cudaEventRecord(a, stream);
            switch (mode) {
                case 0: ubench_launch<0>(buf, blocks, iters, rep); break; case 1: ubench_launch<1>(buf, blocks, iters, rep); break;
                case 2: ubench_launch<2>(buf, blocks, iters, rep); break; case 3: ubench_launch<3>(buf, blocks, iters, rep); break;
                case 4: ubench_launch<4>(buf, blocks, iters, rep); break; case 5: ubench_launch<5>(buf, blocks, iters, rep); break;
                case 6: ubench_launch<6>(buf, blocks, iters, rep); break; case 7: ubench_launch<7>(buf, blocks, iters, rep); break;
                case 8: ubench_launch<8>(buf, blocks, iters, rep); break;
                case 9: ubench_launch<9>(buf, blocks, iters, rep); break;
                default: ubench_launch<10>(buf, blocks, iters, rep); break;
            }
            cudaEventRecord(b, stream);
            cudaEventSynchronize(b);
            float ms = 0.f; cudaEventElapsedTime(&ms, a, b);
            const double ops = (double)blocks * BLOCK * (double)iters * ubench_ops_per_iter(mode);
            if (rep > 0 && ms > 0.f && ops / (ms * 1e-3) > best) best = ops / (ms * 1e-3);
        }
        cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(buf);
        if (!launched("k_ubench")) return false;
        *ops_per_s = best;
        return true;
    }
    bool imad_peak(double* wide, double* lo) { return ubench(UB_WIDE_ACC, wide) && ubench(UB_IMAD_LO, lo); }
};

static_assert(has_fr_scan<CudaBackend>::value, "the shipped library computes the grand product with the device-wide scan of scan.cuh");
static_assert(has_fr_ruffini<CudaBackend>::value, "the shipped library divides the opening aggregates with the device-wide Ruffini scan of scan.cuh");

}  // namespace pg

#define PG_BACKEND pg::CudaBackend
#include "capi.inl"
