// Context internals shared by capi.cu and msm.cu. A jb_ctx is the device half of the
// reference's ProofSession (crates/jolt-kernels/src/backend.rs:283-286).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/jolt_b200.h"

constexpr int JB_MAX_EVALS = 8;                 // evaluations per work item of the scheduler ABI: degree + 1 <= 8
constexpr size_t JB_SMALL_BYTES = 4096;         // staging for round evaluations / points
constexpr int JB_RESULT_SLOTS = 16;             // host-mapped round-result slots (1 KiB each; slot 0 = in-place rounds)

struct Table {
    uint64_t* buf = nullptr;  // current data (len elements)
    size_t cap = 0;           // capacity of buf in elements
    size_t len = 0;
    uint64_t* alt = nullptr;  // ping-pong scratch for LowToHigh binds
    size_t alt_cap = 0;
    bool buf_owned = true;    // false: caller's device memory (jb_table_wrap_device)
    bool alt_owned = true;
    void swap_buffers() {
        uint64_t* b = buf; buf = alt; alt = b;
        size_t c = cap; cap = alt_cap; alt_cap = c;
        bool o = buf_owned; buf_owned = alt_owned; alt_owned = o;
    }
};

struct Srs {
    uint64_t* xy = nullptr;  // n affine points, 8 limbs each (x, y), identity = all zero
    size_t n = 0;
    // optional: rows w = 0..pre_W-1 of 2^(pre_c * w) * P_i (affine), row stride n points (jb_srs_precompute)
    uint64_t* pre = nullptr;
    int pre_c = 0, pre_W = 0;
    // second table for small MSMs: 8-bit windows over the first pre_small_len bases (row stride pre_small_len)
    uint64_t* pre_small = nullptr;
    size_t pre_small_len = 0;
};

struct MsmWorkspace;  // msm.cu
struct ResidentRun;   // resident.cu: one launched resident_rounds_kernel and the members it serves

// Host-mapped mailbox + device state + private stream + event for one resident kernel; pooled per context so
// a batch entering resident service pays no allocation (cudaHostAlloc / stream creation cost tens of microseconds).
struct TailRes {
    void* mb_host = nullptr;
    void* mb_dev = nullptr;
    void* d_state = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t event = nullptr;
};

// Optional per-launch CUDA-event timing of the dominant kernels (bench.py's roofline figure is
// measured live, on this stream, inside the timed region).
struct TimedLaunch {
    cudaEvent_t e0 = nullptr, e1 = nullptr;  // null: a pass inside a resident kernel, timed by the device (ms_direct)
    double ms_direct = 0;
    int kind;        // 0 = fused bind+eval, 1 = bind, 2 = eval-only, 3 = eq, 4 = msm bucket accumulation
    uint64_t items;  // pairs / outputs / terms
    int m;
};

struct jb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    int sm_count = 148;
    std::mutex mu;
    std::unordered_map<uint64_t, Table> tables;
    std::unordered_map<uint64_t, Srs> srs;
    uint64_t next_id = 1;
    std::string err;
    uint64_t launches = 0;
    uint64_t* d_partial = nullptr;  // per-block partial sums of the running fused pass
    size_t partial_cap = 0;         // in elements
    std::vector<TailRes> tail_pool;
    uint64_t diag_wait_ns = 0, diag_waits = 0;  // host time spent waiting for round results
    bool use_tail = true;           // resident kernel service (off under profilers / JB_NO_TAIL: one launch per round)
    long long resident_timeout_cycles = 20000000000LL;  // a resident kernel gives its SMs back after this long without a command
    std::vector<ResidentRun*> runs; // live resident kernels of this context
    // diagnostics: per round of the last completed run: device %globaltimer at command decode / after the fold,
    // host CLOCK_MONOTONIC at post / at receipt (ns)
    uint64_t last_run_log[8 * 64] = {0};
    size_t last_run_rounds = 0;
    // Stops resident kernels that would starve other work of SMs (an exclusive run holds every block slot of the
    // device): called by every entry point that launches or waits on the context's stream. `all`: also the small
    // (<= half the device) runs. The members they served continue with one launch per round.
    void quiesce_resident(bool all = false);
    bool has_exclusive_run() const;
    bool verify_rounds = false;     // compute s(1) and check s(0)+s(1)==claim instead of deriving s(1)
    uint64_t* d_small = nullptr;    // device staging
    uint64_t* h_small = nullptr;    // pinned host staging
    // zero-copy round results: pinned + mapped; JB_RESULT_SLOTS slots of 128 u64: [0, 64) results, [64] sequence flag
    uint64_t* h_result = nullptr;
    uint64_t* d_result_alias = nullptr;  // device address of h_result
    unsigned int* d_counter = nullptr;   // last-block ticket counter (zero between launches)
    uint64_t result_seq = 0;
    MsmWorkspace* msm = nullptr;
    // multi-GPU (comm.cu): NCCL communicator + the lanes buffer the per-round all-reduce runs on
    void* nccl_comm = nullptr;
    int world = 1, rank = 0;
    uint64_t* d_lanes = nullptr;
    // peer-memory exchange (fused all-reduce in the round kernel's epilogue): every rank's buffer mapped here
    uint64_t* xch_peer[16] = {nullptr};
    bool xch_ready = false;
    uint64_t xch_seq = 0;
    uint64_t gather_seq = 0;  // gathers through the arena that follows the exchange area (parity = arena half)
    int comm_allreduce_lanes(uint64_t* d_lanes_buf, size_t n_u64);
    int comm_allgather(const uint64_t* d_send, uint64_t* d_recv, size_t n_u64_per_rank);
    int publish_lanes(const uint64_t* d_lanes_buf, int n_u64);
    bool timing = false;
    uint64_t timing_min_items = 0;
    std::vector<TimedLaunch> timed;

    // returns an index into `timed` (or -1): call before the launch, then timing_end(idx) after it
    int timing_begin(int kind, uint64_t items, int m) {
        if (!timing || items < timing_min_items || timed.size() >= 4096) return -1;
        TimedLaunch t;
        t.kind = kind; t.items = items; t.m = m;
        if (cudaEventCreate(&t.e0) != cudaSuccess || cudaEventCreate(&t.e1) != cudaSuccess) return -1;
        cudaEventRecord(t.e0, stream);
        timed.push_back(t);
        return (int)timed.size() - 1;
    }
    void timing_end(int idx) {
        if (idx >= 0) cudaEventRecord(timed[idx].e1, stream);
    }

    // cudaSetDevice is not free (a runtime lock + context check per call): skip it when this thread is
    // already on the context's device - it sits on the per-round latency path.
    void make_current() {
        int current = -1;
        if (cudaGetDevice(&current) != cudaSuccess || current != device) cudaSetDevice(device);
    }
    int fail(int status, const char* what) {
        err = what;
        return status;
    }
    int check(cudaError_t e, const char* what) {
        if (e == cudaSuccess) return JB_OK;
        err = std::string(what) + ": " + cudaGetErrorString(e);
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? JB_ERR_OOM : JB_ERR_CUDA;
    }
    int dev_alloc(void** p, size_t bytes) {
        cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 32, stream);
        if (e != cudaSuccess) {
            *p = nullptr;
            err = std::string("device allocation failed: ") + cudaGetErrorString(e);
            cudaGetLastError();
            return JB_ERR_OOM;
        }
        return JB_OK;
    }
    void dev_free(void* p) {
        if (p) cudaFreeAsync(p, stream);
    }
    Table* find(uint64_t h) {
        auto it = tables.find(h);
        return it == tables.end() ? nullptr : &it->second;
    }
    int ensure_alt(Table& t, size_t elems) {
        if (t.alt && t.alt_cap >= elems) return JB_OK;
        if (t.alt && t.alt_owned) dev_free(t.alt);
        t.alt = nullptr;
        t.alt_cap = 0;
        t.alt_owned = true;
        int st = dev_alloc((void**)&t.alt, elems * 32);
        if (st == JB_OK) t.alt_cap = elems;
        return st;
    }
    int ensure_partial(size_t elems) {
        if (elems <= partial_cap) return JB_OK;
        if (d_partial) dev_free(d_partial);
        d_partial = nullptr;
        partial_cap = 0;
        size_t want = elems < 8192 ? 8192 : elems;
        int st = dev_alloc((void**)&d_partial, want * 32);
        if (st == JB_OK) partial_cap = want;
        return st;
    }
    void release(Table& t) {
        if (t.buf && t.buf_owned) dev_free(t.buf);
        if (t.alt && t.alt_owned) dev_free(t.alt);
        t.buf = t.alt = nullptr;
    }
    void msm_release();
};

// Serialises a context's entry points (a context = one ProofSession; Rayon threads may call msm concurrently,
// crates/jolt-hyperkzg/src/scheme.rs:141-145). keep_resident: the caller is the resident round path itself.
struct CtxGuard {
    jb_ctx* c;
    std::lock_guard<std::mutex> lk;
    explicit CtxGuard(jb_ctx* ctx, bool keep_resident = false) : c(ctx), lk(ctx->mu) {
        ctx->make_current();
        if (!keep_resident && !ctx->runs.empty()) ctx->quiesce_resident(false);
    }
};

namespace jb {
// msm.cu: commitments of HyperKZG's packed folded polynomials (lengths 2^(h-1) .. 2) in one pipeline pass
int msm_halving_rows_device(jb_ctx* c, uint64_t srs, const uint64_t* d_scalars, int h, uint64_t* out_xyz);
}  // namespace jb
