// Host side of the resident kernel service (resident.cuh): start a run for a batch of members, drive one round
// per mailbox command, stop it. The context lock is held by every caller.
#include "../../include/jolt_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <new>

#include "member.hpp"
#include "resident.cuh"

using namespace jb;
using namespace jbi;

namespace {

using ResKernel = void (*)(const ResArgs);

template <int D, int P>
ResKernel pick_order(int order) {
    return order == JB_HIGH_TO_LOW ? (ResKernel)resident_rounds_kernel<D, P, ORDER_HIGH_TO_LOW>
                                   : (ResKernel)resident_rounds_kernel<D, P, ORDER_LOW_TO_HIGH>;
}

// The instantiated shapes: plain products of 1..4 tables and the two-term degree-2 sum of products
// (IncClaimReduction: A * RamInc + B * RdInc).
ResKernel pick_kernel(int D, int P, int order, size_t* smem) {
    *smem = 0;
    if (P == 1) {
        switch (D) {
            case 1: *smem = FusedShape<1, true>::smem_bytes(RES_BLOCK); return pick_order<1, 1>(order);
            case 2: *smem = FusedShape<2, true>::smem_bytes(RES_BLOCK); return pick_order<2, 1>(order);
            case 3: *smem = FusedShape<3, true>::smem_bytes(RES_BLOCK); return pick_order<3, 1>(order);
            case 4: *smem = FusedShape<4, true>::smem_bytes(RES_BLOCK); return pick_order<4, 1>(order);
            default: return nullptr;
        }
    }
    if (P == 2 && D == 2) {
        *smem = FusedShape<2, true>::smem_bytes(RES_BLOCK);
        return pick_order<2, 2>(order);
    }
    return nullptr;
}

// occupancy of a shape (cached): also forces the module to load before any resident kernel is alive
int kernel_blocks_per_sm(ResKernel k, size_t smem) {
    static std::mutex mu;
    static std::vector<std::pair<ResKernel, int>> cache;
    std::lock_guard<std::mutex> lk(mu);
    for (auto& kv : cache)
        if (kv.first == k) return kv.second;
    cudaFuncSetAttribute((const void*)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, (const void*)k, RES_BLOCK, smem) != cudaSuccess || nb < 1) nb = 1;
    cache.emplace_back(k, nb);
    return nb;
}

int acquire_resources(jb_ctx* c, TailRes* r) {
    if (!c->tail_pool.empty()) {
        *r = c->tail_pool.back();
        c->tail_pool.pop_back();
        return JB_OK;
    }
    TailRes t;
    if (cudaHostAlloc(&t.mb_host, sizeof(ResMailbox), cudaHostAllocMapped) != cudaSuccess ||
        cudaHostGetDevicePointer(&t.mb_dev, t.mb_host, 0) != cudaSuccess ||
        cudaMalloc(&t.d_state, sizeof(ResState)) != cudaSuccess ||
        cudaStreamCreateWithFlags(&t.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&t.event, cudaEventDisableTiming) != cudaSuccess) {
        if (t.mb_host) cudaFreeHost(t.mb_host);
        if (t.d_state) cudaFree(t.d_state);
        if (t.stream) cudaStreamDestroy(t.stream);
        if (t.event) cudaEventDestroy(t.event);
        cudaGetLastError();
        return c->fail(JB_ERR_OOM, "resident: mailbox / stream allocation failed");
    }
    *r = t;
    return JB_OK;
}

// Spins until the kernel has answered command `seq`. Slow path: make sure the kernel is still alive.
int wait_answer(ResidentRun* run, uint64_t seq) {
    jb_ctx* c = run->c;
    ResMailbox* mb = run->mb;
    uint64_t spins = 0;
    volatile uint64_t* flag = &mb->ans[seq & 1].res_seq;
    while (__atomic_load_n(flag, __ATOMIC_ACQUIRE) != seq) {
        if ((++spins & 0x3fffff) == 0) {
            cudaError_t e = cudaStreamQuery(run->res.stream);
            if (e != cudaErrorNotReady && __atomic_load_n(flag, __ATOMIC_ACQUIRE) != seq) {
                run->kernel_live = false;
                return c->check(e == cudaSuccess ? cudaErrorUnknown : e, "resident kernel exited without answering");
            }
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    return JB_OK;
}

void release_run(ResidentRun* run, bool mark_no_resident) {
    jb_ctx* c = run->c;
    {
        const uint64_t nseq = run->seq < 64 ? run->seq : 64;
        for (uint64_t s = 0; s < nseq; ++s) {
            c->last_run_log[8 * s] = run->mb->tlog[2 * s];
            c->last_run_log[8 * s + 1] = run->mb->tlog[2 * s + 1];
            c->last_run_log[8 * s + 2] = run->host_post[s];
            c->last_run_log[8 * s + 3] = run->host_recv[s];
            for (int k = 0; k < 4; ++k) c->last_run_log[8 * s + 4 + k] = run->mb->tlog2[4 * s + k];
        }
        c->last_run_rounds = nseq;
    }
    if (c->timing) {  // the passes of this run, timed on the device (%globaltimer), as launch-like records
        const uint64_t nseq = run->seq < 64 ? run->seq : 64;
        for (uint64_t s = 0; s < nseq; ++s) {
            const ResidentRun::RoundInfo& ri = run->info[s];
            const uint64_t t0 = run->mb->tlog[2 * s], t1 = run->mb->tlog[2 * s + 1];
            if (ri.kind < 0 || ri.items < c->timing_min_items || t1 <= t0 || c->timed.size() >= 4096) continue;
            TimedLaunch t;
            t.kind = ri.kind;
            t.items = ri.items;
            t.m = ri.m;
            t.ms_direct = (double)(t1 - t0) * 1e-6;
            c->timed.push_back(t);
        }
    }
    // later work on the context's stream is ordered after the kernel's exit
    cudaEventRecord(run->res.event, run->res.stream);
    cudaStreamWaitEvent(c->stream, run->res.event, 0);
    for (auto& t : run->deferred) c->release(t);
    c->tail_pool.push_back(run->res);
    for (int i = 0; i < run->n; ++i) {
        if (run->mem[i]) {
            run->mem[i]->run = nullptr;
            if (mark_no_resident) run->mem[i]->no_resident = true;
        }
    }
    auto it = std::find(c->runs.begin(), c->runs.end(), run);
    if (it != c->runs.end()) c->runs.erase(it);
    delete run;
}

}  // namespace

bool resident_eligible(const jb_member* mem) {
    if (!mem || !mem->ctx->use_tail || mem->eq || mem->run) return false;
    if (mem->len < 2 || (mem->len & (mem->len - 1))) return false;
    // a member whose big run had to make room for other work only re-enters service once its run is small
    if (mem->no_resident && mem->len > RES_SMALL_LEN) return false;
    size_t smem;
    return pick_kernel(mem->m, mem->terms, mem->order, &smem) != nullptr;
}

bool jb_ctx::has_exclusive_run() const {
    for (auto* r : runs)
        if (r->exclusive) return true;
    return false;
}

void jb_ctx::quiesce_resident(bool all) {
    std::vector<ResidentRun*> copy = runs;
    for (auto* r : copy)
        if (all || r->exclusive) resident_end(r, true);
}

int resident_begin(jb_ctx* c, jb_member** mems, int n, uint64_t first_len, bool may_evict) {
    if (n < 1 || n > RES_MAX_MEMBERS) return JB_ERR_UNSUPPORTED;
    const int D = mems[0]->m, P = mems[0]->terms, order = mems[0]->order, T = D * P;
    for (int i = 0; i < n; ++i) {
        jb_member* m = mems[i];
        if (m->ctx != c || m->m != D || m->terms != P || m->order != order || !resident_eligible(m)) return JB_ERR_UNSUPPORTED;
    }
    size_t smem = 0;
    ResKernel kernel = pick_kernel(D, P, order, &smem);
    if (!kernel) return JB_ERR_UNSUPPORTED;
    const int per_sm = kernel_blocks_per_sm(kernel, smem);
    const unsigned cap = (unsigned)(c->sm_count * per_sm);
    unsigned grid = 1;
    for (int i = 0; i < n; ++i) {
        // the largest pass member i can ask for: over first_len entries if the caller knows its first round binds
        const uint64_t len0 = (first_len && n == 1) ? first_len : mems[i]->len;
        grid = std::max(grid, res_need_blocks(D, P, len0, cap));
    }
    const bool exclusive = grid > (unsigned)c->sm_count;
    // co-residency budget: small runs may share the device, a big one needs it alone
    unsigned in_use = 0;
    for (auto* r : c->runs) in_use += r->grid;
    if (!c->runs.empty() && (exclusive || c->has_exclusive_run() || in_use + grid > (unsigned)c->sm_count)) {
        if (!may_evict) return JB_ERR_UNSUPPORTED;  // (other runs may have commands in flight)
        c->quiesce_resident(true);
    }

    ResidentRun* run = new (std::nothrow) ResidentRun();
    if (!run) return JB_ERR_OOM;
    run->c = c;
    run->n = n;
    run->grid = grid;
    run->exclusive = exclusive;
    int st = acquire_resources(c, &run->res);
    if (st != JB_OK) {
        delete run;
        return st;
    }
    run->mb = (ResMailbox*)run->res.mb_host;
    ResArgs args;
    std::memset(&args, 0, sizeof args);
    args.n_members = n;
    for (int i = 0; i < n && st == JB_OK; ++i) {
        jb_member* m = mems[i];
        args.mem[i].len = m->len;
        for (int j = 0; j < T && st == JB_OK; ++j) {
            Table& t = m->tables[j];
            if (order == JB_LOW_TO_HIGH) st = c->ensure_alt(t, m->len / 2 ? m->len / 2 : 1);
            args.mem[i].buf[j] = t.buf;
            args.mem[i].alt[j] = t.alt;
        }
    }
    if (st != JB_OK) {
        c->tail_pool.push_back(run->res);
        delete run;
        return st;
    }
    std::memset(run->mb, 0, sizeof(ResMailbox));
    args.mb = (ResMailbox*)run->res.mb_dev;
    args.st = (ResState*)run->res.d_state;
    args.timeout_cycles = c->resident_timeout_cycles;  // ~10 s of SM clocks without a command: give the SMs back
    args.static_pct = RES_STATIC_PCT;
    args.world = c->world;
    args.rank = c->rank;
    for (int g = 0; g < 16; ++g) args.peer[g] = c->xch_peer[g];
    // the kernel starts after everything already queued on the context's stream (uploads, allocations)
    cudaEventRecord(run->res.event, c->stream);
    cudaStreamWaitEvent(run->res.stream, run->res.event, 0);
    cudaMemsetAsync(run->res.d_state, 0, sizeof(ResState), run->res.stream);
    void* kargs[] = {(void*)&args};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)kernel, dim3(grid), dim3(RES_BLOCK), kargs, smem, run->res.stream);
    c->launches++;
    if (e != cudaSuccess) {
        st = c->check(e, "resident_rounds_kernel launch");
        c->tail_pool.push_back(run->res);
        delete run;
        return st;
    }
    run->kernel_live = true;
    for (int i = 0; i < n; ++i) {
        run->mem[i] = mems[i];
        mems[i]->run = run;
        mems[i]->run_idx = i;
    }
    c->runs.push_back(run);
    return JB_OK;
}

int resident_inflight(const ResidentRun* run) { return run ? (int)(run->seq - run->consumed) : 0; }

bool resident_gather_fits(const jb_ctx* c, const jb_member* mem, uint64_t np) {
    // per table: the gathered table (world x np) and its ping-pong partner (half of it)
    const uint64_t glen = np * (uint64_t)c->world;
    return c->xch_ready && c->world <= 16 && (uint64_t)mem->ntables() * (glen + glen / 2) * 32 <= XCH_ARENA_HALF;
}

int resident_post(ResidentRun* run, const unsigned* actions, const uint64_t* challenge, bool exchange, bool gather) {
    jb_ctx* c = run->c;
    if (!run->kernel_live) return c->fail(JB_ERR_INVALID, "resident run is not live");
    if (run->seq - run->consumed >= 2) return c->fail(JB_ERR_INVALID, "resident run: two commands already in flight");
    const uint64_t seq = run->seq + 1;
    ResMailbox* mb = run->mb;
    ResCmdLine* line = &mb->cmd[seq & 1];
    uint64_t cmd = RES_OP_ROUND;
    if (exchange) {
        cmd |= RES_FLAG_EXCHANGE;
        line->xseq = ++c->xch_seq;
    }
    if (gather) {
        if (run->n != 1 || (actions[0] & 0xf) != RES_ACT_BIND_EVAL || exchange) return c->fail(JB_ERR_INVALID, "resident gather: one member, one bind");
        cmd |= RES_FLAG_GATHER;
        line->xseq = ++c->gather_seq;
    }
    ResConsumed* slot = run->ring[seq & 1];
    run->ring_gather[seq & 1] = gather;
    ResidentRun::RoundInfo ri{-1, 0, 0};
    for (int i = 0; i < run->n; ++i) {
        jb_member* m = run->mem[i];
        const unsigned a = actions[i] & 0xf;
        cmd |= (uint64_t)a << (16 + 4 * i);
        slot[i].act = a;
        slot[i].round = m->rounds_done;
        if (gather) {
            // the member leaves its shard for the gathered tables in this rank's arena (views, not owned)
            const uint64_t np = m->len / 2, glen = np * (uint64_t)c->world;
            uint64_t* arena = c->xch_peer[c->rank] + (XCH_ARENA_OFFSET + (size_t)(c->gather_seq & 1) * XCH_ARENA_HALF) / 8;
            const int T = m->ntables();
            for (int j = 0; j < T; ++j) {
                Table& t = m->tables[j];
                run->deferred.push_back(t);  // (the kernel still reads the shard while it executes this command)
                t.buf = arena + (size_t)j * glen * 4;
                t.alt = arena + (size_t)T * glen * 4 + (size_t)j * (glen / 2) * 4;
                t.cap = t.len = glen;
                t.alt_cap = glen / 2;
                t.buf_owned = t.alt_owned = false;
            }
            m->len = glen;
            slot[i].nprime = glen;
            slot[i].thin = res_is_thin(m->m, glen);
            ri.kind = 0;
            ri.items += glen / 2;
            ri.m = T;
            continue;
        }
        slot[i].nprime = a == RES_ACT_BIND_EVAL ? m->len / 2 : m->len;
        slot[i].thin = (a == RES_ACT_EVAL || a == RES_ACT_BIND_EVAL) && res_is_thin(m->m, slot[i].nprime);
        if (a == RES_ACT_EVAL || a == RES_ACT_BIND_EVAL) {
            ri.kind = (a == RES_ACT_BIND_EVAL || ri.kind == 0) ? 0 : 2;
            ri.items += slot[i].nprime / 2;
            ri.m = m->ntables();
        }
        // the host's view of the tables follows the command stream: the device executes commands in order
        if (a == RES_ACT_BIND_EVAL || a == RES_ACT_FINAL) {
            m->len /= 2;
            for (auto& t : m->tables) {
                if (m->order == JB_LOW_TO_HIGH) t.swap_buffers();
                t.len = m->len;
            }
        }
    }
    line->cmd = cmd;
    if (challenge) {
        std::memcpy((void*)line->challenge, challenge, 32);
        std::memcpy(run->ring_challenge[seq & 1], challenge, 32);
    }
    run->seq = seq;
    if (seq <= 64) {
        run->info[seq - 1] = ri;
        run->host_post[seq - 1] = now_ns();
    }
    __atomic_store_n(&line->cmd_seq, seq, __ATOMIC_RELEASE);
    return JB_OK;
}

int resident_consume(ResidentRun* run, uint64_t* out, ResConsumed* info) {
    jb_ctx* c = run->c;
    if (run->consumed >= run->seq) return c->fail(JB_ERR_INVALID, "resident run: no command in flight");
    WaitAcc acc(c);
    const uint64_t seq = run->consumed + 1;
    ResMailbox* mb = run->mb;
    int st = wait_answer(run, seq);
    if (st != JB_OK) return st;
    if (seq <= 64) run->host_recv[seq - 1] = now_ns();
    if (mb->ans[seq & 1].status != 0) {
        run->kernel_live = false;
        if (mb->ans[seq & 1].status == 2) return c->fail(JB_ERR_CUDA, "peer exchange timed out (a rank did not arrive)");
        return JB_RES_LOST;  // the kernel stopped waiting for commands: nothing from `seq` on was executed
    }
    run->consumed = seq;
    const uint64_t* result = mb->result[seq & 1];
    if (out) std::memcpy(out, (const void*)result, (size_t)run->n * RES_SLOT_U64 * 8);
    const ResConsumed* slot = run->ring[seq & 1];
    if (info) std::memcpy(info, slot, sizeof(ResConsumed) * run->n);
    bool all_done = run->consumed == run->seq;
    for (int i = 0; i < run->n; ++i) {
        jb_member* m = run->mem[i];
        if (slot[i].act == RES_ACT_FINAL && slot[i].nprime == 2) {  // the member is fully bound: its values came along
            std::memcpy(m->final_vals, (const void*)(result + (size_t)i * RES_SLOT_U64), (size_t)m->ntables() * 32);
            m->has_final = true;
        }
        if (m->len >= 2) all_done = false;
    }
    if (all_done) {  // every member is fully bound: the kernel has returned on its own
        run->kernel_live = false;
        release_run(run, false);
    }
    return JB_OK;
}

int resident_recover(ResidentRun* run) {
    jb_ctx* c = run->c;
    run->kernel_live = false;
    cudaStreamSynchronize(run->res.stream);  // the kernel has exited (it answered the lost command with status 1)
    const uint64_t first = run->consumed + 1, last = run->seq;
    for (uint64_t q = first; q <= last; ++q)
        if (run->ring_gather[q & 1]) {
            release_run(run, true);
            return c->fail(JB_ERR_CUDA, "resident kernel lost during a cross-rank gather (not replayable)");
        }
    // the host's view ran ahead of the device by the unexecuted commands: step it back ...
    for (uint64_t q = last; q >= first; --q) {
        const ResConsumed* slot = run->ring[q & 1];
        for (int i = 0; i < run->n; ++i) {
            if (slot[i].act != RES_ACT_BIND_EVAL && slot[i].act != RES_ACT_FINAL) continue;
            jb_member* m = run->mem[i];
            m->len *= 2;
            for (auto& t : m->tables) {
                if (m->order == JB_LOW_TO_HIGH) t.swap_buffers();
                t.len = m->len;
            }
        }
    }
    // ... and replay their binds, in order, with ordinary launches
    int st = JB_OK;
    cudaEventRecord(run->res.event, run->res.stream);
    cudaStreamWaitEvent(c->stream, run->res.event, 0);
    for (uint64_t q = first; q <= last && st == JB_OK; ++q) {
        const ResConsumed* slot = run->ring[q & 1];
        for (int i = 0; i < run->n && st == JB_OK; ++i) {
            if (slot[i].act != RES_ACT_BIND_EVAL && slot[i].act != RES_ACT_FINAL) continue;
            jb_member* m = run->mem[i];
            for (auto& t : m->tables) {
                st = bind_table(c, t, run->ring_challenge[q & 1], m->order);
                if (st != JB_OK) break;
            }
            if (st == JB_OK) m->len /= 2;
        }
    }
    for (int i = 0; i < run->n; ++i) run->mem[i]->look_ok = false;
    run->consumed = run->seq;
    release_run(run, true);
    return st;
}

int resident_round(ResidentRun* run, const unsigned* actions, const uint64_t* challenge, bool exchange, uint64_t* out) {
    int st = JB_OK;
    while (st == JB_OK && run->consumed < run->seq) st = resident_consume(run, nullptr, nullptr);  // (never releases: a
    if (st == JB_OK) st = resident_post(run, actions, challenge, exchange);                         //  round is still to come)
    if (st == JB_OK) st = resident_consume(run, out, nullptr);
    return st;  // JB_RES_LOST: the caller recovers (resident_recover) and redoes the round with launches
}

void resident_end(ResidentRun* run, bool mark_no_resident) {
    if (!run) return;
    // answers still on their way belong to commands the host's view of the tables already includes: take them first
    while (run->kernel_live && run->consumed < run->seq) {
        jb_ctx* c = run->c;
        const bool last = run->consumed + 1 == run->seq;
        bool done = last;
        for (int i = 0; i < run->n && done; ++i) done = run->mem[i]->len < 2;
        const int cs = resident_consume(run, nullptr, nullptr);
        if (cs == JB_RES_LOST) {
            resident_recover(run);  // replays the unexecuted binds and releases the run
            return;
        }
        if (cs != JB_OK) break;
        if (done) {  // that consume released the run (every member fully bound)
            (void)c;
            return;
        }
    }
    if (run->kernel_live) {
        ResMailbox* mb = run->mb;
        const uint64_t seq = run->seq + 1;
        mb->cmd[seq & 1].cmd = RES_OP_ABORT;
        run->seq = seq;
        __atomic_store_n(&mb->cmd[seq & 1].cmd_seq, seq, __ATOMIC_RELEASE);
        wait_answer(run, seq);
        run->kernel_live = false;
    }
    release_run(run, mark_no_resident);
}

int resident_run_size(const ResidentRun* run) { return run ? run->n : 0; }
