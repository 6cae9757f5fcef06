// Sumcheck members on the device: ProveRounds (crates/jolt-sumcheck/src/prover.rs:52-72) for sum-of-products
// relations over dense tables, the split-eq (Gruen) member, the index-sharded member, and the device
// RoundScheduler (prover.rs:106-120). See include/jolt_b200.h for the per-function reference citations.
#include "../../include/jolt_b200.h"

#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "member.hpp"
#include "resident.cuh"
#include "sumcheck_host.hpp"

using namespace jb;
using namespace jbi;
using Guard = CtxGuard;


// result slots in host-mapped memory: slot s = h_result + s * JB_SLOT_U64: [0, 64) values, [64] sequence flag
constexpr int JB_SLOT_U64 = 128;

namespace {

// One launch per round, 256 threads x 2 blocks per SM. WEIGHTED: the split-eq pass (s(1) from the claim).
template <int M, int P, int ORDER, bool BIND, bool HI4, bool SKIP1, bool WEIGHTED = false>
int launch_fused(jb_ctx* c, const TablePtrs& tp, size_t pairs, const BindScalar& s, RoundOut out) {
    auto kernel = fused_round_kernel<M, P, ORDER, BIND, HI4, SKIP1, 256, 2, WEIGHTED>;
    constexpr size_t smem = FusedShape<M, SKIP1>::smem_bytes(256);
    static int per_sm = [&] {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, 256, smem) != cudaSuccess || nb < 1) nb = 1;
        return nb;
    }();
    // grid-stride over whole waves of resident blocks; tiny rounds take one (small) block
    size_t need = (pairs + 255) / 256;
    size_t resident = (size_t)c->sm_count * per_sm;
    size_t grid = need < resident ? need : resident;
    if (grid < 1) grid = 1;
    constexpr int K = FusedShape<M, SKIP1>::K;
    int st = c->ensure_partial(grid * K);
    if (st != JB_OK) return st;
    out.partial = c->d_partial;
    int tix = c->timing_begin(BIND ? 0 : 2, pairs, M * P);
    // latency path: a round of <= 32 pairs runs as one warp (no barriers, no shared-memory stage)
    const unsigned block = pairs <= 32 ? 32u : 256u;
    kernel<<<(unsigned)grid, block, smem, c->stream>>>(tp, pairs, s, out);
    c->timing_end(tix);
    c->launches++;
    return c->check(cudaGetLastError(), WEIGHTED ? "fused_round_kernel (weighted) launch" : "fused_round_kernel launch");
}

template <int M, int ORDER>
int dispatch_weighted1(jb_ctx* c, const TablePtrs& tp, size_t pairs, bool bind, bool hi4, const BindScalar& s,
                       const RoundOut& out) {
    if (!bind) return launch_fused<M, 1, ORDER, false, false, true, true>(c, tp, pairs, s, out);
    return hi4 ? launch_fused<M, 1, ORDER, true, true, true, true>(c, tp, pairs, s, out)
               : launch_fused<M, 1, ORDER, true, false, true, true>(c, tp, pairs, s, out);
}

int dispatch_weighted(jb_ctx* c, int m, int order, const TablePtrs& tp, size_t pairs, bool bind, bool hi4, const BindScalar& s,
                      const RoundOut& out) {
    const bool l2h = order == JB_LOW_TO_HIGH;
    switch (m) {
        case 1: return l2h ? dispatch_weighted1<1, ORDER_LOW_TO_HIGH>(c, tp, pairs, bind, hi4, s, out)
                           : dispatch_weighted1<1, ORDER_HIGH_TO_LOW>(c, tp, pairs, bind, hi4, s, out);
        case 2: return l2h ? dispatch_weighted1<2, ORDER_LOW_TO_HIGH>(c, tp, pairs, bind, hi4, s, out)
                           : dispatch_weighted1<2, ORDER_HIGH_TO_LOW>(c, tp, pairs, bind, hi4, s, out);
        case 3: return l2h ? dispatch_weighted1<3, ORDER_LOW_TO_HIGH>(c, tp, pairs, bind, hi4, s, out)
                           : dispatch_weighted1<3, ORDER_HIGH_TO_LOW>(c, tp, pairs, bind, hi4, s, out);
        default: return launch_wide_round(c, m, order, true, true, tp, pairs, bind, hi4, s, out);  // m = 4..8
    }
}


template <int M, int P, int ORDER, bool SKIP1>
int dispatch_fused2(jb_ctx* c, const TablePtrs& tp, size_t pairs, bool bind, bool hi4, const BindScalar& s,
                    const RoundOut& out) {
    if (!bind) return launch_fused<M, P, ORDER, false, false, SKIP1>(c, tp, pairs, s, out);
    return hi4 ? launch_fused<M, P, ORDER, true, true, SKIP1>(c, tp, pairs, s, out)
               : launch_fused<M, P, ORDER, true, false, SKIP1>(c, tp, pairs, s, out);
}

template <int M, int P>
int dispatch_fused1(jb_ctx* c, int order, bool skip1, const TablePtrs& tp, size_t pairs, bool bind, bool hi4,
                    const BindScalar& s, const RoundOut& out) {
    if (order == JB_HIGH_TO_LOW)
        return skip1 ? dispatch_fused2<M, P, ORDER_HIGH_TO_LOW, true>(c, tp, pairs, bind, hi4, s, out)
                     : dispatch_fused2<M, P, ORDER_HIGH_TO_LOW, false>(c, tp, pairs, bind, hi4, s, out);
    return skip1 ? dispatch_fused2<M, P, ORDER_LOW_TO_HIGH, true>(c, tp, pairs, bind, hi4, s, out)
                 : dispatch_fused2<M, P, ORDER_LOW_TO_HIGH, false>(c, tp, pairs, bind, hi4, s, out);
}

// the instantiated shapes: products of 1..8 tables (5..8 in wide_product.cu); the two-term degree-2 sum of products
bool shape_supported(int m, int terms) { return (terms == 1 && m >= 1 && m <= JB_MAX_TABLES) || (terms == 2 && m == 2); }

int dispatch_fused(jb_ctx* c, int m, int terms, int order, bool skip1, const TablePtrs& tp, size_t pairs, bool bind,
                   bool hi4, const BindScalar& s, const RoundOut& out) {
    if (terms == 2 && m == 2) return dispatch_fused1<2, 2>(c, order, skip1, tp, pairs, bind, hi4, s, out);
    if (terms != 1) return c->fail(JB_ERR_UNSUPPORTED, "member: unsupported sum-of-products shape");
    switch (m) {
        case 1: return dispatch_fused1<1, 1>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        case 2: return dispatch_fused1<2, 1>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        case 3: return dispatch_fused1<3, 1>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        case 4: return dispatch_fused1<4, 1>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        default: return launch_wide_round(c, m, order, skip1, false, tp, pairs, bind, hi4, s, out);  // m = 5..8
    }
}

}  // namespace

extern "C" {

// ---- sumcheck member -------------------------------------------------------------------
static int member_create_common(jb_ctx* c, const jb_table* handles, size_t m, size_t terms, int order, jb_member** out) {
    if (!c || !handles || !out) return JB_ERR_INVALID;
    Guard g(c);
    if (!shape_supported((int)m, (int)terms))
        return c->fail(JB_ERR_UNSUPPORTED, "member: supported shapes are products of 1..8 tables and 2 terms x 2 factors");
    if (order != JB_HIGH_TO_LOW && order != JB_LOW_TO_HIGH) return c->fail(JB_ERR_INVALID, "member: unknown order");
    const size_t T = m * terms;
    size_t len = 0;
    for (size_t j = 0; j < T; ++j) {
        Table* t = c->find(handles[j]);
        if (!t) return c->fail(JB_ERR_INVALID, "member: unknown table handle");
        for (size_t k = 0; k < j; ++k)
            if (handles[k] == handles[j]) return c->fail(JB_ERR_INVALID, "member: duplicate table handle");
        if (j == 0) len = t->len;
        if (t->len != len) return c->fail(JB_ERR_INVALID, "member: tables differ in length");
    }
    if (len == 0 || (len & (len - 1))) return c->fail(JB_ERR_INVALID, "member: table length must be a power of two");
    jb_member* mem = new (std::nothrow) jb_member();
    if (!mem) return JB_ERR_OOM;
    mem->ctx = c;
    mem->m = (int)m;
    mem->terms = (int)terms;
    mem->order = order;
    mem->len = len;
    mem->rounds = 0;
    while (((size_t)1 << mem->rounds) < len) ++mem->rounds;
    for (size_t j = 0; j < T; ++j) {
        auto it = c->tables.find(handles[j]);
        mem->tables.push_back(it->second);
        c->tables.erase(it);  // ownership moves into the member
    }
    *out = mem;
    return JB_OK;
}

int jb_member_create(jb_ctx* c, const jb_table* handles, size_t m, int order, jb_member** out) {
    return member_create_common(c, handles, m, 1, order, out);
}

int jb_member_create_sop(jb_ctx* c, const jb_table* handles, size_t factors, size_t terms, int order, jb_member** out) {
    return member_create_common(c, handles, factors, terms, order, out);
}

int jb_member_num_rounds(jb_member* mem, size_t* rounds) {
    if (!mem || !rounds) return JB_ERR_INVALID;
    *rounds = mem->rounds;
    return JB_OK;
}

int jb_member_degree(jb_member* mem, size_t* degree) {
    if (!mem || !degree) return JB_ERR_INVALID;
    *degree = (size_t)mem->m + (mem->eq ? 1 : 0);
    return JB_OK;
}

jb_ctx* jb_member_context(jb_member* mem) { return mem ? mem->ctx : nullptr; }

int jb_member_num_tables(jb_member* mem, size_t* tables) {
    if (!mem || !tables) return JB_ERR_INVALID;
    *tables = (size_t)mem->ntables();
    return JB_OK;
}

// Runs the fused pass; on return result slot `slot` will hold the K sums (canonical) or, if lanes_out,
// lanes_out holds them widened to one 32-bit limb per u64.
static void* const JB_LANES_EXCHANGE = (void*)(uintptr_t)1;  // sentinel: all-reduce in the kernel epilogue

struct EqRound {
    const uint64_t* e_out;
    const uint64_t* e_in;
    int in_bits;
};

static int member_round(jb_member* mem, const uint64_t* bind, bool skip1, void* lanes_out, const EqRound* eqr = nullptr,
                        int slot = 0, uint64_t* seq_out = nullptr) {
    jb_ctx* c = mem->ctx;
    bool do_bind = bind != nullptr;
    bool hi4 = false;
    BindScalar s;
    std::memset(&s, 0, sizeof s);
    size_t len = mem->len;
    if (do_bind) {
        if (!canonical_fr(bind)) return c->fail(JB_ERR_INVALID, "prove_round: challenge limbs not canonical");
        if (len < 4) return c->fail(JB_ERR_INVALID, "prove_round: no round left after this bind (use finish_rounds)");
        s = make_scalar(bind, &hi4);
        len /= 2;
    } else if (len < 2) {
        return c->fail(JB_ERR_INVALID, "prove_round: member is fully bound");
    }
    size_t pairs = len / 2;
    TablePtrs tp;
    std::memset(&tp, 0, sizeof tp);
    const int T = mem->ntables();
    for (int j = 0; j < T; ++j) {
        Table& t = mem->tables[j];
        tp.in[j] = t.buf;
        tp.out[j] = t.buf;
        if (do_bind && mem->order == JB_LOW_TO_HIGH) {
            int st = c->ensure_alt(t, len);
            if (st != JB_OK) return st;
            tp.out[j] = t.alt;
        }
    }
    RoundOut ro;
    ro.partial = nullptr;  // set by launch_fused
    ro.counter = c->d_counter;
    ro.lanes = lanes_out ? 1 : 0;
    ro.world = 1;
    ro.rank = 0;
    ro.xseq = 0;
    ro.timeout_cycles = 0;
    for (int g2 = 0; g2 < 16; ++g2) ro.peer[g2] = nullptr;
    ro.seq = ++c->result_seq;
    if (seq_out) *seq_out = ro.seq;
    uint64_t* slot_dev = c->d_result_alias + (size_t)slot * JB_SLOT_U64;
    if (lanes_out == JB_LANES_EXCHANGE) {  // fused all-reduce over peer memory, totals (lanes) to the host
        ro.lanes = 2;
        ro.result = slot_dev;
        ro.flag = slot_dev + 64;
        for (int g2 = 0; g2 < 16; ++g2) ro.peer[g2] = c->xch_peer[g2];
        ro.world = c->world;
        ro.rank = c->rank;
        ro.xseq = ++c->xch_seq;
        ro.timeout_cycles = 20000000000LL;
    } else if (lanes_out) {
        ro.result = (uint64_t*)lanes_out;
        ro.flag = nullptr;
    } else {
        ro.result = slot_dev;
        ro.flag = slot_dev + 64;
    }
    int st;
    if (eqr) {
        tp.e_out = eqr->e_out;
        tp.e_in = eqr->e_in;
        tp.in_bits = eqr->in_bits;
        st = dispatch_weighted(c, mem->m, mem->order, tp, pairs, do_bind, hi4, s, ro);
    } else {
        st = dispatch_fused(c, mem->m, mem->terms, mem->order, skip1, tp, pairs, do_bind, hi4, s, ro);
    }
    if (st != JB_OK) return st;
    if (do_bind) {
        for (int j = 0; j < T; ++j) {
            if (mem->order == JB_LOW_TO_HIGH) mem->tables[j].swap_buffers();
            mem->tables[j].len = len;
        }
        mem->len = len;
    }
    return JB_OK;
}

// Spin until the last block of the launch that took sequence number `want` has published into `slot`.
static int wait_round_result(jb_ctx* c, int slot, uint64_t want) {
    WaitAcc acc_(c);
    volatile uint64_t* flag = c->h_result + (size_t)slot * JB_SLOT_U64 + 64;
    uint64_t spins = 0;
    while (*flag != want) {
        if ((++spins & 0xfffff) == 0) {  // every ~1M spins make sure the stream has not died
            cudaError_t e = cudaStreamQuery(c->stream);
            if (e != cudaSuccess && e != cudaErrorNotReady) return c->check(e, "round kernel failed");
            if (e == cudaSuccess && *flag != want) return c->fail(JB_ERR_CUDA, "round kernel finished without publishing its result");
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    return JB_OK;
}
static int wait_round_result0(jb_ctx* c) { return wait_round_result(c, 0, c->result_seq); }

static int sharded_prove_round(jb_member* mem, const uint64_t* bind, size_t round, const uint64_t* claim,
                               uint64_t* out_evals);
static int resident_values(int D, const uint64_t* lanes, uint64_t* vals);

static int eq_prove_round(jb_member* mem, const uint64_t* bind, size_t round, const uint64_t* claim, uint64_t* out_evals);

struct RoundConsts {
    HostFr w[JB_MAX_TABLES], ipow[JB_MAX_TABLES], mpow;
};
static const RoundConsts& round_consts(int M) {  // M in 2..JB_MAX_TABLES
    static RoundConsts table[JB_MAX_TABLES + 1];
    static const bool init = [] {
        uint64_t binom[JB_MAX_TABLES + 1][JB_MAX_TABLES + 1] = {};  // Pascal's triangle: binom[m][i] = C(m, i)
        for (int m = 0; m <= JB_MAX_TABLES; ++m) {
            binom[m][0] = 1;
            for (int i = 1; i <= m; ++i) binom[m][i] = binom[m - 1][i - 1] + binom[m - 1][i];
        }
        for (int m = 2; m <= JB_MAX_TABLES; ++m) {
            for (int i = 0; i < m; ++i) {
                HostFr ti = HostFr::one();  // i^m
                for (int e = 0; e < m; ++e) ti = ti * HostFr::from_u64((uint64_t)i);
                table[m].ipow[i] = ti;
                const HostFr b = HostFr::from_u64(binom[m][i]);
                table[m].w[i] = ((m - 1 - i) & 1) ? HostFr::zero() - b : b;
            }
            HostFr tm = HostFr::one();  // m^m
            for (int e = 0; e < m; ++e) tm = tm * HostFr::from_u64((uint64_t)m);
            table[m].mpow = tm;
        }
        return true;
    }();
    (void)init;
    return table[M];
}

// Assembles s(0..M) from the K published values. Kernel order: s(0), [s(1)], s(2..M-1), s(inf) for
// M >= 2 (s(0), [s(1)] for M == 1); with skip1, s(1) = claim - s(0). s(M) is rebuilt from the leading
// coefficient: q(t) = s(t) - s(inf) t^M has degree < M, so q(M) = sum_{i<M} (-1)^(M-1-i) C(M,i) q(i).
// In verify mode the claim is checked (naive.rs:301-308).
static int assemble_evals(jb_ctx* c, int M, bool skip1, const uint64_t* vals, const uint64_t* claim, size_t round,
                          uint64_t* out_evals) {
    HostFr ev[jb::JB_MEMBER_EVALS];
    int k = 0;
    ev[0] = HostFr::from_limbs(vals + 4 * k++);
    if (skip1) ev[1] = HostFr::from_limbs(claim) - ev[0];
    else ev[1] = HostFr::from_limbs(vals + 4 * k++);
    if (M >= 2) {
        for (int t = 2; t < M; ++t) ev[t] = HostFr::from_limbs(vals + 4 * k++);
        const HostFr lead = HostFr::from_limbs(vals + 4 * k++);
        // s(M) = sum_{i<M} w_i (s(i) - lead i^M) + lead M^M with w_i = (-1)^(M-1-i) C(M,i); the constants are built
        // once (this runs on the Fiat-Shamir round trip of every round)
        const RoundConsts& rc = round_consts(M);
        HostFr qM = HostFr::zero();
        for (int i = 0; i < M; ++i) qM = qM + rc.w[i] * (ev[i] - lead * rc.ipow[i]);
        ev[M] = qM + lead * rc.mpow;
    }
    for (int t = 0; t <= M; ++t) ev[t].store(out_evals + 4 * t);
    if (claim && !skip1 && (ev[0] + ev[1]) != HostFr::from_limbs(claim)) {
        char buf[96];
        std::snprintf(buf, sizeof buf, "RoundCheckFailed { round: %zu }", round);
        return c ? c->fail(JB_ERR_ROUND_CHECK, buf) : (int)JB_ERR_ROUND_CHECK;
    }
    return JB_OK;
}

int jb_round_evals_from_kernel_values(int m, int skip_t1, const uint64_t* kernel_values, const uint64_t* claim_or_null,
                                      uint64_t* out_evals) {
    if (!kernel_values || !out_evals || m < 1 || m > 4) return JB_ERR_INVALID;
    if (skip_t1 && !claim_or_null) return JB_ERR_INVALID;
    const int k = m == 1 ? (skip_t1 ? 1 : 2) : (skip_t1 ? m : m + 1);
    for (int t = 0; t < k; ++t)
        if (!canonical_fr(kernel_values + 4 * t)) return JB_ERR_INVALID;
    if (claim_or_null && !canonical_fr(claim_or_null)) return JB_ERR_INVALID;
    return assemble_evals(nullptr, m, skip_t1 != 0, kernel_values, claim_or_null, 0, out_evals);
}

// ---- rounds served by a resident kernel -----------------------------------------------------------------
// K canonical kernel values (s(0), [s(2..D-1)], s(inf)) of one member from an answer's lanes.
static void answer_values(const jb_member* mem, const ResConsumed& info, const uint64_t* lanes, uint64_t* vals) {
    if (info.thin) {  // s(0) = S0 + S6, s(inf) = S2 + S7: add the integer lanes, reduce once each
        uint64_t sum[2 * 17];
        for (int w = 0; w < 17; ++w) {
            sum[w] = lanes[0 * 17 + w] + lanes[6 * 17 + w];
            sum[17 + w] = lanes[2 * 17 + w] + lanes[7 * 17 + w];
        }
        jb_wide_lanes_reduce_host(sum, 2, vals);
    } else {
        resident_values(mem->m, lanes, vals);
    }
}

// A thin answer also determines the NEXT round's polynomial as a function of the challenge that round binds.
static void harvest_lookahead(jb_member* mem, const ResConsumed& info, const uint64_t* lanes) {
    if ((info.act == RES_ACT_EVAL || info.act == RES_ACT_BIND_EVAL) && info.thin && info.nprime >= 4) {
        jb_wide_lanes_reduce_host(lanes, 6, mem->look);
        mem->look_ok = true;
        mem->look_round = info.round + 1;
    } else if (info.act != RES_ACT_NONE) {
        mem->look_ok = false;
    }
}

// s(0)(r) = S0 + r (S1 - S0 - S2) + r^2 S2 and s(inf)(r) = S3 + r (S4 - S3 - S5) + r^2 S5 at the drawn challenge
static void lookahead_values(const jb_member* mem, const uint64_t* r_limbs, uint64_t* vals) {
    const HostFr r = HostFr::from_limbs(r_limbs);
    for (int h = 0; h < 2; ++h) {
        const HostFr a0 = HostFr::from_limbs(mem->look + (3 * h) * 4), a1 = HostFr::from_limbs(mem->look + (3 * h + 1) * 4),
                     lead = HostFr::from_limbs(mem->look + (3 * h + 2) * 4);
        ((lead * r + (a1 - a0 - lead)) * r + a0).store(vals + 4 * h);
    }
}

struct RunItem {
    jb_member* mem;
    const uint64_t* bind;   // null on the member's first round
    const uint64_t* claim;  // the running claim (s(1) = claim - s(0))
    size_t round;
    uint64_t* out_evals;
};

// One round of `n` members of one run: ONE mailbox command. Members whose previous answer carried lookahead sums
// are answered at once from those (their command stays in flight: the device's bind + next sums overlap the
// caller's Fiat-Shamir step); the others wait for this command's own answer.
static int run_round(jb_ctx* c, ResidentRun* run, RunItem* items, int n, const uint64_t* shared_bind, bool exchange,
                     bool gather = false) {
    unsigned actions[RES_MAX_MEMBERS] = {0};
    for (int i = 0; i < n; ++i) actions[items[i].mem->run_idx] = items[i].bind ? RES_ACT_BIND_EVAL : RES_ACT_EVAL;
    jb_member* mems[RES_MAX_MEMBERS];
    const int rn = run->n;
    for (int i = 0; i < rn; ++i) mems[i] = run->mem[i];
    int st = resident_post(run, actions, shared_bind, exchange, gather);
    if (st != JB_OK) return st;
    uint64_t out[RES_MAX_MEMBERS * RES_SLOT_U64];
    ResConsumed info[RES_MAX_MEMBERS];
    bool lost = false;
    while (!lost && resident_inflight(run) > 1) {  // the previous command's answer: it carries this round's lookahead
        st = resident_consume(run, out, info);
        if (st == JB_RES_LOST) lost = true;
        else if (st != JB_OK) return st;
        else for (int i = 0; i < rn; ++i) harvest_lookahead(mems[i], info[i], out + (size_t)i * RES_SLOT_U64);
    }
    uint64_t vals[RES_MAX_MEMBERS][jb::JB_MEMBER_EVALS * 4];
    bool hit[RES_MAX_MEMBERS], need_now = false;
    for (int i = 0; i < n && !lost; ++i) {
        jb_member* m = items[i].mem;
        hit[i] = items[i].bind && m->look_ok && m->look_round == items[i].round && m->m == 2;
        if (hit[i]) lookahead_values(m, items[i].bind, vals[i]);
        else need_now = true;
    }
    if (need_now && !lost) {
        st = resident_consume(run, out, info);  // (cannot release the run: the members of this round are not fully bound)
        if (st == JB_RES_LOST) lost = true;
        else if (st != JB_OK) return st;
    }
    if (lost) {
        // the kernel gave up waiting (the host was held up): replay the unexecuted binds with launches and compute
        // this round's sums with one eval-only launch per member - the proof is unchanged, only slower
        st = resident_recover(run);
        if (st != JB_OK) return st;
        for (int i = 0; i < n; ++i) {
            jb_member* m = items[i].mem;
            st = member_round(m, nullptr, true, nullptr);
            if (st == JB_OK) st = wait_round_result0(c);
            if (st == JB_OK) st = assemble_evals(c, m->m, true, c->h_result, items[i].claim, items[i].round, items[i].out_evals);
            if (st != JB_OK) return st;
            m->rounds_done++;
        }
        return JB_OK;
    }
    if (need_now) {
        for (int i = 0; i < n; ++i)
            if (!hit[i]) {
                const int idx = items[i].mem->run_idx;
                answer_values(items[i].mem, info[idx], out + (size_t)idx * RES_SLOT_U64, vals[i]);
            }
        for (int i = 0; i < rn; ++i) harvest_lookahead(mems[i], info[i], out + (size_t)i * RES_SLOT_U64);
    }
    for (int i = 0; i < n; ++i) {
        jb_member* m = items[i].mem;
        st = assemble_evals(c, m->m, true, vals[i], items[i].claim, items[i].round, items[i].out_evals);
        if (st != JB_OK) return st;
        m->rounds_done++;
    }
    return JB_OK;
}

// This round of one member through its resident kernel (starting one if the member is eligible). Returns
// JB_ERR_UNSUPPORTED if the member is not served by a run: the caller launches instead.
static int resident_member_prove(jb_member* mem, const uint64_t* bind, const uint64_t* claim, size_t round, bool exchange,
                                 uint64_t* out_evals, bool gather = false) {
    jb_ctx* c = mem->ctx;
    if (!mem->run) {
        if (!resident_eligible(mem)) return JB_ERR_UNSUPPORTED;
        jb_member* one[1] = {mem};
        int st = resident_begin(c, one, 1);
        if (st != JB_OK) return st;
    }
    RunItem it{mem, bind, claim, round, out_evals};
    int st = run_round(c, mem->run, &it, 1, bind, exchange, gather);
    if (st != JB_OK && mem->run) resident_end(mem->run, true);
    return st;
}

// The terminal bind of one member through its run (the run is released when every member is fully bound).
static int resident_member_final(jb_member* mem, const uint64_t* bind) {
    unsigned actions[RES_MAX_MEMBERS] = {0};
    actions[mem->run_idx] = RES_ACT_FINAL;
    int st = resident_round(mem->run, actions, bind, false, nullptr);
    if (st == JB_RES_LOST) return resident_recover(mem->run);  // (replays the terminal bind with a launch)
    if (st != JB_OK && mem->run) resident_end(mem->run, true);
    return st;
}

// Stops whatever resident kernel would be in the way of a launch for this member.
static void before_launch(jb_member* mem) {
    if (mem->run) resident_end(mem->run, true);
    mem->ctx->quiesce_resident(false);
}

int jb_member_prove_round(jb_member* mem, const uint64_t* bind, size_t round, const uint64_t* claim,
                          uint64_t* out_evals) {
    if (!mem || !out_evals) return JB_ERR_INVALID;
    jb_ctx* c = mem->ctx;
    if (mem->sharded) {
        int st = sharded_prove_round(mem, bind, round, claim, out_evals);
        if (st == JB_OK) mem->rounds_done++;
        return st;
    }
    Guard g(c, true);
    if (round != mem->rounds_done) return c->fail(JB_ERR_INVALID, "prove_round: round index out of sequence");
    if ((mem->rounds_done == 0) != (bind == nullptr))
        return c->fail(JB_ERR_INVALID, "prove_round: bind must be absent exactly on the first round");
    if (bind && !canonical_fr(bind)) return c->fail(JB_ERR_INVALID, "prove_round: challenge limbs not canonical");
    if (mem->len < (bind ? 4u : 2u))
        return c->fail(JB_ERR_INVALID, bind ? "prove_round: no round left after this bind (use finish_rounds)"
                                            : "prove_round: member is fully bound");
    if (mem->eq) {
        before_launch(mem);
        int st = eq_prove_round(mem, bind, round, claim, out_evals);
        if (st == JB_OK) mem->rounds_done++;
        return st;
    }
    // With a claim and round verification off (the default, = the reference's optimized tier) the
    // kernel skips t = 1 and s(1) = claim - s(0); with verification on (or no claim) it computes
    // every point and the claim, if given, is checked (the reference tier, naive.rs:301-308).
    const bool skip1 = claim != nullptr && !c->verify_rounds;
    int st;
    if (skip1) {
        // the resident kernel serves this and every later round of the member: no launch per round
        st = resident_member_prove(mem, bind, claim, round, false, out_evals);  // (counts the round itself)
        if (st != JB_ERR_UNSUPPORTED) return st;
    }
    before_launch(mem);
    st = member_round(mem, bind, skip1, nullptr);
    if (st != JB_OK) return st;
    st = wait_round_result0(c);
    if (st != JB_OK) return st;
    st = assemble_evals(c, mem->m, skip1, c->h_result, claim, round, out_evals);
    if (st == JB_OK) mem->rounds_done++;
    return st;
}

// ---- split-eq member: one round ------------------------------------------------------------------------
// scalar <- scalar * eq(w_v, r) for the variable v just bound (GruenSplitEqPolynomial::bind, split_eq.rs:347-352)
static void eq_absorb_bind(jb_member* mem, size_t var, const uint64_t* r) {
    HostFr wv = HostFr::from_limbs(mem->eq_w.data() + 4 * var), rr = HostFr::from_limbs(r);
    HostFr prod = wv * rr;
    HostFr f = HostFr::one() - wv - rr + prod + prod;
    (HostFr::from_limbs(mem->eq_scalar) * f).store(mem->eq_scalar);
}

static int eq_prove_round(jb_member* mem, const uint64_t* bind, size_t round, const uint64_t* claim, uint64_t* out_evals) {
    jb_ctx* c = mem->ctx;
    if (!claim) return c->fail(JB_ERR_INVALID, "eq member: the running claim is required (Gruen hint s(0)+s(1))");
    const size_t n = mem->eq_n, M = (size_t)mem->m;
    if (round >= n) return c->fail(JB_ERR_INVALID, "prove_round: member is fully bound");
    const bool l2h = mem->order == JB_LOW_TO_HIGH;
    if (bind) {
        if (!canonical_fr(bind)) return c->fail(JB_ERR_INVALID, "prove_round: challenge limbs not canonical");
        eq_absorb_bind(mem, l2h ? n - round : round - 1, bind);  // the previous round's variable
    }
    EqRound er;
    size_t cur_var;
    if (l2h) {
        const size_t cur = n - round;  // unbound variables including the current one (index cur - 1)
        const size_t head = cur - 1;
        const size_t out_bits = head < mem->eq_split ? head : mem->eq_split;
        const size_t in_bits = head - out_bits;
        er.e_out = mem->eq_tabs + 4 * (((size_t)1 << out_bits) - 1);
        er.e_in = mem->eq_tabs + 4 * (mem->eq_in_base + ((size_t)1 << in_bits) - 1);
        er.in_bits = (int)in_bits;
        cur_var = cur - 1;
    } else {
        // HighToLow (split_eq.rs:233-257): the current variable is w[round]; the remaining ones w[round + 1 .. n)
        // are the pair index MSB-first: the unbound suffix of in_point = w[1 .. 1 + s) on top of out_point =
        // w[1 + s .. n) (evals_cached_rev: suffix tables), then suffixes of out_point alone
        const size_t sp = mem->eq_split;  // s = |in_point|
        const size_t nlo = n - 1 - sp;    // |out_point|
        const size_t hi_k = round < sp ? round : sp;          // hi table: eq(w[1 + hi_k .. 1 + s))
        const size_t lo_k = round < sp ? 0 : round - sp;      // lo table: eq(w[1 + s + lo_k .. n))
        er.e_out = mem->eq_tabs + 4 * mem->eq_hi_off[hi_k];
        er.e_in = mem->eq_tabs + 4 * mem->eq_lo_off[lo_k];
        er.in_bits = (int)(nlo - lo_k);
        cur_var = round;
    }
    // the current variable's linear factor l(t) = l0 + t (l1 - l0) is known before the pass runs
    const HostFr scalar = HostFr::from_limbs(mem->eq_scalar);
    const HostFr wc = HostFr::from_limbs(mem->eq_w.data() + 4 * cur_var);
    const HostFr l1 = scalar * wc, l0 = scalar - l1;
    if (l1.is_zero()) return c->fail(JB_ERR_INVALID, "eq member: current eq evaluation at one must be invertible");
    int st = member_round(mem, bind, true, nullptr, &er);
    if (st != JB_OK) return st;
    // a field inversion is ~400 host multiplications (~13 us): do it while the device runs the pass
    const HostFr l1_inv = l1.inverse();
    st = wait_round_result0(c);
    if (st != JB_OK) return st;
    // kernel order: q(0), q(2), .., q(M-1), q(inf)   (M values; q(0) only for M == 1)
    const HostFr q0 = HostFr::from_limbs(c->h_result);
    const HostFr q1 = (HostFr::from_limbs(claim) - l0 * q0) * l1_inv;
    uint64_t vals[jb::JB_MEMBER_EVALS * 4], qe[jb::JB_MEMBER_EVALS * 4];
    q0.store(vals);
    q1.store(vals + 4);
    if (M > 1) std::memcpy(vals + 8, c->h_result + 4, (M - 1) * 32);
    st = assemble_evals(c, (int)M, false, vals, nullptr, round, qe);  // q(0..M)
    if (st != JB_OK) return st;
    // q(M+1) by extrapolation (degree M), then s(t) = l(t) q(t), t = 0..M+1
    std::vector<HostFr> qv(M + 1);
    for (size_t t = 0; t <= M; ++t) qv[t] = HostFr::from_limbs(qe + 4 * t);
    jb::UnivariatePoly qp = jb::UnivariatePoly::from_evals(qv);
    const HostFr dl = l1 - l0;
    HostFr lt = l0;
    for (size_t t = 0; t <= M + 1; ++t) {
        HostFr qt = t <= M ? qv[t] : qp.evaluate(HostFr::from_u64(t));
        (lt * qt).store(out_evals + 4 * t);
        lt = lt + dl;
    }
    return JB_OK;
}

int jb_eq_member_create(jb_ctx* c, const jb_table* handles, size_t m, const uint64_t* w, size_t nvars,
                        const uint64_t* scale_or_null, int order, jb_member** out) {
    if (!c || !handles || !w || !out) return JB_ERR_INVALID;
    if (order != JB_LOW_TO_HIGH && order != JB_HIGH_TO_LOW) return c->fail(JB_ERR_INVALID, "eq member: unknown binding order");
    if (m < 1 || m > JB_MAX_TABLES) return c->fail(JB_ERR_UNSUPPORTED, "eq member: m must be 1..8");
    for (size_t i = 0; i < nvars; ++i)
        if (!canonical_fr(w + 4 * i)) return c->fail(JB_ERR_INVALID, "eq member: point limbs not canonical");
    if (scale_or_null && !canonical_fr(scale_or_null)) return c->fail(JB_ERR_INVALID, "eq member: scale not canonical");
    int st = jb_member_create(c, handles, m, order, out);
    if (st != JB_OK) return st;
    jb_member* mem = *out;
    if (mem->rounds != nvars || nvars == 0) {
        jb_member_destroy(mem);
        *out = nullptr;
        return c->fail(JB_ERR_INVALID, "eq member: point length must equal log2(table length) >= 1");
    }
    {
    Guard g(c);
    mem->eq = true;
    mem->eq_n = nvars;
    mem->eq_split = nvars / 2;
    mem->eq_w.assign(w, w + 4 * nvars);
    HostFr sc = scale_or_null ? HostFr::from_limbs(scale_or_null) : HostFr::one();
    sc.store(mem->eq_scalar);
    if (order == JB_LOW_TO_HIGH) {
        // prefix tables (EqPolynomial::evals_cached, eq.rs:322-340): Eo[k] over w[0..k), Ei[k] over w[split..split+k)
        const size_t split = mem->eq_split, nin = nvars - 1 - (split < nvars - 1 ? split : nvars - 1);
        const size_t out_max = split < nvars - 1 ? split : nvars - 1;
        mem->eq_in_base = ((size_t)2 << out_max) - 1;
        const size_t total = mem->eq_in_base + ((size_t)2 << nin) - 1;
        st = c->dev_alloc((void**)&mem->eq_tabs, total * 32);
        for (size_t k = 0; k <= out_max && st == JB_OK; ++k)
            st = eq_build(c, w, k, nullptr, mem->eq_tabs + 4 * (((size_t)1 << k) - 1));
        for (size_t k = 0; k <= nin && st == JB_OK; ++k)
            st = eq_build(c, w + 4 * split, k, nullptr, mem->eq_tabs + 4 * (mem->eq_in_base + ((size_t)1 << k) - 1));
    } else {
        // HighToLow (split_eq.rs:233-257): tail = w[1..], in_point = tail[..s], out_point = tail[s..] with
        // s = min(n / 2, n - 1); suffix tables (evals_cached_rev): hi[k] = eq(w[1 + k .. 1 + s)), lo[j] = eq(w[1 + s + j .. n))
        const size_t sp = mem->eq_split < nvars - 1 ? mem->eq_split : nvars - 1;
        mem->eq_split = sp;
        const size_t nlo = nvars - 1 - sp;
        size_t total = 0;
        for (size_t k = 0; k <= sp; ++k) {
            mem->eq_hi_off.push_back(total);
            total += (size_t)1 << (sp - k);
        }
        for (size_t j = 0; j <= nlo; ++j) {
            mem->eq_lo_off.push_back(total);
            total += (size_t)1 << (nlo - j);
        }
        st = c->dev_alloc((void**)&mem->eq_tabs, total * 32);
        for (size_t k = 0; k <= sp && st == JB_OK; ++k)
            st = eq_build(c, w + 4 * (1 + k), sp - k, nullptr, mem->eq_tabs + 4 * mem->eq_hi_off[k]);
        for (size_t j = 0; j <= nlo && st == JB_OK; ++j)
            st = eq_build(c, w + 4 * (1 + sp + j), nlo - j, nullptr, mem->eq_tabs + 4 * mem->eq_lo_off[j]);
    }
    }  // the context lock is released before the member is torn down (jb_member_destroy takes it)
    if (st != JB_OK) {
        jb_member_destroy(mem);
        *out = nullptr;
    }
    return st;
}

// eq(w, r) * scale after all rounds (the member's eq factor of the final claim)
int jb_eq_member_scalar(jb_member* mem, uint64_t out[4]) {
    if (!mem || !out || !mem->eq) return JB_ERR_INVALID;
    std::memcpy(out, mem->eq_scalar, 32);
    return JB_OK;
}
// ---- index-sharded member ----------------------------------------------------------------------
// HighToLow shards are strided (rank g owns global[j * G + g]): gathered[g][j] -> global[j * G + g]
static __global__ void __launch_bounds__(256) interleave_shards_kernel(const uint64_t* gathered, uint64_t* global, size_t len,
                                                                       size_t G) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= len * G) return;
    const size_t g = idx / len, j = idx % len;
    st_elem(global, j * G + g, ld_elem<Fr>(gathered, idx));
}

static int gather_into_tail(jb_member* mem) {  // called with the context lock held
    jb_ctx* c = mem->ctx;
    const size_t len = mem->len, G = (size_t)c->world;
    jb_member* tail = new (std::nothrow) jb_member();
    if (!tail) return JB_ERR_OOM;
    tail->ctx = c;
    tail->m = mem->m;
    tail->terms = mem->terms;
    tail->order = mem->order;
    tail->len = len * G;
    tail->rounds = 0;
    while (((size_t)1 << tail->rounds) < tail->len) ++tail->rounds;
    int st = JB_OK;
    for (int j = 0; j < mem->ntables() && st == JB_OK; ++j) {
        Table t;
        st = c->dev_alloc((void**)&t.buf, tail->len * 32);
        if (st != JB_OK) break;
        t.cap = t.len = tail->len;
        tail->tables.push_back(t);  // owned by the tail from here on (released below on failure)
        if (mem->order == JB_LOW_TO_HIGH) {
            // rank order == global order for contiguous blocks under LowToHigh binding
            st = c->comm_allgather(mem->tables[j].buf, t.buf, len * 4);
        } else {
            uint64_t* tmp = nullptr;
            st = c->dev_alloc((void**)&tmp, tail->len * 32);
            if (st == JB_OK) st = c->comm_allgather(mem->tables[j].buf, tmp, len * 4);
            if (st == JB_OK) {
                interleave_shards_kernel<<<(unsigned)((tail->len + 255) / 256), 256, 0, c->stream>>>(tmp, t.buf, len, G);
                c->launches++;
                st = c->check(cudaGetLastError(), "interleave_shards launch");
            }
            c->dev_free(tmp);
        }
    }
    if (st != JB_OK) {
        for (auto& t : tail->tables) c->release(t);
        delete tail;
        return st;
    }
    mem->tail = tail;
    return JB_OK;
}

static int sharded_prove_round(jb_member* mem, const uint64_t* bind, size_t round, const uint64_t* claim,
                               uint64_t* out_evals) {
    jb_ctx* c = mem->ctx;
    {
        Guard g(c, true);
        if (round != mem->rounds_done) return c->fail(JB_ERR_INVALID, "prove_round: round index out of sequence");
        if (bind && !canonical_fr(bind)) return c->fail(JB_ERR_INVALID, "prove_round: challenge limbs not canonical");
        if (mem->gathered) {
            // gathered inside the resident kernel: an ordinary member from here on
            if (bind && mem->len < 4) return c->fail(JB_ERR_INVALID, "prove_round: no round left after this bind (use finish_rounds)");
            const bool skip1 = claim != nullptr && !c->verify_rounds;
            int st = JB_ERR_UNSUPPORTED;
            if (skip1) {
                st = resident_member_prove(mem, bind, claim, round, false, out_evals);
                if (st == JB_OK) mem->rounds_done--;
                if (st != JB_ERR_UNSUPPORTED) return st;
            }
            before_launch(mem);
            st = member_round(mem, bind, skip1, nullptr);
            if (st == JB_OK) st = wait_round_result0(c);
            if (st != JB_OK) return st;
            return assemble_evals(c, mem->m, skip1, c->h_result, claim, round, out_evals);
        }
        if (!mem->tail) {
            const size_t len_after = bind ? mem->len / 2 : mem->len;
            if (len_after > mem->gather_len) {
                // a sharded round: local fused pass -> lanes -> ONE all-reduce -> host fold
                const bool skip1 = claim != nullptr && !c->verify_rounds;
                const int K = skip1 ? mem->m : mem->m + 1;
                int st = JB_ERR_UNSUPPORTED;
                if (skip1 && c->xch_ready) {
                    // resident kernel: the all-reduce over NVLink peer memory rides in the round's own epilogue,
                    // no launch and no NCCL call per round
                    st = resident_member_prove(mem, bind, claim, round, true, out_evals);
                    if (st == JB_OK) mem->rounds_done--;  // (the caller counts sharded rounds)
                    if (st != JB_ERR_UNSUPPORTED) return st;
                }
                if (st == JB_ERR_UNSUPPORTED) {
                    before_launch(mem);
                    if (c->xch_ready) {
                        st = member_round(mem, bind, skip1, JB_LANES_EXCHANGE);
                    } else {
                        st = member_round(mem, bind, skip1, c->d_lanes);
                        if (st == JB_OK) st = c->comm_allreduce_lanes(c->d_lanes, (size_t)K * 8);
                        if (st == JB_OK) st = c->publish_lanes(c->d_lanes, K * 8);
                    }
                    if (st == JB_OK) st = wait_round_result0(c);
                    if (st != JB_OK) return st;
                    if (c->h_result[0] == ~0ull && c->h_result[1] == ~0ull)
                        return c->fail(JB_ERR_CUDA, "peer exchange timed out (a rank did not arrive)");
                }
                uint64_t vals[jb::JB_MEMBER_EVALS * 4];
                st = jb_lanes_reduce_host(c->h_result, (size_t)K, vals);
                if (st != JB_OK) return st;
                return assemble_evals(c, mem->m, skip1, vals, claim, round, out_evals);
            }
            // the shard is small. If its resident kernel is alive and the arena holds the gathered tables, the
            // kernel itself gathers: it binds, writes the bound shard into every rank's arena over NVLink, waits for
            // the peers' shards and sweeps the gathered tables - no kernel exit, no NCCL call; from here on this
            // member proves its remaining rounds un-sharded (identically on every rank)
            const bool skip1g = claim != nullptr && !c->verify_rounds;
            if (bind && skip1g && mem->run && len_after == mem->gather_len && resident_gather_fits(c, mem, len_after)) {
                int st = resident_member_prove(mem, bind, claim, round, false, out_evals, true);
                if (st == JB_OK) {
                    mem->rounds_done--;  // (the caller counts sharded rounds)
                    mem->gathered = true;
                }
                return st;
            }
            // otherwise: stop the resident kernel (its tables are consistent at a round boundary),
            // apply the pending bind, gather with NCCL, continue on the tail
            if (mem->run) resident_end(mem->run, false);
            c->quiesce_resident(false);
            if (bind) {
                for (int j = 0; j < mem->ntables(); ++j) {
                    int st = bind_table(c, mem->tables[j], bind, mem->order);
                    if (st != JB_OK) return st;
                }
                mem->len /= 2;
                bind = nullptr;
            }
            int st = gather_into_tail(mem);
            if (st != JB_OK) return st;
        }
    }
    return jb_member_prove_round(mem->tail, bind, mem->tail->rounds_done, claim, out_evals);
}

int jb_sharded_member_create(jb_ctx* c, const jb_table* handles, size_t m, int order, size_t gather_log, jb_member** out) {
    if (!c || !out) return JB_ERR_INVALID;
    if (!c->nccl_comm) return c->fail(JB_ERR_INVALID, "sharded member: no communicator (jb_comm_init)");
    if (order != JB_LOW_TO_HIGH && order != JB_HIGH_TO_LOW) return c->fail(JB_ERR_INVALID, "sharded member: unknown binding order");
    // the per-round lanes and the peer exchange slots hold K <= 5 sums: sharded members stay at 1..4 tables
    if (m < 1 || m > 4) return c->fail(JB_ERR_UNSUPPORTED, "sharded member: m must be 1..4");
    int st = jb_member_create(c, handles, m, order, out);
    if (st != JB_OK) return st;
    jb_member* mem = *out;
    size_t log_g = 0;
    while ((1 << log_g) < c->world) ++log_g;
    mem->sharded = true;
    mem->gather_len = (size_t)1 << gather_log;
    if (mem->gather_len > mem->len) mem->gather_len = mem->len;
    mem->rounds += log_g;
    return JB_OK;
}

int jb_member_prove_round_partials(jb_member* mem, const uint64_t* bind, size_t round, int skip_t1, void* lanes_out) {
    (void)round;
    if (!mem || !lanes_out) return JB_ERR_INVALID;
    Guard g(mem->ctx, true);
    // the lanes of K <= 5 sums (K * 8 u64) are what the partials path reduces and exchanges
    if (mem->m > 4) return mem->ctx->fail(JB_ERR_UNSUPPORTED, "partials: members of 1..4 tables only");
    before_launch(mem);
    return member_round(mem, bind, skip_t1 != 0, lanes_out);
}

int jb_ctx_set_verify_rounds(jb_ctx* c, int on) {
    if (!c) return JB_ERR_INVALID;
    Guard g(c);
    c->verify_rounds = on != 0;
    return JB_OK;
}

// carry-propagate 8 x (sums of 32-bit limbs) and fold mod r: O(count) host work, no device needed.
int jb_lanes_reduce_host(const uint64_t* lanes, size_t count, uint64_t* out) {
    if (!lanes || !out) return JB_ERR_INVALID;
    for (size_t k = 0; k < count; ++k) {
        const uint64_t* lane = lanes + 8 * k;
        uint32_t w[10];
        unsigned __int128 carry = 0;
        for (int i = 0; i < 8; ++i) {
            carry += lane[i];
            w[i] = (uint32_t)carry;
            carry >>= 32;
        }
        w[8] = (uint32_t)carry;
        w[9] = (uint32_t)(carry >> 32);
        // value < 2^32 * r < 2^286; fold by subtracting (r << sh) from the top down
        uint64_t v[5] = {(uint64_t)w[0] | ((uint64_t)w[1] << 32), (uint64_t)w[2] | ((uint64_t)w[3] << 32),
                         (uint64_t)w[4] | ((uint64_t)w[5] << 32), (uint64_t)w[6] | ((uint64_t)w[7] << 32),
                         (uint64_t)w[8] | ((uint64_t)w[9] << 32)};
        for (int sh = 33; sh >= 0; --sh) {
            uint64_t ps[5] = {0, 0, 0, 0, 0};  // r << sh
            for (int i = 0; i < 4; ++i) {
                ps[i] |= sh ? (HostFr::P[i] << sh) : HostFr::P[i];
                if (sh) ps[i + 1] |= HostFr::P[i] >> (64 - sh);
            }
            bool ge = true;
            for (int i = 4; i >= 0; --i)
                if (v[i] != ps[i]) { ge = v[i] > ps[i]; break; }
            if (ge) {
                uint64_t borrow = 0;
                for (int i = 0; i < 5; ++i) {
                    unsigned __int128 t = (unsigned __int128)v[i] - ps[i] - borrow;
                    v[i] = (uint64_t)t;
                    borrow = (uint64_t)(t >> 64) & 1;
                }
            }
        }
        std::memcpy(out + 4 * k, v, 32);
    }
    return JB_OK;
}

// The serial tail of a round of the resident kernel: `count` values, each the 17 u64 lanes of a block-summed
// unreduced accumulator sum_y a_y b_y over Montgomery operands (lane w = sum of the 32-bit limbs of weight 2^(32 w),
// < 2^64). V = sum_w lane_w 2^(32 w) < 2^577 = lo + h0 2^256 + h1 2^512; the field value is V R^-1 mod p =
// REDC(lo) + h0 + h1 R, each term one word-serial Montgomery product with the wide operand as the multiplier.
int jb_wide_lanes_reduce_host(const uint64_t* lanes, size_t count, uint64_t* out) {
    if (!lanes || !out) return JB_ERR_INVALID;
    static const HostFr raw_one{{1, 0, 0, 0}};
    static const HostFr r1{{HostFr::R1[0], HostFr::R1[1], HostFr::R1[2], HostFr::R1[3]}};
    static const HostFr r2{{HostFr::R2[0], HostFr::R2[1], HostFr::R2[2], HostFr::R2[3]}};
    for (size_t k = 0; k < count; ++k) {
        const uint64_t* lane = lanes + 17 * k;
        uint32_t w[20];
        unsigned __int128 carry = 0;
        for (int i = 0; i < 17; ++i) {
            carry += lane[i];
            w[i] = (uint32_t)carry;
            carry >>= 32;
        }
        for (int i = 17; i < 20; ++i) {
            w[i] = (uint32_t)carry;
            carry >>= 32;
        }
        HostFr lo, h0, h1;
        for (int i = 0; i < 4; ++i) {
            lo.l[i] = (uint64_t)w[2 * i] | ((uint64_t)w[2 * i + 1] << 32);
            h0.l[i] = (uint64_t)w[8 + 2 * i] | ((uint64_t)w[8 + 2 * i + 1] << 32);
        }
        h1 = HostFr{{(uint64_t)w[16] | ((uint64_t)w[17] << 32), (uint64_t)w[18] | ((uint64_t)w[19] << 32), 0, 0}};
        const HostFr v = raw_one * lo + r1 * h0 + r2 * h1;
        v.store(out + 4 * k);
    }
    return JB_OK;
}

// lanes of one member's round (as the resident kernel publishes them) -> K canonical values
static int resident_values(int D, const uint64_t* lanes, uint64_t* vals) {
    return D == 1 ? jb_lanes_reduce_host(lanes, 1, vals) : jb_wide_lanes_reduce_host(lanes, (size_t)D, vals);
}

int jb_partials_finalize(jb_ctx* c, const void* device_lanes, size_t count, uint64_t* out) {
    if (!c || !device_lanes || !out || count == 0 || count * 64 > JB_SMALL_BYTES) return JB_ERR_INVALID;
    Guard g(c);
    int st = c->check(cudaMemcpyAsync(c->h_small, device_lanes, count * 64, cudaMemcpyDeviceToHost, c->stream),
                      "partials D2H");
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "partials sync");
    if (st != JB_OK) return st;
    return jb_lanes_reduce_host(c->h_small, count, out);
}


// Copies table j of a member (its current, possibly partly bound, contents) into caller device memory.
int jb_member_export_table(jb_member* mem, size_t j, void* device_dst, size_t cap_elems, size_t* len_out) {
    if (!mem || !device_dst) return JB_ERR_INVALID;
    jb_ctx* c = mem->ctx;
    Guard g(c, true);
    before_launch(mem);  // the host's view of the tables (buffer parity, length) is exact at a round boundary
    if (j >= (size_t)mem->ntables()) return c->fail(JB_ERR_INVALID, "export_table: table index out of range");
    if (cap_elems < mem->len) return c->fail(JB_ERR_INVALID, "export_table: destination too small");
    if (len_out) *len_out = mem->len;
    return c->check(cudaMemcpyAsync(device_dst, mem->tables[j].buf, mem->len * 32, cudaMemcpyDeviceToDevice, c->stream),
                    "export_table D2D");
}

int jb_member_finish_rounds(jb_member* mem, const uint64_t bind[4]) {
    if (!mem || !bind) return JB_ERR_INVALID;
    jb_ctx* c = mem->ctx;
    if (mem->sharded && !mem->gathered) {
        if (!mem->tail) return c->fail(JB_ERR_INVALID, "finish_rounds: sharded member has not reached its tail");
        return jb_member_finish_rounds(mem->tail, bind);
    }
    Guard g(c, true);
    if (mem->len < 2) return c->fail(JB_ERR_INVALID, "finish_rounds: member already fully bound");
    if (!canonical_fr(bind)) return c->fail(JB_ERR_INVALID, "finish_rounds: challenge limbs not canonical");
    if (mem->eq) {
        size_t var = 0;
        for (size_t l = mem->len; l > 2; l >>= 1) ++var;  // unbound variables besides the one being bound
        // LowToHigh binds w[var] (the most significant unbound one is w[0]); HighToLow binds w[n - 1 - var]
        eq_absorb_bind(mem, mem->order == JB_LOW_TO_HIGH ? var : mem->eq_n - 1 - var, bind);
    }
    if (mem->run) {
        // the terminal bind is one more mailbox command; a fully bound member gets its values back with the
        // acknowledgement (has_final), so nothing is read from the device afterwards
        return resident_member_final(mem, bind);
    }
    before_launch(mem);
    for (int j = 0; j < mem->ntables(); ++j) {
        int st = bind_table(c, mem->tables[j], bind, mem->order);
        if (st != JB_OK) return st;
    }
    mem->len /= 2;
    return JB_OK;
}

int jb_member_final_evals(jb_member* mem, uint64_t* out) {
    if (!mem || !out) return JB_ERR_INVALID;
    jb_ctx* c = mem->ctx;
    if (mem->sharded && !mem->gathered) {
        if (!mem->tail) return c->fail(JB_ERR_INVALID, "NotFullyBound (sharded member before its tail)");
        return jb_member_final_evals(mem->tail, out);
    }
    Guard g(c, true);
    const int T = mem->ntables();
    if (mem->has_final) {
        std::memcpy(out, mem->final_vals, (size_t)T * 32);
        return JB_OK;
    }
    if (mem->len != 1) {
        char buf[96];
        size_t remaining = 0;
        for (size_t l = mem->len; l > 1; l >>= 1) ++remaining;
        std::snprintf(buf, sizeof buf, "NotFullyBound { remaining: %zu }", remaining);
        return c->fail(JB_ERR_INVALID, buf);
    }
    before_launch(mem);
    for (int j = 0; j < T; ++j) {
        int st = c->check(cudaMemcpyAsync(c->h_small + 4 * j, mem->tables[j].buf, 32, cudaMemcpyDeviceToHost, c->stream),
                          "final evals D2H");
        if (st != JB_OK) return st;
    }
    int st = c->check(cudaStreamSynchronize(c->stream), "final evals sync");
    if (st != JB_OK) return st;
    std::memcpy(out, c->h_small, (size_t)T * 32);
    return JB_OK;
}

void jb_member_destroy(jb_member* mem) {
    if (!mem) return;
    if (mem->tail) jb_member_destroy(mem->tail);
    Guard g(mem->ctx, true);
    if (mem->run) resident_end(mem->run, false);
    if (mem->eq_tabs) mem->ctx->dev_free(mem->eq_tabs);
    for (auto& t : mem->tables) mem->ctx->release(t);
    delete mem;
}

// ---- device RoundScheduler (crates/jolt-sumcheck/src/prover.rs:106-120; BuildRoundScheduler,
//      crates/jolt-kernels/src/backend.rs:64-70) ------------------------------------------------------------
// "Order and transport are free": a batch round costs ONE host round trip whatever the member count.
//   * homogeneous batches (same shape and order, <= RES_MAX_MEMBERS members) are served by ONE resident kernel:
//     a single mailbox command carries every member's action and the shared challenge, the kernel answers
//     with every member's round sums;
//   * otherwise every active member's pass is enqueued before the first wait (one result slot per member;
//     short members through their own small resident kernels), then the results are collected.
struct jb_scheduler {
    jb_ctx* ctx;
    std::vector<jb_member*> members;
    bool homogeneous = false;
    bool run_failed = false;  // a resident batch could not be started: stay on the overlapped launches
};

int jb_scheduler_create(jb_ctx* c, jb_member** members, size_t n, jb_scheduler** out) {
    if (!c || !members || !out || n == 0) return JB_ERR_INVALID;
    Guard g(c, true);
    jb_scheduler* s = new (std::nothrow) jb_scheduler();
    if (!s) return JB_ERR_OOM;
    s->ctx = c;
    s->homogeneous = n <= (size_t)RES_MAX_MEMBERS;
    for (size_t i = 0; i < n; ++i) {
        jb_member* m = members[i];
        if (!m || m->ctx != c) {
            delete s;
            return c->fail(JB_ERR_INVALID, "scheduler: members must belong to the scheduler's context");
        }
        for (size_t k = 0; k < i; ++k)
            if (members[k] == m) {
                delete s;
                return c->fail(JB_ERR_INVALID, "scheduler: duplicate member");
            }
        // out_evals carries JB_MAX_EVALS values per work item: a member of higher degree runs outside the scheduler
        if ((size_t)m->m + (m->eq ? 1 : 0) + 1 > (size_t)JB_MAX_EVALS) {
            delete s;
            return c->fail(JB_ERR_UNSUPPORTED, "scheduler: members of degree > 7 do not fit the 8 evaluations per work item");
        }
        s->members.push_back(m);
        if (m->sharded || m->eq || m->m != members[0]->m || m->terms != members[0]->terms || m->order != members[0]->order)
            s->homogeneous = false;
    }
    *out = s;
    return JB_OK;
}

void jb_scheduler_destroy(jb_scheduler* s) { delete s; }

// starts the batch's resident kernel over every member that still has rounds to prove
static int scheduler_begin_run(jb_scheduler* s) {
    jb_ctx* c = s->ctx;
    std::vector<jb_member*> live;
    for (auto* m : s->members) {
        if (m->run) return JB_ERR_UNSUPPORTED;  // already served by another run
        if (m->len >= 2) {
            if (!resident_eligible(m)) return JB_ERR_UNSUPPORTED;
            live.push_back(m);
        }
    }
    if (live.empty()) return JB_ERR_UNSUPPORTED;
    return resident_begin(c, live.data(), (int)live.size());
}

int jb_scheduler_prove_round(jb_scheduler* s, const jb_round_work* work, size_t n_work, uint64_t* out_evals) {
    if (!s || (n_work && (!work || !out_evals))) return JB_ERR_INVALID;
    jb_ctx* c = s->ctx;
    // sharded members synchronise across ranks inside their own round: no overlap to win, run them in order
    for (size_t i = 0; i < n_work; ++i) {
        if (work[i].member >= s->members.size()) return c->fail(JB_ERR_INVALID, "scheduler: member index out of range");
        if (s->members[work[i].member]->sharded) {
            for (size_t k = 0; k < n_work; ++k) {
                const jb_round_work& w = work[k];
                int st = jb_member_prove_round(s->members[w.member], w.has_bind ? w.bind : nullptr, w.round,
                                               w.has_claim ? w.claim : nullptr, out_evals + k * JB_MAX_EVALS * 4);
                if (st != JB_OK) return st;
            }
            return JB_OK;
        }
    }
    Guard g(c, true);
    const uint64_t* shared_bind = nullptr;
    bool all_skip1 = !c->verify_rounds, same_bind = true;
    for (size_t i = 0; i < n_work; ++i) {
        const jb_round_work& w = work[i];
        jb_member* m = s->members[w.member];
        for (size_t k = 0; k < i; ++k)
            if (work[k].member == w.member) return c->fail(JB_ERR_INVALID, "scheduler: a member appears twice in one round");
        if (w.round != m->rounds_done) return c->fail(JB_ERR_INVALID, "prove_round: round index out of sequence");
        if ((m->rounds_done == 0) != (w.has_bind == 0))
            return c->fail(JB_ERR_INVALID, "prove_round: bind must be absent exactly on the first round");
        if (w.has_bind && !canonical_fr(w.bind)) return c->fail(JB_ERR_INVALID, "prove_round: challenge limbs not canonical");
        if (w.has_claim && !canonical_fr(w.claim)) return c->fail(JB_ERR_INVALID, "prove_round: claim limbs not canonical");
        if (m->len < (w.has_bind ? 4u : 2u)) return c->fail(JB_ERR_INVALID, "prove_round: member has no round left");
        if (!w.has_claim) all_skip1 = false;
        if (w.has_bind) {
            if (shared_bind && std::memcmp(shared_bind, w.bind, 32) != 0) same_bind = false;
            shared_bind = w.bind;
        }
    }
    // ---- one resident kernel for the whole batch -------------------------------------------------------
    if (s->homogeneous && !s->run_failed && all_skip1 && same_bind && c->use_tail && n_work) {
        ResidentRun* run = s->members[work[0].member]->run;
        bool ok = true;
        if (!run) {
            int st = scheduler_begin_run(s);
            if (st == JB_OK) run = s->members[work[0].member]->run;
            else if (st == JB_ERR_UNSUPPORTED) ok = false;
            else return st;
        }
        for (size_t i = 0; ok && i < n_work; ++i) ok = s->members[work[i].member]->run == run;
        if (ok && run) {
            RunItem items[RES_MAX_MEMBERS];
            for (size_t i = 0; i < n_work; ++i)
                items[i] = RunItem{s->members[work[i].member], work[i].has_bind ? work[i].bind : nullptr, work[i].claim,
                                   work[i].round, out_evals + i * JB_MAX_EVALS * 4};
            int st = run_round(c, run, items, (int)n_work, shared_bind, false);
            if (st != JB_OK && s->members[work[0].member]->run) resident_end(s->members[work[0].member]->run, true);
            return st;
        }
        s->run_failed = true;
    }
    // ---- overlapped: enqueue every member's pass, then collect -----------------------------------------
    if (n_work >= JB_RESULT_SLOTS) return c->fail(JB_ERR_UNSUPPORTED, "scheduler: too many active members in one round");
    c->quiesce_resident(false);
    enum { VIA_LAUNCH = 0, VIA_RUN = 1 };
    int via[JB_RESULT_SLOTS];
    uint64_t seqs[JB_RESULT_SLOTS];
    bool skip[JB_RESULT_SLOTS];
    for (size_t i = 0; i < n_work; ++i) {
        const jb_round_work& w = work[i];
        jb_member* m = s->members[w.member];
        const uint64_t* bind = w.has_bind ? w.bind : nullptr;
        skip[i] = w.has_claim && !c->verify_rounds;
        via[i] = VIA_LAUNCH;
        if (m->eq) {  // the Gruen member needs host work between its launch and its result: run it in place
            int st = eq_prove_round(m, bind, w.round, w.has_claim ? w.claim : nullptr, out_evals + i * JB_MAX_EVALS * 4);
            if (st != JB_OK) return st;
            m->rounds_done++;
            via[i] = -1;
            continue;
        }
        const size_t len_after = bind ? m->len / 2 : m->len;
        if (skip[i] && len_after <= RES_SMALL_LEN && (m->run || resident_eligible(m))) {
            // short member: its own small resident kernel (a few blocks), one mailbox command
            if (!m->run) {
                jb_member* one[1] = {m};
                int st = resident_begin(c, one, 1, len_after, false);
                if (st != JB_OK && st != JB_ERR_UNSUPPORTED) return st;
            }
            if (m->run && resident_run_size(m->run) == 1) {
                unsigned actions[RES_MAX_MEMBERS] = {0};
                actions[m->run_idx] = bind ? RES_ACT_BIND_EVAL : RES_ACT_EVAL;
                int st = JB_OK;
                while (st == JB_OK && resident_inflight(m->run) > 0) st = resident_consume(m->run, nullptr, nullptr);
                if (st == JB_OK) st = resident_post(m->run, actions, bind, false);
                if (st == JB_RES_LOST) st = resident_recover(m->run);  // back to launches (below)
                else if (st != JB_OK) return st;
                else {
                    m->look_ok = false;
                    via[i] = VIA_RUN;
                    continue;
                }
                if (st != JB_OK) return st;
            }
        }
        if (m->run) resident_end(m->run, true);
        int st = member_round(m, bind, skip[i], nullptr, nullptr, (int)i + 1, &seqs[i]);
        if (st != JB_OK) return st;
    }
    for (size_t i = 0; i < n_work; ++i) {
        if (via[i] < 0) continue;
        const jb_round_work& w = work[i];
        jb_member* m = s->members[w.member];
        int st;
        if (via[i] == VIA_RUN) {
            uint64_t out[RES_MAX_MEMBERS * RES_SLOT_U64];
            ResConsumed info[RES_MAX_MEMBERS];
            st = resident_consume(m->run, out, info);
            if (st == JB_RES_LOST) {  // recover (replays this round's bind), then an eval-only launch
                st = resident_recover(m->run);
                if (st == JB_OK) st = member_round(m, nullptr, true, nullptr);
                if (st == JB_OK) st = wait_round_result0(c);
                if (st == JB_OK) st = assemble_evals(c, m->m, true, c->h_result, w.claim, w.round, out_evals + i * JB_MAX_EVALS * 4);
            } else if (st == JB_OK) {
                uint64_t vals[jb::JB_MEMBER_EVALS * 4];
                answer_values(m, info[0], out, vals);
                st = assemble_evals(c, m->m, true, vals, w.claim, w.round, out_evals + i * JB_MAX_EVALS * 4);
            }
        } else {
            st = wait_round_result(c, (int)i + 1, seqs[i]);
            if (st == JB_OK)
                st = assemble_evals(c, m->m, skip[i], c->h_result + (i + 1) * JB_SLOT_U64, w.has_claim ? w.claim : nullptr, w.round,
                                    out_evals + i * JB_MAX_EVALS * 4);
        }
        if (st != JB_OK) return st;
        m->rounds_done++;
    }
    return JB_OK;
}

int jb_scheduler_finish_rounds(jb_scheduler* s, const jb_finish_work* work, size_t n_work) {
    if (!s || (n_work && !work)) return JB_ERR_INVALID;
    jb_ctx* c = s->ctx;
    {
        Guard g(c, true);
        // every finishing member of one resident run takes its terminal bind in ONE command
        ResidentRun* run = nullptr;
        bool one_run = n_work > 0;
        for (size_t i = 0; i < n_work && one_run; ++i) {
            if (work[i].member >= s->members.size()) return c->fail(JB_ERR_INVALID, "scheduler: member index out of range");
            jb_member* m = s->members[work[i].member];
            if (!m->run || m->eq || m->sharded || m->len != 2 || !canonical_fr(work[i].bind)) one_run = false;
            else if (!run) run = m->run;
            else if (m->run != run) one_run = false;
            if (one_run && std::memcmp(work[0].bind, work[i].bind, 32) != 0) one_run = false;
        }
        if (one_run && run) {
            unsigned actions[RES_MAX_MEMBERS] = {0};
            for (size_t i = 0; i < n_work; ++i) actions[s->members[work[i].member]->run_idx] = RES_ACT_FINAL;
            int st = resident_round(run, actions, work[0].bind, false, nullptr);
            return st == JB_RES_LOST ? resident_recover(run) : st;
        }
    }
    for (size_t i = 0; i < n_work; ++i) {
        if (work[i].member >= s->members.size()) return c->fail(JB_ERR_INVALID, "scheduler: member index out of range");
        int st = jb_member_finish_rounds(s->members[work[i].member], work[i].bind);
        if (st != JB_OK) return st;
    }
    return JB_OK;
}

}  // extern "C"
