// Internals shared by the sumcheck-member translation units (member.cu, resident.cu, capi.cu).
#pragma once
#include <cstring>
#include <ctime>
#include <vector>

#include "ctx.hpp"
#include "host_fr.hpp"
#include "poly_kernels.cuh"
#include "resident.cuh"

namespace jbi {

using jb::BindScalar;
using jb::HostFr;

inline uint64_t now_ns() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec;
}

inline BindScalar make_scalar(const uint64_t r[4], bool* hi4) {
    BindScalar s;
    for (int i = 0; i < 4; ++i) {
        s.w[2 * i] = (uint32_t)r[i];
        s.w[2 * i + 1] = (uint32_t)(r[i] >> 32);
    }
    *hi4 = (r[0] == 0 && r[1] == 0);
    return s;
}

inline bool canonical_fr(const uint64_t r[4]) { return !HostFr::geq_p(r); }

// capi.cu
int bind_table(jb_ctx* c, Table& t, const uint64_t r[4], int order);  // Polynomial::bind_with_order on one table
int eq_build(jb_ctx* c, const uint64_t* r, size_t nvars, const uint64_t* scale, uint64_t* d_out);

// wide_product.cu: one round of a product of m = 5..8 tables, or (weighted) of a split-eq member of m = 4..8 tables
// (always SKIP1), with the outputs of fused_round_kernel; JB_ERR_UNSUPPORTED for any other m.
int launch_wide_round(jb_ctx* c, int m, int order, bool skip1, bool weighted, const jb::TablePtrs& tp, size_t pairs,
                      bool bind, bool hi4, const BindScalar& s, const jb::RoundOut& out);

// Accumulates the host time spent waiting for a round result (jb_ctx_diag).
struct WaitAcc {
    jb_ctx* c;
    uint64_t t0;
    explicit WaitAcc(jb_ctx* ctx) : c(ctx), t0(now_ns()) {}
    ~WaitAcc() {
        c->diag_wait_ns += now_ns() - t0;
        c->diag_waits++;
    }
};

}  // namespace jbi

// One ProveRounds member on the device (~ Box<dyn SumcheckKernel>): the relation
//   sum_x sum_{k<P} prod_{j<D} f_{kD+j}(x)       (degree D, T = D * P dense tables)
// optionally weighted by a split eq polynomial, optionally index-sharded over ranks.
struct jb_member {
    jb_ctx* ctx;
    std::vector<Table> tables;
    int m;       // D: factors per term = degree of the (unweighted) relation
    int terms = 1;  // P
    int order;
    size_t rounds;  // total (for a sharded member: local rounds + log2(world))
    size_t len;     // current (local) table length
    size_t rounds_done = 0;  // prove_round calls completed
    // index-sharded member (SURVEY 8e): this rank holds the contiguous block `rank` of the global
    // tables; rounds run with one all-reduce each until the shard is `gather_len` long, then the
    // shards are all-gathered into `tail`, which finishes the remaining rounds locally.
    bool sharded = false;
    size_t gather_len = 0;
    jb_member* tail = nullptr;
    bool gathered = false;  // the shards were gathered inside the resident kernel: the member continues un-sharded
    // split-eq member (GruenSplitEqPolynomial, crates/jolt-poly/src/split_eq.rs:159-447): the relation is
    // sum_x eq(w, x) prod_j f_j(x); eq is never materialised - per round the sweep is weighted by
    // E_out (x) E_in over the not-yet-current variables and the current variable's linear factor
    // l(t) = scalar * ((1 - w_cur) + t (2 w_cur - 1)) is multiplied in on the host.
    bool eq = false;
    size_t eq_n = 0, eq_split = 0;
    std::vector<uint64_t> eq_w;        // n elements, w[0] <-> most significant index bit
    uint64_t eq_scalar[4] = {0, 0, 0, 0};
    uint64_t* eq_tabs = nullptr;       // prefix tables Eo[k] (k <= split) then Ei[k] (k <= n-1-split), table k at 2^k - 1
    size_t eq_in_base = 0;             // element offset of the Ei family
    std::vector<size_t> eq_hi_off, eq_lo_off;  // HighToLow: element offsets of the suffix tables (see jb_eq_member_create)
    // resident service (resident.cuh): the launched kernel that serves this member's rounds from a mailbox
    ResidentRun* run = nullptr;
    int run_idx = 0;
    bool no_resident = false;  // a run of this member was stopped to make room for other work: stay on launches
    bool has_final = false;
    uint64_t final_vals[jb::JB_MAX_TABLES * 4];
    // lookahead (thin rounds, resident.cuh): the sums S0..S5 that determine round `look_round`'s polynomial as a
    // function of the challenge that round binds - harvested from the answer to the previous round's command
    bool look_ok = false;
    size_t look_round = 0;
    uint64_t look[6 * 4];
    int ntables() const { return m * terms; }
};

// resident.cu ------------------------------------------------------------------------------------------------
// Starts a resident kernel serving `n` members (same D, P, order, same context; n <= RES_MAX_MEMBERS). Members
// must be plain (not eq / sharded-with-tail). `exchange`: the kernel may be asked to all-reduce member 0's sums
// over peer memory (sharded rounds). JB_ERR_UNSUPPORTED = not eligible (caller falls back to launches).
// first_len: entries of the largest pass a single-member run will be asked for (0 = the member's current length);
// may_evict: stop other runs of the context if the device cannot hold this one next to them (false:
// JB_ERR_UNSUPPORTED instead).
int resident_begin(jb_ctx* c, jb_member** mems, int n, uint64_t first_len = 0, bool may_evict = true);
// What a consumed command had asked of member i of the run.
struct ResConsumed {
    unsigned act = 0;       // RES_ACT_*
    bool thin = false;      // the answer carries the 8 thin sums (x 17 lanes) instead of K sums
    size_t round = 0;       // member-local round the command proved
    uint64_t nprime = 0;    // entries of the tables the round swept (after its bind)
};
// One launched resident_rounds_kernel and the members it serves.
struct ResidentRun {
    jb_ctx* c = nullptr;
    TailRes res;
    jb::ResMailbox* mb = nullptr;  // host view of the mailbox
    uint64_t seq = 0;          // commands posted
    uint64_t consumed = 0;     // answers consumed (<= seq <= consumed + 2: the mailbox is a ring of two)
    int n = 0;
    jb_member* mem[jb::RES_MAX_MEMBERS] = {nullptr};
    unsigned grid = 0;
    ResConsumed ring[2][jb::RES_MAX_MEMBERS];  // what command s (slot s & 1) asked of every member
    uint64_t ring_challenge[2][4];             // ... and the challenge it carried (to replay it if the kernel is lost)
    bool ring_gather[2] = {false, false};      // ... and whether it was a gather (not replayable)
    std::vector<Table> deferred;               // shard buffers a gather made obsolete: freed when the run ends
    struct RoundInfo { int kind; uint64_t items; int m; };
    RoundInfo info[64];                       // what command s (< 64) asked for, for the device-timed pass log
    uint64_t host_post[64], host_recv[64];    // CLOCK_MONOTONIC ns (diagnostics)
    bool kernel_live = false;
    bool exclusive = false;  // holds more than half of the device's block slots: other kernels may starve
};

// The mailbox is a ring of two commands. post: actions[i] in RES_ACT_* (challenge may be null when no action binds);
// the host's view of the tables (len, ping-pong) advances at once - the device executes commands in order.
// consume: waits for the OLDEST unanswered command; `out` (may be null) receives n x RES_SLOT_U64 mailbox words per
// member (lanes, see resident.cuh; with `exchange` member 0's lanes are all-reduced over the ranks), `info` what
// the command had asked. The run is released when every member is fully bound and nothing is in flight (the run
// pointer is dead after that: check mem->run). round = drain + post + consume.
// gather (single-member run of an index-sharded member, action BIND_EVAL): bind, scatter the bound shard into every
// rank's arena and sweep the gathered tables; afterwards the member's tables ARE its arena views (len x world).
int resident_post(ResidentRun* run, const unsigned* actions, const uint64_t* challenge, bool exchange, bool gather = false);
bool resident_gather_fits(const jb_ctx* c, const jb_member* mem, uint64_t shard_len_after_bind);
int resident_consume(ResidentRun* run, uint64_t* out, ResConsumed* info);
int resident_inflight(const ResidentRun* run);
// resident_consume returns JB_RES_LOST when the kernel gave up waiting for commands (the host was held up for
// ~10 s: a debugger, a tool patching a module, an absorb callback that blocks) and exited WITHOUT executing the
// commands still in flight. The tables are consistent at the last executed round. resident_recover then replays
// the unexecuted commands' binds with ordinary launches (the host's view of the tables is exact again), releases the
// run and marks its members for one launch per round; the caller recomputes the current round's sums with an
// eval-only launch. A member never fails because its resident kernel went away.
constexpr int JB_RES_LOST = -1000;
int resident_recover(ResidentRun* run);
int resident_round(ResidentRun* run, const unsigned* actions, const uint64_t* challenge, bool exchange, uint64_t* out);
int resident_run_size(const ResidentRun* run);
// Stops the kernel (if it still runs), orders the context's stream after it and detaches the members.
void resident_end(ResidentRun* run, bool mark_no_resident);
bool resident_eligible(const jb_member* mem);
