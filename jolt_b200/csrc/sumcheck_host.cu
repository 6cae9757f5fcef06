// Host-side sumcheck engine over device-backed members: the C++ mirror of
//   jolt_sumcheck::prove_batch           crates/jolt-sumcheck/src/prover.rs:193-362
//   ProveRounds / SequentialRounds       crates/jolt-sumcheck/src/prover.rs:52-72, 127-148
//   UnivariatePoly::{from_evals,evaluate} crates/jolt-poly/src/univariate.rs:58-69, 198-202
// The Rust toolchain is absent from this image, so the host side above the C ABI is C++ (the
// reference is compiled code); the Rust adapter a maintainer would write is in INTEGRATION.md.
// Everything here is O(members * rounds * degree) field work; tables never leave the device.
#include <cstring>
#include <vector>

#include "../../include/jolt_b200.h"
#include "host_fr.hpp"
#include "sumcheck_host.hpp"

namespace jb {

// ---- UnivariatePoly ---------------------------------------------------------------------------
HostFr UnivariatePoly::evaluate(const HostFr& x) const {
    if (coefficients.empty()) return HostFr::zero();
    HostFr acc = coefficients.back();
    for (size_t i = coefficients.size() - 1; i-- > 0;) acc = acc * x + coefficients[i];
    return acc;
}

// Interpolation on nodes 0..n-1. The reference solves the Vandermonde system by Gaussian
// elimination (univariate.rs:470-487); the interpolant is unique, so Newton's divided
// differences on equally spaced nodes give identical coefficients.
namespace {
// 1/k! for k < 32, computed once (a field inversion is ~400 multiplications - far too slow to
// repeat on the per-round latency path).
const HostFr* inverse_factorials() {
    static HostFr table[32];
    static bool init = [] {
        HostFr f = HostFr::one();
        table[0] = f;
        for (uint64_t k = 1; k < 32; ++k) {
            f = f * HostFr::from_u64(k);
            table[k] = f.inverse();
        }
        return true;
    }();
    (void)init;
    return table;
}
}  // namespace

UnivariatePoly UnivariatePoly::from_evals(const std::vector<HostFr>& evals) {
    const size_t n = evals.size();
    UnivariatePoly out;
    out.coefficients.assign(n, HostFr::zero());
    if (n == 0) return out;
    // This runs once per member per round on the Fiat-Shamir round trip: no heap traffic beyond the result for the
    // degrees a sumcheck sees (n <= 16); larger inputs take the same path with heap scratch.
    constexpr size_t STACK_N = 16;
    HostFr stack_scratch[3 * STACK_N + 1];
    std::vector<HostFr> heap_scratch;
    HostFr* scratch = stack_scratch;
    if (n > STACK_N) {
        heap_scratch.resize(3 * n + 1);
        scratch = heap_scratch.data();
    }
    HostFr* diff = scratch;              // n
    HostFr* newton = scratch + n;        // n
    HostFr* basis = scratch + 2 * n;     // n + 1
    const HostFr* inv_fact = inverse_factorials();
    for (size_t i = 0; i < n; ++i) diff[i] = evals[i];
    size_t dlen = n;
    for (size_t k = 0; k < n; ++k) {
        const HostFr fact_inv = k < 32 ? inv_fact[k] : HostFr::zero();
        newton[k] = diff[0] * fact_inv;  // k-th forward difference / k!
        for (size_t i = 0; i + 1 < dlen; ++i) diff[i] = diff[i + 1] - diff[i];
        if (dlen) --dlen;
    }
    // expand sum_k newton[k] * x (x-1) ... (x-k+1); basis holds the falling factorial of degree k (k + 1 coefficients)
    basis[0] = HostFr::one();
    size_t blen = 1;
    for (size_t k = 0; k < n; ++k) {
        for (size_t i = 0; i < blen; ++i) out.coefficients[i] = out.coefficients[i] + newton[k] * basis[i];
        if (k + 1 == n) break;
        // basis *= (x - k), in place from the top coefficient down
        const HostFr kk = HostFr::from_u64(k);
        basis[blen] = basis[blen - 1];
        for (size_t i = blen - 1; i > 0; --i) basis[i] = basis[i - 1] - kk * basis[i];
        basis[0] = HostFr::zero() - kk * basis[0];
        ++blen;
    }
    return out;
}

// ---- DeviceProductMember ----------------------------------------------------------------------
size_t DeviceProductMember::num_rounds() const {
    size_t r = 0;
    jb_member_num_rounds(mem_, &r);
    return r;
}

int DeviceProductMember::prove_round(const HostFr* bind, size_t round, const HostFr& previous_claim,
                                     UnivariatePoly* out) {
    size_t degree = 0;
    jb_member_degree(mem_, &degree);
    uint64_t ev[JB_MEMBER_EVALS * 4];
    if (degree + 1 > JB_MEMBER_EVALS) return JB_ERR_UNSUPPORTED;
    int st = jb_member_prove_round(mem_, bind ? bind->l : nullptr, round, check_rounds_ ? previous_claim.l : nullptr, ev);
    if (st != JB_OK) return st;
    evals_.resize(degree + 1);
    for (size_t t = 0; t <= degree; ++t) evals_[t] = HostFr::from_limbs(ev + 4 * t);
    *out = UnivariatePoly::from_evals(evals_);
    return JB_OK;
}

int DeviceProductMember::finish_rounds(const HostFr& bind) { return jb_member_finish_rounds(mem_, bind.l); }

// ---- SequentialRounds (prover.rs:127-148) ----------------------------------------------------------
int SequentialRounds::batch_prove_round(std::vector<MemberRound>& work) {
    for (auto& item : work) {
        int st = item.member->prove_round(item.has_bind ? &item.bind : nullptr, item.local_round, item.claim,
                                          &item.message);
        if (st != JB_OK) return st;
        item.has_message = true;
    }
    return JB_OK;
}

int SequentialRounds::batch_finish_rounds(std::vector<MemberFinish>& finishes) {
    for (auto& f : finishes) {
        int st = f.member->finish_rounds(f.bind);
        if (st != JB_OK) return st;
    }
    return JB_OK;
}

// ---- DeviceRoundScheduler ---------------------------------------------------------------------------
DeviceRoundScheduler::~DeviceRoundScheduler() {
    if (sched_) jb_scheduler_destroy(sched_);
}

int DeviceRoundScheduler::init(jb_ctx* ctx, const std::vector<DeviceProductMember*>& members) {
    members_ = members;
    std::vector<jb_member*> raw;
    for (auto* m : members) raw.push_back(m->device_member());
    return jb_scheduler_create(ctx, raw.data(), raw.size(), &sched_);
}

size_t DeviceRoundScheduler::index_of(const ProveRounds* m) const {
    for (size_t i = 0; i < members_.size(); ++i)
        if (members_[i] == m) return i;
    return members_.size();
}

int DeviceRoundScheduler::batch_prove_round(std::vector<MemberRound>& work) {
    work_.resize(work.size());
    evals_.resize(work.size() * 32);
    for (size_t i = 0; i < work.size(); ++i) {
        const size_t idx = index_of(work[i].member);
        if (idx == members_.size()) return JB_ERR_INVALID;
        jb_round_work& w = work_[i];
        w.member = idx;
        w.round = work[i].local_round;
        w.has_bind = work[i].has_bind ? 1 : 0;
        w.has_claim = members_[idx]->passes_claim() ? 1 : 0;
        std::memcpy(w.bind, work[i].bind.l, 32);
        std::memcpy(w.claim, work[i].claim.l, 32);
    }
    int st = jb_scheduler_prove_round(sched_, work_.data(), work_.size(), evals_.data());
    if (st != JB_OK) return st;
    for (size_t i = 0; i < work.size(); ++i) {
        size_t degree = 0;
        jb_member_degree(members_[work_[i].member]->device_member(), &degree);
        tmp_.resize(degree + 1);
        for (size_t t = 0; t <= degree; ++t) tmp_[t] = HostFr::from_limbs(evals_.data() + i * 32 + 4 * t);
        work[i].message = UnivariatePoly::from_evals(tmp_);
        work[i].has_message = true;
    }
    return JB_OK;
}

int DeviceRoundScheduler::batch_finish_rounds(std::vector<MemberFinish>& finishes) {
    std::vector<jb_finish_work> fw(finishes.size());
    for (size_t i = 0; i < finishes.size(); ++i) {
        const size_t idx = index_of(finishes[i].member);
        if (idx == members_.size()) return JB_ERR_INVALID;
        fw[i].member = idx;
        std::memcpy(fw[i].bind, finishes[i].bind.l, 32);
    }
    return jb_scheduler_finish_rounds(sched_, fw.data(), fw.size());
}

// ---- prove_batch (prover.rs:193-362) -----------------------------------------------------------------
int prove_batch(const BatchPrelude& prelude, std::vector<ProveRounds*>& members, RoundScheduler& scheduler,
                AbsorbRound& recorder, ProvedBatch* out, std::string* err) {
    auto fail = [&](int st, const char* what) {
        if (err) *err = what;
        return st;
    };
    if (members.size() != prelude.members.size()) return fail(JB_ERR_INVALID, "BatchMemberCountMismatch");
    for (size_t i = 0; i < members.size(); ++i) {
        if (members[i]->num_rounds() != prelude.members[i].rounds) return fail(JB_ERR_INVALID, "BatchMemberRoundsMismatch");
        if (prelude.members[i].offset + prelude.members[i].rounds > prelude.max_num_vars)
            return fail(JB_ERR_INVALID, "BatchMemberWindowOutOfRange");
    }
    const size_t max_num_vars = prelude.max_num_vars;
    if (max_num_vars > 0 && prelude.max_degree < 1) return fail(JB_ERR_INVALID, "ZeroBatchDegree");

    static const HostFr two_inv = HostFr::from_u64(2).inverse();
    std::vector<HostFr> member_claims(members.size());
    for (size_t i = 0; i < members.size(); ++i) {
        HostFr c = prelude.members[i].input_claim;  // input_claim * 2^(max - rounds)
        for (size_t k = 0; k < max_num_vars - prelude.members[i].rounds; ++k) c = c + c;
        member_claims[i] = c;
    }
    HostFr running_claim = prelude.claimed_sum;
    out->challenges.clear();
    out->round_polynomials.clear();
    std::vector<HostFr> pending(members.size());
    std::vector<char> has_pending(members.size(), 0);

    std::vector<HostFr> batched;
    std::vector<MemberRound> work;
    work.reserve(members.size());
    out->challenges.reserve(max_num_vars);
    out->round_polynomials.reserve(max_num_vars);
    for (size_t round = 0; round < max_num_vars; ++round) {
        batched.assign(prelude.max_degree + 1, HostFr::zero());
        work.clear();
        for (size_t i = 0; i < members.size(); ++i) {
            const BatchMember& d = prelude.members[i];
            bool active = round >= d.offset && round < d.offset + d.rounds;
            if (!active) {  // the constant polynomial claim/2 (prover.rs:272-280)
                member_claims[i] = member_claims[i] * two_inv;
                batched[0] = batched[0] + d.coefficient * member_claims[i];
                continue;
            }
            MemberRound w;
            w.index = i;
            w.local_round = round - d.offset;
            w.has_bind = has_pending[i];
            w.bind = pending[i];
            has_pending[i] = 0;
            w.claim = member_claims[i];
            w.member = members[i];
            work.push_back(w);
        }
        int st = scheduler.batch_prove_round(work);
        if (st != JB_OK) return fail(st, st == JB_ERR_ROUND_CHECK ? "RoundCheckFailed (member)" : "member prove_round failed");
        for (auto& item : work) {
            if (!item.has_message) return fail(JB_ERR_INVALID, "MissingRoundMessage");
            if (item.message.degree() > prelude.max_degree) return fail(JB_ERR_INVALID, "DegreeBoundExceeded");
            const HostFr& coeff = prelude.members[item.index].coefficient;
            for (size_t k = 0; k < item.message.coefficients.size(); ++k)
                batched[k] = batched[k] + coeff * item.message.coefficients[k];
        }
        while (batched.size() > 2 && batched.back().is_zero()) batched.pop_back();  // trim_round_polynomial
        UnivariatePoly batched_poly;
        batched_poly.coefficients = batched;
        HostFr round_sum = batched_poly.evaluate(HostFr::zero()) + batched_poly.evaluate(HostFr::one());
        if (round_sum != running_claim) return fail(JB_ERR_ROUND_CHECK, "RoundCheckFailed");
        HostFr challenge;
        st = recorder.absorb_round(round, batched_poly, &challenge);
        if (st != JB_OK) return fail(st, "absorb_round failed");
        running_claim = batched_poly.evaluate(challenge);
        out->challenges.push_back(challenge);
        out->round_polynomials.push_back(batched_poly);
        for (auto& item : work) {
            member_claims[item.index] = item.message.evaluate(challenge);
            pending[item.index] = challenge;
            has_pending[item.index] = 1;
        }
    }
    std::vector<MemberFinish> finishes;
    for (size_t i = 0; i < members.size(); ++i)
        if (has_pending[i]) finishes.push_back(MemberFinish{pending[i], members[i]});
    int st = scheduler.batch_finish_rounds(finishes);
    if (st != JB_OK) return fail(st, "finish_rounds failed");
    out->final_claim = running_claim;
    out->member_claims = member_claims;
    return JB_OK;
}

}  // namespace jb

// ---- C entry point over the engine -----------------------------------------------------------------
namespace {
struct CallbackRecorder : jb::AbsorbRound {
    jb_absorb_round_fn fn;
    void* user;
    std::vector<uint64_t> flat;
    int absorb_round(size_t round, const jb::UnivariatePoly& poly, jb::HostFr* challenge) override {
        flat.resize(poly.coefficients.size() * 4);
        for (size_t i = 0; i < poly.coefficients.size(); ++i) poly.coefficients[i].store(flat.data() + 4 * i);
        uint64_t c[4];
        int st = fn(user, round, flat.data(), poly.coefficients.size(), c);
        if (st != 0) return JB_ERR_INVALID;
        if (jb::HostFr::geq_p(c)) return JB_ERR_INVALID;
        *challenge = jb::HostFr::from_limbs(c);
        return JB_OK;
    }
};
}  // namespace

extern "C" {

// Deterministic stand-in for the Fiat-Shamir transcript (which stays on the host and is out of
// scope): a 125-bit challenge [0,0,lo,hi] derived from the round polynomial's
// limbs with SplitMix64. `user` points at a uint64_t seed.
int jb_absorb_round_splitmix125(void* user, size_t round, const uint64_t* coeffs, size_t ncoeffs, uint64_t out[4]) {
    (void)round;  // the challenge depends on the seed and the polynomial only, so a sumcheck that is
    // re-split across engines / GPUs mid-way (jolt_b200/dist.py) derives the same challenges
    uint64_t s = (user ? *(const uint64_t*)user : 0) ^ 0x9E3779B97F4A7C15ULL;
    auto mix = [&](uint64_t v) {
        s += 0x9E3779B97F4A7C15ULL + v;
        uint64_t z = s;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
        return z ^ (z >> 31);
    };
    uint64_t lo = 0, hi = 0;
    for (size_t i = 0; i < ncoeffs * 4; ++i) {
        lo ^= mix(coeffs[i]);
        hi ^= mix(lo);
    }
    out[0] = 0;
    out[1] = 0;
    out[2] = lo;
    out[3] = hi & (~0ULL >> 3);
    return 0;
}

int jb_prove_batch(jb_member** members, const jb_batch_member* desc, size_t n_members, size_t max_num_vars,
                   size_t max_degree, const uint64_t claimed_sum[4], int check_member_rounds,
                   jb_absorb_round_fn absorb, void* user, uint64_t* out_challenges, uint64_t out_final_claim[4],
                   uint64_t* out_member_claims, uint64_t* out_round_polys, size_t* out_round_poly_lens) {
    if (!members || !desc || !claimed_sum || !absorb) return JB_ERR_INVALID;
    jb::BatchPrelude prelude;
    prelude.max_num_vars = max_num_vars;
    prelude.max_degree = max_degree;
    prelude.claimed_sum = jb::HostFr::from_limbs(claimed_sum);
    std::vector<jb::DeviceProductMember> owned;
    owned.reserve(n_members);
    std::vector<jb::ProveRounds*> ptrs;
    for (size_t i = 0; i < n_members; ++i) {
        if (!members[i]) return JB_ERR_INVALID;
        jb::BatchMember bm;
        bm.input_claim = jb::HostFr::from_limbs(desc[i].input_claim);
        bm.coefficient = jb::HostFr::from_limbs(desc[i].coefficient);
        bm.rounds = desc[i].rounds;
        bm.offset = desc[i].offset;
        prelude.members.push_back(bm);
        owned.emplace_back(members[i], check_member_rounds != 0);
    }
    for (auto& m : owned) ptrs.push_back(&m);
    // the device traversal: one host round trip per batch round; the reference's declaration-order traversal if
    // the device scheduler cannot be set up
    jb::SequentialRounds seq_sched;
    jb::DeviceRoundScheduler dev_sched;
    jb::RoundScheduler* sched_ptr = &seq_sched;
    if (n_members > 0) {
        std::vector<jb::DeviceProductMember*> dm;
        for (auto& m : owned) dm.push_back(&m);
        jb_ctx* ctx = jb_member_context(members[0]);
        if (ctx && dev_sched.init(ctx, dm) == JB_OK) sched_ptr = &dev_sched;
    }
    jb::RoundScheduler& sched = *sched_ptr;
    CallbackRecorder rec;
    rec.fn = absorb;
    rec.user = user;
    jb::ProvedBatch proved;
    std::string err;
    int st = jb::prove_batch(prelude, ptrs, sched, rec, &proved, &err);
    if (st != JB_OK) return st;
    for (size_t r = 0; r < proved.challenges.size(); ++r) {
        if (out_challenges) proved.challenges[r].store(out_challenges + 4 * r);
        if (out_round_polys) {
            std::memset(out_round_polys + r * (max_degree + 1) * 4, 0, (max_degree + 1) * 32);
            for (size_t k = 0; k < proved.round_polynomials[r].coefficients.size(); ++k)
                proved.round_polynomials[r].coefficients[k].store(out_round_polys + (r * (max_degree + 1) + k) * 4);
        }
        if (out_round_poly_lens) out_round_poly_lens[r] = proved.round_polynomials[r].coefficients.size();
    }
    if (out_final_claim) proved.final_claim.store(out_final_claim);
    if (out_member_claims)
        for (size_t i = 0; i < n_members; ++i) proved.member_claims[i].store(out_member_claims + 4 * i);
    return JB_OK;
}

}  // extern "C"
