// C++ mirror of the reference's sumcheck seam (see sumcheck_host.cu for citations).
#pragma once
#include <cstddef>
#include <string>
#include <vector>

#include "../../include/jolt_b200.h"
#include "host_fr.hpp"

namespace jb {

// evaluations of one member's round: degree + 1 <= 10 (a split-eq member of 8 tables has degree 9)
constexpr int JB_MEMBER_EVALS = 10;

// jolt_poly::UnivariatePoly (crates/jolt-poly/src/univariate.rs:27-29): ascending coefficients.
struct UnivariatePoly {
    std::vector<HostFr> coefficients;
    size_t degree() const { return coefficients.empty() ? 0 : coefficients.size() - 1; }
    HostFr evaluate(const HostFr& x) const;
    static UnivariatePoly from_evals(const std::vector<HostFr>& evals);
};

// jolt_sumcheck::ProveRounds (crates/jolt-sumcheck/src/prover.rs:52-72). Status codes stand in
// for Result<_, SumcheckError>.
struct ProveRounds {
    virtual ~ProveRounds() = default;
    virtual size_t num_rounds() const = 0;
    virtual int prove_round(const HostFr* bind, size_t round, const HostFr& previous_claim, UnivariatePoly* out) = 0;
    virtual int finish_rounds(const HostFr& bind) = 0;
};

// The device-backed member: product of m dense tables (jb_member).
class DeviceProductMember : public ProveRounds {
   public:
    DeviceProductMember(jb_member* mem, bool check_rounds) : mem_(mem), check_rounds_(check_rounds) {}
    size_t num_rounds() const override;
    int prove_round(const HostFr* bind, size_t round, const HostFr& previous_claim, UnivariatePoly* out) override;
    int finish_rounds(const HostFr& bind) override;

    jb_member* device_member() const { return mem_; }
    bool passes_claim() const { return check_rounds_; }

   private:
    jb_member* mem_;
    bool check_rounds_;
    std::vector<HostFr> evals_;  // reused across rounds (no allocation on the round trip)
};

// MemberRound / MemberFinish (prover.rs:75-104)
struct MemberRound {
    size_t index = 0;
    size_t local_round = 0;
    bool has_bind = false;
    HostFr bind{};
    HostFr claim{};
    ProveRounds* member = nullptr;
    bool has_message = false;
    UnivariatePoly message;
};
struct MemberFinish {
    HostFr bind;
    ProveRounds* member;
};

// RoundScheduler (prover.rs:110-120): order and transport are free.
struct RoundScheduler {
    virtual ~RoundScheduler() = default;
    virtual int batch_prove_round(std::vector<MemberRound>& work) = 0;
    virtual int batch_finish_rounds(std::vector<MemberFinish>& finishes) = 0;
};
struct SequentialRounds : RoundScheduler {
    int batch_prove_round(std::vector<MemberRound>& work) override;
    int batch_finish_rounds(std::vector<MemberFinish>& finishes) override;
};

// The device traversal (BuildRoundScheduler, crates/jolt-kernels/src/backend.rs:64-70): every active member's
// round in ONE host round trip through jb_scheduler_* (a resident kernel for homogeneous batches, overlapped
// launches otherwise). Members must be DeviceProductMember over one context.
class DeviceRoundScheduler : public RoundScheduler {
   public:
    DeviceRoundScheduler() = default;
    ~DeviceRoundScheduler() override;
    int init(jb_ctx* ctx, const std::vector<DeviceProductMember*>& members);
    int batch_prove_round(std::vector<MemberRound>& work) override;
    int batch_finish_rounds(std::vector<MemberFinish>& finishes) override;

   private:
    jb_scheduler* sched_ = nullptr;
    std::vector<DeviceProductMember*> members_;
    std::vector<jb_round_work> work_;     // reused across rounds
    std::vector<uint64_t> evals_;
    std::vector<HostFr> tmp_;
    size_t index_of(const ProveRounds* m) const;
};

// BatchMember / BatchPrelude (crates/jolt-sumcheck/src/batch.rs:24-71)
struct BatchMember {
    HostFr input_claim;
    HostFr coefficient;
    size_t rounds;
    size_t offset;
};
struct BatchPrelude {
    std::vector<BatchMember> members;
    size_t max_num_vars = 0;
    size_t max_degree = 0;
    HostFr claimed_sum{};
};

// SumcheckRecorder::absorb_round + transcript squeeze (recorder.rs:118-130): host-owned.
struct AbsorbRound {
    virtual ~AbsorbRound() = default;
    virtual int absorb_round(size_t round, const UnivariatePoly& poly, HostFr* challenge) = 0;
};

// ProvedBatch (prover.rs:153-157) + the batched round polynomials the recorder saw.
struct ProvedBatch {
    std::vector<HostFr> challenges;
    HostFr final_claim{};
    std::vector<HostFr> member_claims;
    std::vector<UnivariatePoly> round_polynomials;
};

int prove_batch(const BatchPrelude& prelude, std::vector<ProveRounds*>& members, RoundScheduler& scheduler,
                AbsorbRound& recorder, ProvedBatch* out, std::string* err);

}  // namespace jb
