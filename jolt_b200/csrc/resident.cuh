// Resident sumcheck kernel: ONE launch serves every round of a batch of members.
//
// A sumcheck has log N sequential Fiat-Shamir round trips (the challenge of round k depends on the round
// polynomial of round k; the transcript is host-owned, specs/clean-slate-prover.md:579-584). With one launch per
// round each trip costs launch + ramp + drain + publish (~19 us on top of the pass itself, r01 BENCH) - at 2^22
// that was 65 % of the whole sumcheck. Here the kernel is launched once per batch (cooperatively: every block is
// co-resident), and every round is driven through a mailbox in host-mapped pinned memory:
//
//   host : writes {actions, challenge} then cmd_seq            (one 64-byte line)
//   blk 0: warp 0 polls that line over PCIe (one coalesced 64 B read per poll), then re-publishes it in DEVICE
//          memory (ResState) with a release store; the other blocks spin on that word with acquire loads (L2)
//   all  : run their share of the fused bind + sweep pass of every active member (the same fused_pass body as
//          the one-launch-per-round kernel) and add the block's UNREDUCED column sums - K values x 17 u64 lanes of
//          32-bit limb sums - into the round's lane accumulators with integer REDs (exact, order-free), then arrive
//          on a ticket counter
//   last : the last block to arrive copies the lanes to the mailbox (and zeroes them), resets the ticket and raises
//          res_seq, which the host spins on. The O(K) serial tail - carry propagation and the Montgomery reduction
//          of each 544-bit sum - runs on the HOST (jb_wide_lanes_reduce_host): one CPU core does it in ~0.2 us,
//          one GPU lane needs ~2 us, and it sits on the latency path of every round.
//
// The bind -> next round's reads dependency between DIFFERENT blocks is carried by that same chain
// (stores -> bar.sync -> fence -> ticket atomic ... res_seq -> host -> cmd_seq -> release/acquire -> bar.sync ->
// loads): it is the grid barrier of cooperative groups with the host's Fiat-Shamir step in the middle. Tables
// are therefore read with coherent loads here (fused_pass<.., NC = false>), never through the read-only path.
//
// Blocks that can have no work in any later round (the tables only shrink) exit; the ticket target of a round is
// the number of live blocks, which every block derives from the same state. With one live block the kernel
// degenerates into the r01 "persistent tail": no broadcast, no ticket.
//
// Multi-GPU: for index-sharded rounds the last block also performs the all-reduce of the round sums over NVLink
// peer memory (CUDA-IPC mapped exchange buffers): one warp stores this rank's lanes into every peer's slot,
// raises a flag per peer, waits for the peers' flags in its own buffer and sums - before the totals go to the
// host. No NCCL launch, no extra kernel (comm.cu owns the buffers).
#pragma once
#include "poly_kernels.cuh"

namespace jb {

constexpr int RES_MAX_MEMBERS = 8;
constexpr int RES_BLOCK = 256;
constexpr size_t RES_SMALL_LEN = 8192;  // tables this short need few blocks: such runs coexist with other work
// big passes: this share (%) of the pair range is laid out statically, the rest is claimed warp by warp (ResArgs::static_pct;
// passed as an argument rather than folded in, which keeps the kernel's register allocation as measured)
constexpr int RES_STATIC_PCT = 75;
// Degree-2 rounds with at most this many pair indices run as THIN passes (thin_pass below): latency-shaped, and
// they also return the lookahead sums that let the host answer the NEXT round without waiting for the device.
constexpr uint64_t RES_THIN_PAIRS = 1ull << 17;  // (2^17: the first thin round costs what the generic pass costs there, and one more round is pipelined)
// mailbox / accumulator words per member: a thin round returns 8 sums x 17 lanes; a generic round K <= 4 values
// x 17 lanes (products) or x 8 lanes (D = 1); a terminal bind the T final values x 4 limbs
constexpr int RES_SLOT_U64 = 136;

// per-member action of a round command (4 bits each, member i at bits [16 + 4i, 20 + 4i) of cmd)
enum : unsigned { RES_ACT_NONE = 0, RES_ACT_EVAL = 1, RES_ACT_BIND_EVAL = 2, RES_ACT_FINAL = 3 };
enum : uint64_t { RES_OP_ROUND = 1, RES_OP_ABORT = 2 };
constexpr uint64_t RES_FLAG_EXCHANGE = 1ull << 8;  // member 0's sums are all-reduced over peer memory
// member 0 (index-sharded): bind, then write the bound shard into EVERY rank's gather arena, wait for the peers'
// shards, and sweep the GATHERED tables (G x the shard) - the member continues un-sharded, in the same kernel
constexpr uint64_t RES_FLAG_GATHER = 1ull << 9;

// The mailbox is a ring of TWO commands / answers (command s uses slot s & 1): with lookahead the host posts
// command s + 1 while the answer to command s is still on its way.
struct alignas(64) ResCmdLine {
    // 64 B, host -> device. The host writes the payload first and cmd_seq last; the device reads the whole line
    // with ONE coalesced 64-byte request, so a snapshot that shows the new sequence number also shows its payload.
    volatile uint64_t cmd_seq;
    uint64_t cmd;           // RES_OP_* | flags | actions << 16
    uint64_t challenge[4];  // Montgomery limbs of the bind scalar (shared by every member of the batch round)
    uint64_t xseq;          // exchange sequence number (RES_FLAG_EXCHANGE)
    uint64_t pad0;
};
struct alignas(64) ResAnswerLine {
    volatile uint64_t res_seq;
    uint64_t status;  // 0 ok, 1 aborted / timed out, 2 exchange timed out
    uint64_t pad1[6];
};
struct alignas(64) ResMailbox {
    ResCmdLine cmd[2];
    ResAnswerLine ans[2];
    // per answer, per member: the round's sums as lanes (32-bit limb column sums, see resident_pass / thin_pass),
    // or - after a terminal bind that left the member fully bound - its T final values (4 limbs each)
    uint64_t result[2][RES_MAX_MEMBERS * RES_SLOT_U64];
    // observability (specs/clean-slate-prover.md:585-587): %globaltimer (ns) when block 0 decoded command s and
    // when the last block had collected the round's sums, at [2 (s - 1 mod 64)] and [.. + 1]
    uint64_t tlog[2 * 64];
    // finer stamps of the same rounds (diagnostics): [4 s + 0] block 0 finished its passes, [4 s + 1] block 0 arrived
    // on the ticket, [4 s + 2] the last block saw that it is last, [4 s + 3] spare
    uint64_t tlog2[4 * 64];
};

// Device-side re-publication of the command line, the arrival counter and the round's lane accumulators.
struct alignas(128) ResState {
    uint64_t seq;
    uint64_t cmd[7];
    uint64_t pad[8];
    unsigned int ticket;
    unsigned int pad2[31];
    // sequence number of the last round whose sums have been collected (lanes zeroed, ticket reset). With two
    // commands in flight block 0 may SEE command s + 1 before round s is complete: it re-publishes it only after
    // done == s, so no block can miss (or tear) a command and no RED of round s + 1 lands in round s's lanes.
    uint64_t done;
    uint64_t bar_epoch;          // in-command grid barrier (gather): arrivals in bar_count, release by epoch
    unsigned int bar_count;
    unsigned int pad3a;
    uint64_t pad3[13];
    uint64_t lanes[RES_MAX_MEMBERS * RES_SLOT_U64];  // zero between rounds
    // dynamic-tail claim counters of the big passes, one 128-byte line per member; zero between rounds
    unsigned int work[RES_MAX_MEMBERS * 32];
};

struct ResMemberArg {
    uint64_t* buf[JB_MAX_TABLES];
    uint64_t* alt[JB_MAX_TABLES];  // LowToHigh ping-pong partner (>= len/2 entries); unused under HighToLow
    uint64_t len;
};

struct ResArgs {
    ResMemberArg mem[RES_MAX_MEMBERS];
    int n_members;
    ResMailbox* mb;     // host-mapped
    ResState* st;       // device
    long long timeout_cycles;
    int static_pct;     // big passes: this share of the pair range is laid out statically, the rest is claimed (100 = off)
    // peer exchange (world > 1): exchange buffer of every rank as mapped in THIS process
    uint64_t* peer[16];
    int world, rank;
};

__device__ __forceinline__ uint64_t ld_acquire_gpu(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(uint64_t* p, uint64_t v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t global_timer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// How `items` independent work items (pair indices / bind outputs) are laid over at most `cap` blocks.
// Large rounds fill every block (256 threads, grid-stride). Once there is less than one item per thread the
// pass is pure latency - a warp's chain of dependent IMAD.WIDEs - so the items are spread THIN: two warps per
// block over as many SMs as are alive rather than eight warps contending for one SM's multiplier; up to 256
// items stay in a single block (no broadcast, no ticket).
struct ResShape {
    unsigned nblk, tpb;
};
__host__ __device__ inline ResShape res_shape(uint64_t items, unsigned cap) {
    ResShape s;
    if (items <= (uint64_t)RES_BLOCK || cap <= 1) {
        s.nblk = 1;
        const uint64_t t = items < (uint64_t)RES_BLOCK ? ((items + 31) / 32) * 32 : RES_BLOCK;
        s.tpb = t < 32 ? 32u : (unsigned)t;
        return s;
    }
    const uint64_t want = (items + 63) / 64;
    s.nblk = (unsigned)(want < cap ? want : cap);
    const uint64_t per = (items + s.nblk - 1) / s.nblk;
    const uint64_t t = ((per + 31) / 32) * 32;
    s.tpb = t > (uint64_t)RES_BLOCK ? (unsigned)RES_BLOCK : (unsigned)t;
    return s;
}
__host__ __device__ inline unsigned res_blocks_for(uint64_t items, unsigned cap) { return res_shape(items, cap).nblk; }

// One member's pass as an out-of-line call: the pass body gets the whole register budget to itself (the round
// loop's own state is saved around ONE call per round instead of squeezing the inner loop into spills).
// The block's sums leave as lanes (K x 17 column sums for products, K x 8 limbs for D = 1): added into the round's
// accumulators at `g_lanes` with integer REDs, or - when this block is the only live one - left straight in
// shared memory at `s_dst`: no trip through L2 on the latency path.
template <int D, int P, int ORDER, bool BIND, bool HI4>
__device__ __noinline__ void resident_pass(const TablePtrs tp, size_t pairs, const BindScalar sc, uint32_t* dsm, size_t first,
                                           size_t stride, uint64_t* g_lanes, uint64_t* s_dst) {
    constexpr int K = D;
    Fr acc[K];
    fused_pass<D, P, ORDER, BIND, HI4, true, RES_BLOCK, false, false, (D > 1), true>(tp, pairs, sc, dsm, first, stride, acc);
    const int tid = threadIdx.x;
    if (D > 1) {
        const uint64_t* colsum = reinterpret_cast<const uint64_t*>(dsm + FusedShape<D, true>::acc_words(RES_BLOCK));
        if (tid < K * 17) {
            const uint64_t v = colsum[tid];
            if (s_dst) s_dst[tid] = v;
            else atomicAdd(reinterpret_cast<unsigned long long*>(g_lanes) + tid, (unsigned long long)v);
        }
    } else if (tid == 0) {
#pragma unroll
        for (int e = 0; e < K; ++e)
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                if (s_dst) s_dst[e * 8 + w] = acc[e].v[w];
                else atomicAdd(reinterpret_cast<unsigned long long*>(g_lanes) + e * 8 + w, (unsigned long long)acc[e].v[w]);
            }
    }
}

// ---- thin pass (degree 2): short rounds are pure latency, and they come with lookahead ------------------------
// T' = the tables of this round (after the pending bind, if any), n' entries each. The next bind will pair T'
// entries again, so T' is walked in QUADS: (a, b) is the pair that the next challenge r folds into the next round's
// lo, (c, d) the pair it folds into hi:   lo(r) = a + r (b - a),   hi(r) = c + r (d - c).
//   LowToHigh : a, b, c, d = T'[4q .. 4q + 3]
//   HighToLow : a = T'[q], b = T'[q + n'/2], c = T'[q + n'/4], d = T'[q + 3n'/4]
// For every quad q and term k, EIGHT lanes - one per warp of the block, lane g of warp p serves group g - each
// produce ONE of the 8 bound values (table j = p / 4, position p % 4: one load pair + one bind product), exchange
// them through shared memory, and each accumulate ONE product of the pair (x, x') = (table 0, table 1):
//   S0 = a a'          S1 = b b'           S2 = (b - a)(b' - a')
//   S3 = (c - a)(..)'  S4 = (d - b)(..)'   S5 = (d - c - b + a)(..)'     S6 = c c'      S7 = (d - c)(d' - c')
// so the longest dependent chain of a round is one bind and one product instead of four binds and two products.
// This round's polynomial is  s(0) = S0 + S6,  s(inf) = S2 + S7.  And the NEXT round's polynomial, as a function
// of the not yet known challenge r, is determined by S0..S5:
//   s_next(0)(r)   = sum lo lo'  = S0 + r (S1 - S0 - S2) + r^2 S2
//   s_next(inf)(r) = sum (hi - lo)(hi' - lo') = S3 + r (S4 - S3 - S5) + r^2 S5
// - the host evaluates these the moment it has drawn r, posts r, and does NOT wait for the device: the device's
// bind + sums for round k + 1 overlap the host's Fiat-Shamir step of round k (the answers trail one command behind).
// Each warp's 17-word accumulator stays in registers and is summed over the warp with two REDUX per word.
// n' == 2 (the last round): a and b only; c = d = 0, S6 = S7 = 0.
template <int P, int ORDER, bool BIND>
__device__ __noinline__ void thin_pass(const TablePtrs tp, uint64_t nprime, const BindScalar sc, bool hi4, uint32_t* dsm,
                                       unsigned b, unsigned nblk, uint64_t* g_lanes, uint64_t* s_dst) {
    const int tid = threadIdx.x, g = tid & 31, p = tid >> 5;
    uint32_t* sval = dsm;  // [8 values][8 words][32 groups]
    const uint64_t quads = nprime >= 4 ? nprime / 4 : 1;
    const uint64_t ngroups = quads * P;
    const int j = p >> 2, pos = p & 3;
    uint32_t A[17];
#pragma unroll
    for (int w = 0; w < 17; ++w) A[w] = 0;
    for (uint64_t base = (uint64_t)b * 32; base < ngroups; base += (uint64_t)nblk * 32) {
        const uint64_t grp = base + g;
        const bool valid = grp < ngroups;
        const uint64_t q = P == 1 ? grp : grp / P;
        const int k = P == 1 ? 0 : (int)(grp % P);
        Fr v = Fr::zero();
        if (valid && (nprime >= 4 || pos < 2)) {
            const int t = k * 2 + j;
            uint64_t ip;
            if (nprime < 4) ip = (uint64_t)pos;
            else if (ORDER == ORDER_LOW_TO_HIGH) ip = 4 * q + pos;
            else ip = q + (uint64_t)(pos & 1) * (nprime / 2) + (uint64_t)(pos >> 1) * (nprime / 4);
            if (BIND) {
                const uint64_t* in = tp.in[t];
                const Fr lo = ld_elem_rw<Fr>(in, ORDER == ORDER_LOW_TO_HIGH ? 2 * ip : ip);
                const Fr hi = ld_elem_rw<Fr>(in, ORDER == ORDER_LOW_TO_HIGH ? 2 * ip + 1 : ip + nprime);
                v = hi4 ? bind_pair<true>(lo, hi, sc) : bind_pair<false>(lo, hi, sc);
                st_elem(tp.out[t], ip, v);
            } else {
                v = ld_elem_rw<Fr>(tp.in[t], ip);
            }
        }
#pragma unroll
        for (int w = 0; w < 8; ++w) sval[(p * 8 + w) * 32 + g] = v.v[w];
        __syncthreads();
        if (valid) {
            Fr x[2];
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
                const uint32_t* sv = sval + jj * 4 * 8 * 32 + g;
                auto rd = [&](int ps) {
                    Fr r;
#pragma unroll
                    for (int w = 0; w < 8; ++w) r.v[w] = sv[(ps * 8 + w) * 32];
                    return r;
                };
                switch (p) {  // warp-uniform
                    case 0: x[jj] = rd(0); break;
                    case 1: x[jj] = rd(1); break;
                    case 2: x[jj] = fp_sub_lazy(rd(1), rd(0)); break;
                    case 3: x[jj] = fp_sub_lazy(rd(2), rd(0)); break;
                    case 4: x[jj] = fp_sub_lazy(rd(3), rd(1)); break;
                    case 5: x[jj] = fp_sub_lazy(fp_sub(rd(3), rd(2)), fp_sub(rd(1), rd(0))); break;
                    case 6: x[jj] = rd(2); break;
                    default: x[jj] = fp_sub_lazy(rd(3), rd(2)); break;
                }
            }
            mul_wide_acc_reg(A, x[0].v, x[1].v);
        }
        __syncthreads();
    }
    // warp p holds product p: sum each accumulator word over the 32 lanes (16-bit halves: no overflow in REDUX)
    uint64_t mine = 0;
#pragma unroll
    for (int w = 0; w < 17; ++w) {
        const uint32_t lo = __reduce_add_sync(0xffffffffu, A[w] & 0xffffu);
        const uint32_t hi = __reduce_add_sync(0xffffffffu, A[w] >> 16);
        if (g == w) mine = (uint64_t)lo + ((uint64_t)hi << 16);
    }
    if (g < 17) {
        if (s_dst) s_dst[p * 17 + g] = mine;
        else atomicAdd(reinterpret_cast<unsigned long long*>(g_lanes) + p * 17 + g, (unsigned long long)mine);
    }
}

// lanes a member's round leaves in the accumulators / mailbox
template <int D>
__host__ __device__ constexpr int res_lanes(bool thin) {
    return thin ? 8 * 17 : (D == 1 ? 8 : D * 17);
}
__host__ __device__ inline bool res_is_thin(int D, uint64_t nprime) { return D == 2 && nprime / 2 <= RES_THIN_PAIRS; }
// blocks a thin pass over n' entries (P terms) uses out of `cap`
__host__ __device__ inline unsigned res_thin_blocks(uint64_t nprime, int P, unsigned cap) {
    const uint64_t ngroups = (nprime >= 4 ? nprime / 4 : 1) * (uint64_t)P;
    if (ngroups <= 64 || cap <= 1) return 1;
    const uint64_t want = (ngroups + 31) / 32;
    return (unsigned)(want < cap ? want : cap);
}
// blocks the largest pass a member with `len` entries can still ask for needs (an eval over len entries if it has
// not started, else a bind + eval over len / 2, or a terminal bind over len / 2 outputs)
__host__ __device__ inline unsigned res_need_blocks(int D, int P, uint64_t len, unsigned cap) {
    if (len < 2) return 0;
    unsigned need = res_is_thin(D, len) ? res_thin_blocks(len, P, cap) : res_blocks_for(len / 2, cap);
    const unsigned fin = res_blocks_for(len / 2, cap);
    return need > fin ? need : fin;
}

template <int D, int P, int ORDER>
__global__ void __launch_bounds__(RES_BLOCK, 2) resident_rounds_kernel(const __grid_constant__ ResArgs a) {
    constexpr int T = D * P;
    constexpr int K = D;  // s(1) always comes from the running claim (the optimized tier's convention)
    extern __shared__ uint32_t dsm[];
    __shared__ uint64_t s_line[8];
    __shared__ uint64_t* s_cur[RES_MAX_MEMBERS][T];
    __shared__ uint64_t* s_oth[RES_MAX_MEMBERS][T];
    __shared__ uint64_t s_len[RES_MAX_MEMBERS];
    __shared__ int s_kl[RES_MAX_MEMBERS];  // lanes each member produced this round
    __shared__ unsigned s_live_next;
    __shared__ int s_last;
    __shared__ uint64_t s_lanes[RES_MAX_MEMBERS * RES_SLOT_U64];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned b = blockIdx.x, grid = gridDim.x;
    const int NM = a.n_members;
    if (tid < NM) {
        s_len[tid] = a.mem[tid].len;
#pragma unroll
        for (int j = 0; j < T; ++j) {
            s_cur[tid][j] = a.mem[tid].buf[j];
            s_oth[tid][j] = a.mem[tid].alt[j];
        }
    }
    __syncthreads();
    unsigned live = grid;
    uint64_t seq = 0;
    while (true) {
        // ---- receive command seq + 1 ------------------------------------------------------------------
        if (b == 0) {
            if (tid < 32) {
                const long long t0 = clock64();
                const volatile uint64_t* line = reinterpret_cast<const volatile uint64_t*>(&a.mb->cmd[(seq + 1) & 1]);
                uint64_t v = 0;
                bool got = false;
                while (true) {
                    if (lane < 8) v = line[lane];
                    const uint64_t sq = __shfl_sync(0xffffffffu, v, 0);
                    if (sq == seq + 1) {
                        got = true;
                        break;
                    }
                    const int expired = __shfl_sync(0xffffffffu, (int)(clock64() - t0 > a.timeout_cycles), 0);
                    if (expired) break;  // host went away: give the SMs back
                    __nanosleep(20);
                }
                if (!got && lane == 1) v = RES_OP_ABORT;
                if (lane < 8) s_line[lane] = v;
                if (live > 1) {  // re-publish for the other blocks: payload, then the sequence number (release)
                    uint64_t w[7];
#pragma unroll
                    for (int k = 0; k < 7; ++k) w[k] = __shfl_sync(0xffffffffu, v, k + 1);
                    if (lane == 0) {
                        const long long t1 = clock64();
                        while (ld_acquire_gpu(&a.st->done) != seq)  // the previous round is complete
                            if (clock64() - t1 > a.timeout_cycles) break;
#pragma unroll
                        for (int k = 0; k < 7; ++k) a.st->cmd[k] = w[k];
                        st_release_gpu(&a.st->seq, seq + 1);
                    }
                }
            }
        } else if (tid == 0) {
            const long long t0 = clock64();
            bool got = true;
            while (ld_acquire_gpu(&a.st->seq) != seq + 1) {
                if (clock64() - t0 > a.timeout_cycles) {
                    got = false;
                    break;
                }
            }
            if (got) {
#pragma unroll
                for (int k = 0; k < 7; ++k) s_line[k + 1] = a.st->cmd[k];
            } else {
                s_line[1] = RES_OP_ABORT;
            }
        }
        __syncthreads();
        ++seq;
        const uint64_t cmdw = s_line[1];
        const uint64_t xseq = s_line[6];
        if ((cmdw & 0xff) != RES_OP_ROUND) {
            if (b == 0 && tid == 0) {
                a.mb->ans[seq & 1].status = 1;
                __threadfence_system();
                a.mb->ans[seq & 1].res_seq = seq;
            }
            return;
        }
        if (b == 0 && tid == 0) a.mb->tlog[2 * ((seq - 1) & 63)] = global_timer_ns();
        const unsigned actions = (unsigned)(cmdw >> 16);
        BindScalar sc;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            sc.w[2 * i] = (uint32_t)s_line[2 + i];
            sc.w[2 * i + 1] = (uint32_t)(s_line[2 + i] >> 32);
        }
        const bool hi4 = (s_line[2] | s_line[3]) == 0;  // 125-bit challenge [0,0,lo,hi]: 4-row product

        unsigned eff_actions = actions;  // what the member loop below executes (a gather turns its bind into an eval)
        if (cmdw & RES_FLAG_GATHER) {
            // ---- bind member 0's shard and scatter it into every rank's arena --------------------------------
            const int G = a.world, par = (int)(xseq & 1);
            const uint64_t len = s_len[0], np = len / 2;      // np = this rank's bound shard
            const uint64_t glen = np * (uint64_t)G;           // the gathered table
            const ResShape sh = res_shape(np, live);
            if (b < sh.nblk && tid < (int)sh.tpb) {
                for (uint64_t i = (uint64_t)b * sh.tpb + tid; i < np; i += (uint64_t)sh.nblk * sh.tpb) {
                    // LowToHigh shards are contiguous blocks of the global table, HighToLow shards are strided
                    const uint64_t gpos = ORDER == ORDER_LOW_TO_HIGH ? (uint64_t)a.rank * np + i : i * (uint64_t)G + a.rank;
#pragma unroll
                    for (int j = 0; j < T; ++j) {
                        const uint64_t* in = s_cur[0][j];
                        const Fr lo = ld_elem_rw<Fr>(in, ORDER == ORDER_HIGH_TO_LOW ? i : 2 * i);
                        const Fr hi = ld_elem_rw<Fr>(in, ORDER == ORDER_HIGH_TO_LOW ? i + np : 2 * i + 1);
                        const Fr o = hi4 ? bind_pair<true>(lo, hi, sc) : bind_pair<false>(lo, hi, sc);
                        for (int g = 0; g < G; ++g)
                            st_elem(a.peer[g] + (XCH_ARENA_OFFSET + (size_t)par * XCH_ARENA_HALF) / 8 + (size_t)j * glen * 4, gpos, o);
                    }
                }
            }
            // ---- grid barrier; its last arriver also waits for every peer's shard ------------------------------
            __syncthreads();
            if (tid == 0) {
                bool ok = true;
                if (live > 1) {
                    __threadfence_system();
                    const uint64_t epoch = ld_acquire_gpu(&a.st->bar_epoch);
                    if (atomicAdd(&a.st->bar_count, 1u) == live - 1) {
                        a.st->bar_count = 0;
                        __threadfence_system();  // every block's peer stores (ordered before its arrival) before the flags
                        for (int g = 0; g < G; ++g) *(volatile uint64_t*)(a.peer[g] + XCH_GFLAG_BASE + par * 16 + a.rank) = xseq;
                        const long long t0 = clock64();
                        uint64_t* mine = a.peer[a.rank];
                        for (int src = 0; src < G && ok; ++src)
                            while (*(volatile uint64_t*)(mine + XCH_GFLAG_BASE + par * 16 + src) != xseq)
                                if (clock64() - t0 > a.timeout_cycles) {
                                    ok = false;
                                    break;
                                }
                        __threadfence_system();
                        st_release_gpu(&a.st->bar_epoch, epoch + 1 + (ok ? 0 : (1ull << 32)));
                    } else {
                        const long long t0 = clock64();
                        while ((uint32_t)ld_acquire_gpu(&a.st->bar_epoch) == (uint32_t)epoch)
                            if (clock64() - t0 > a.timeout_cycles) break;
                    }
                } else {
                    __threadfence_system();
                    for (int g = 0; g < G; ++g) *(volatile uint64_t*)(a.peer[g] + XCH_GFLAG_BASE + par * 16 + a.rank) = xseq;
                    const long long t0 = clock64();
                    uint64_t* mine = a.peer[a.rank];
                    for (int src = 0; src < G && ok; ++src)
                        while (*(volatile uint64_t*)(mine + XCH_GFLAG_BASE + par * 16 + src) != xseq)
                            if (clock64() - t0 > a.timeout_cycles) {
                                ok = false;
                                break;
                            }
                    __threadfence_system();
                }
                // the member continues on the gathered tables (and their ping-pong partners) in THIS rank's arena
                uint64_t* arena = a.peer[a.rank] + (XCH_ARENA_OFFSET + (size_t)par * XCH_ARENA_HALF) / 8;
                for (int j = 0; j < T; ++j) {
                    s_cur[0][j] = arena + (size_t)j * glen * 4;
                    s_oth[0][j] = arena + (size_t)T * glen * 4 + (size_t)j * (glen / 2) * 4;
                }
                s_len[0] = glen;
            }
            __syncthreads();
            eff_actions = (actions & ~0xfu) | RES_ACT_EVAL;
        }
        // ---- this block's share of every active member's pass -------------------------------------------
        for (int m = 0; m < NM; ++m) {
            const unsigned act = (eff_actions >> (4 * m)) & 0xf;
            if (act == RES_ACT_NONE) continue;
            const uint64_t len = s_len[m];
            if (act == RES_ACT_FINAL) {  // terminal bind: no sweep
                const uint64_t half = len / 2;
                const ResShape sh = res_shape(half, live);
                if (b < sh.nblk && tid < (int)sh.tpb) {
                    for (uint64_t i = (uint64_t)b * sh.tpb + tid; i < half; i += (uint64_t)sh.nblk * sh.tpb) {
#pragma unroll
                        for (int j = 0; j < T; ++j) {
                            const uint64_t* in = s_cur[m][j];
                            const Fr lo = ld_elem_rw<Fr>(in, ORDER == ORDER_HIGH_TO_LOW ? i : 2 * i);
                            const Fr hi = ld_elem_rw<Fr>(in, ORDER == ORDER_HIGH_TO_LOW ? i + half : 2 * i + 1);
                            const Fr o = hi4 ? bind_pair<true>(lo, hi, sc) : bind_pair<false>(lo, hi, sc);
                            st_elem(ORDER == ORDER_HIGH_TO_LOW ? s_cur[m][j] : s_oth[m][j], i, o);
                        }
                    }
                }
                continue;
            }
            const bool bind = act == RES_ACT_BIND_EVAL;
            const uint64_t nprime = bind ? len / 2 : len;
            const uint64_t pairs = nprime / 2;
            const bool thin = res_is_thin(D, nprime);
            if (tid == 0) s_kl[m] = res_lanes<D>(thin);
            if constexpr (D == 2) if (thin) {
                const unsigned nb = res_thin_blocks(nprime, P, live);
                if (b < nb) {
                    TablePtrs tp;
#pragma unroll
                    for (int j = 0; j < T; ++j) {
                        tp.in[j] = s_cur[m][j];
                        tp.out[j] = (ORDER == ORDER_LOW_TO_HIGH && bind) ? s_oth[m][j] : s_cur[m][j];
                    }
                    tp.e_out = tp.e_in = nullptr;
                    tp.in_bits = 0;
                    tp.work = nullptr;
                    tp.static_end = ~(size_t)0;
                    uint64_t* gl = a.st->lanes + m * RES_SLOT_U64;
                    uint64_t* sl = live == 1 ? s_lanes + m * RES_SLOT_U64 : nullptr;
                    if (bind) thin_pass<P, ORDER, true>(tp, nprime, sc, hi4, dsm, b, nb, gl, sl);
                    else thin_pass<P, ORDER, false>(tp, nprime, sc, hi4, dsm, b, nb, gl, sl);
                }
                continue;
            }
            const ResShape sh = res_shape(pairs, live);
            if (b < sh.nblk) {
                TablePtrs tp;
#pragma unroll
                for (int j = 0; j < T; ++j) {
                    tp.in[j] = s_cur[m][j];
                    tp.out[j] = (ORDER == ORDER_LOW_TO_HIGH && bind) ? s_oth[m][j] : s_cur[m][j];
                }
                tp.e_out = tp.e_in = nullptr;
                tp.in_bits = 0;
                // threads beyond this round's width have no pair (they still take part in the block reduction)
                const size_t first = tid < (int)sh.tpb ? (size_t)b * sh.tpb + tid : (size_t)pairs;
                const size_t stride = (size_t)sh.nblk * sh.tpb;
                // passes of >= 2 full sweeps of the grid: the tail of the range is claimed warp by warp
                tp.work = a.st->work + m * 32;
                tp.static_end = ~(size_t)0;
                if (a.static_pct < 100 && live > 1 && sh.tpb == RES_BLOCK && (size_t)pairs >= 2 * stride)
                    tp.static_end = ((size_t)pairs / 100 * (size_t)a.static_pct / stride) * stride;
                uint64_t* gl = a.st->lanes + m * RES_SLOT_U64;
                uint64_t* sl = live == 1 ? s_lanes + m * RES_SLOT_U64 : nullptr;
                if (!bind)
                    resident_pass<D, P, ORDER, false, false>(tp, pairs, sc, dsm, first, stride, gl, sl);
                else if (hi4)
                    resident_pass<D, P, ORDER, true, true>(tp, pairs, sc, dsm, first, stride, gl, sl);
                else
                    resident_pass<D, P, ORDER, true, false>(tp, pairs, sc, dsm, first, stride, gl, sl);
            }
        }
        if (b == 0 && tid == 0) a.mb->tlog2[4 * ((seq - 1) & 63)] = global_timer_ns();
        __syncthreads();
        // ---- state update (identical in every block) + arrival ------------------------------------------
        if (tid == 0) {
            unsigned ln = 0;
            for (int m = 0; m < NM; ++m) {
                const unsigned act = (eff_actions >> (4 * m)) & 0xf;
                if (act == RES_ACT_BIND_EVAL || act == RES_ACT_FINAL) {
                    if (ORDER == ORDER_LOW_TO_HIGH) {
#pragma unroll
                        for (int j = 0; j < T; ++j) {
                            uint64_t* t = s_cur[m][j];
                            s_cur[m][j] = s_oth[m][j];
                            s_oth[m][j] = t;
                        }
                    }
                    s_len[m] /= 2;
                }
                // largest pass this member can still ask for: an eval over len/2 pairs (not started) or a
                // terminal bind over len/2 outputs
                const unsigned need = res_need_blocks(D, P, s_len[m], grid);
                ln = need > ln ? need : ln;
            }
            s_live_next = ln < live ? ln : live;  // (a gather enlarges the tables; blocks that have left stay gone)
            if (live > 1) {
                __threadfence();
                const unsigned ticket = atomicAdd(&a.st->ticket, 1u);
                s_last = (ticket == live - 1);
            } else {
                s_last = 1;
            }
            if (b == 0) a.mb->tlog2[4 * ((seq - 1) & 63) + 1] = global_timer_ns();
            if (s_last) a.mb->tlog2[4 * ((seq - 1) & 63) + 2] = global_timer_ns();
        }
        __syncthreads();
        const unsigned ln = s_live_next;
        // A block that is alone (live == 1) is poller AND answerer: its warp 0 goes straight back to polling for the
        // next command while warps 1..7 publish this round's answer - the system-scope fence of the publication
        // (~2 us over PCIe) then overlaps the poll's PCIe read instead of preceding it. With lookahead the next
        // command is usually already posted, so this is on the critical path of every short round.
        const bool solo = live == 1;
        if (s_last && !(solo && warp == 0)) {
            // ---- the last block to arrive collects every member's lanes and answers the host ------------
            const int pt = solo ? tid - 32 : tid, pn = solo ? RES_BLOCK - 32 : RES_BLOCK;  // publisher threads
            if (live > 1) {
                __threadfence();
                for (int idx = tid; idx < NM * RES_SLOT_U64; idx += RES_BLOCK) {
                    const int m = idx / RES_SLOT_U64, i = idx % RES_SLOT_U64;
                    const unsigned act = (actions >> (4 * m)) & 0xf;
                    if ((act == RES_ACT_EVAL || act == RES_ACT_BIND_EVAL) && i < s_kl[m]) {
                        s_lanes[idx] = __ldcg(a.st->lanes + idx);
                        a.st->lanes[idx] = 0;  // back to zero for the next round
                    }
                }
                if (tid < NM) a.st->work[tid * 32] = 0;
                __syncthreads();
            }
            uint64_t status = 0;
            uint64_t* const result = a.mb->result[seq & 1];
            if (cmdw & RES_FLAG_EXCHANGE) {
                // all-reduce of member 0's lanes over NVLink peer memory (integer sums: exact, order-free)
                if (pt < 32) {
                    const int KL = s_kl[0];
                    const int par = (int)(xseq & 1);
                    const int slot = (par * 16 + a.rank) * XCH_SLOT_U64;
                    for (int idx = lane; idx < a.world * KL; idx += 32) {
                        const int g = idx / KL, i = idx % KL;
                        *(volatile uint64_t*)(a.peer[g] + slot + i) = s_lanes[i];
                    }
                    __syncwarp();
                    __threadfence_system();  // cumulative: covers the other lanes' stores ordered by the barrier
                    if (lane < a.world) *(volatile uint64_t*)(a.peer[lane] + XCH_FLAG_BASE + par * 16 + a.rank) = xseq;
                    uint64_t* mine = a.peer[a.rank];
                    bool ok = true;
                    if (lane < a.world) {
                        const long long t0 = clock64();
                        while (*(volatile uint64_t*)(mine + XCH_FLAG_BASE + par * 16 + lane) != xseq) {
                            if (clock64() - t0 > a.timeout_cycles) {
                                ok = false;
                                break;
                            }
                        }
                    }
                    ok = __all_sync(0xffffffffu, ok);
                    __threadfence_system();
                    for (int i = lane; i < KL; i += 32) {
                        uint64_t sum = 0;
                        for (int src = 0; src < a.world; ++src)
                            sum += *(volatile uint64_t*)(mine + (par * 16 + src) * XCH_SLOT_U64 + i);
                        result[i] = sum;
                    }
                    if (!ok) status = 2;
                }
            } else {
                for (int idx = pt; idx < NM * RES_SLOT_U64; idx += pn) {
                    const int m = idx / RES_SLOT_U64, i = idx % RES_SLOT_U64;
                    const unsigned act = (actions >> (4 * m)) & 0xf;
                    if ((act == RES_ACT_EVAL || act == RES_ACT_BIND_EVAL) && i < s_kl[m]) result[idx] = s_lanes[idx];
                }
            }
            // terminal binds that left a member fully bound hand the T values back with the acknowledgement
            for (int idx = pt; idx < NM * T; idx += pn) {
                const int m = idx / T, j = idx % T;
                const unsigned act = (actions >> (4 * m)) & 0xf;
                if (act == RES_ACT_FINAL && s_len[m] == 1) {
                    const Fr v = ld_elem_cg<Fr>(s_cur[m][j], 0);
#pragma unroll
                    for (int w = 0; w < 4; ++w)
                        result[m * RES_SLOT_U64 + j * 4 + w] = (uint64_t)v.v[2 * w] | ((uint64_t)v.v[2 * w + 1] << 32);
                }
            }
            if (solo) asm volatile("bar.sync 1, 224;" ::: "memory");  // the seven publishing warps
            else __syncthreads();
            if (pt == 0) {
                a.mb->tlog[2 * ((seq - 1) & 63) + 1] = global_timer_ns();
                if (live > 1) {
                    a.st->ticket = 0;
                    st_release_gpu(&a.st->done, seq);  // (orders the lane zeroing and the ticket reset before it)
                }
                a.mb->ans[seq & 1].status = status;
                __threadfence_system();  // cumulative over the publishers' result stores (ordered by the barrier)
                a.mb->ans[seq & 1].res_seq = seq;
            }
        }
        if (b >= ln) return;
        live = ln;
        // s_last / s_lanes / s_kl are rewritten only after the next command's barrier; a solo block's warp 0 must
        // not wait for its publishers here (it only touches s_line while it polls)
        if (!solo) __syncthreads();
    }
}

}  // namespace jb
