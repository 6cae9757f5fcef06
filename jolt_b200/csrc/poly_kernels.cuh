// Device kernels for the sumcheck hot path over BN254 Fr (sm_100a):
//   * bind            - Polynomial::bind_with_order, crates/jolt-poly/src/dense.rs:180-263
//                       (legacy DensePolynomial::bind, jolt-prover-legacy/src/poly/dense_mlpoly.rs:71-221)
//   * fused bind+eval - the fused ProveRounds contract, crates/jolt-sumcheck/src/prover.rs:45-72,
//                       restating NaiveSumcheckProver::prove_round (jolt-kernels/src/reference/naive.rs:241-310)
//                       for Expr = product of m dense tables, degree m
//   * eq expansion    - EqPolynomial::evals, crates/jolt-poly/src/eq.rs:221-231, 299-315 (r[0] <-> MSB)
// All are HBM-streaming integer kernels: one field element (32 B) per 256-bit request, one
// output index per thread per iteration, grid-stride over a grid sized in multiples of the SM
// count. No tensor cores (there is no dense contraction on this path).
#pragma once
#include "field.cuh"

namespace jb {

enum : int { ORDER_HIGH_TO_LOW = 0, ORDER_LOW_TO_HIGH = 1 };

// The bind multiplier: either a generic 254-bit element or a 125-bit challenge [0,0,lo,hi].
struct BindScalar {
    uint32_t w[8];
};

template <bool HI4>
__device__ __forceinline__ Fr bind_pair(const Fr& lo, const Fr& hi, const BindScalar& s) {
    Fr d = fp_sub_lazy(hi, lo);  // in (0, 2p)
    Fr m;
    if (HI4) {
        m = fp_mul_hi4(d, s.w + 4);
    } else {
        Fr sv;
#pragma unroll
        for (int i = 0; i < 8; ++i) sv.v[i] = s.w[i];
        m = fp_mul(d, sv);
    }
    return fp_add(lo, m);  // canonical
}

// out[i] = lo + s*(hi - lo).  HighToLow: (in[i], in[i+half]) - may run in place (out == in);
// LowToHigh: (in[2i], in[2i+1]) - out must not alias in.
template <int ORDER, bool HI4>
__global__ void __launch_bounds__(256) bind_kernel(const uint64_t* in, uint64_t* out, size_t half, BindScalar s) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < half; i += stride) {
        if (i + stride < half) {
            if (ORDER == ORDER_HIGH_TO_LOW) {
                prefetch_l2(in, i + stride);
                prefetch_l2(in, i + stride + half);
            } else {
                prefetch_l2(in, 2 * (i + stride));
            }
        }
        Fr lo, hi;
        if (ORDER == ORDER_HIGH_TO_LOW) {
            lo = ld_elem_rw<Fr>(in, i);
            hi = ld_elem_rw<Fr>(in, i + half);
        } else {
            lo = ld_elem<Fr>(in, 2 * i);
            hi = ld_elem<Fr>(in, 2 * i + 1);
        }
        st_elem(out, i, bind_pair<HI4>(lo, hi, s));
    }
}

// ---- block reduction of field elements (warp shuffle, then one smem stage) ---------------------
__device__ __forceinline__ Fr warp_sum(Fr x) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        Fr y;
#pragma unroll
        for (int k = 0; k < 8; ++k) y.v[k] = __shfl_down_sync(0xffffffffu, x.v[k], off);
        x = fp_add(x, y);
    }
    return x;
}

// Sums K accumulators over the block; thread 0 ends up with the totals. smem: (blockDim/32)*K*8 words.
template <int K>
__device__ __forceinline__ void block_sum(Fr (&acc)[K], uint32_t* smem) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    if (nwarps == 1) {  // latency path: a one-warp block needs no shared-memory stage
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = warp_sum(acc[k]);
        return;
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        acc[k] = warp_sum(acc[k]);
        if (lane == 0) {
#pragma unroll
            for (int w = 0; w < 8; ++w) smem[(warp * K + k) * 8 + w] = acc[k].v[w];
        }
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            Fr x = Fr::zero();
            if (lane < nwarps) {
#pragma unroll
                for (int w = 0; w < 8; ++w) x.v[w] = smem[(lane * K + k) * 8 + w];
            }
            acc[k] = warp_sum(x);
        }
    }
}

// Where a fused pass leaves its M+1 round sums. The last block to finish (ticket from `counter`)
// folds the per-block partials, so a round is ONE launch; the totals go either to host-mapped
// pinned memory followed by a sequence flag the host spins on (no memcpy, no stream sync - the
// Fiat-Shamir round trip is the latency floor of a sumcheck), or to device lanes for NCCL.
struct RoundOut {
    uint64_t* partial;    // gridDim.x * K canonical elements
    unsigned int* counter;  // zero on entry, reset to zero by the last block
    uint64_t* result;     // lanes == 0: K canonical elements (host-mapped); lanes == 1: K*8 u64 device lanes
    volatile uint64_t* flag;  // host-mapped; set to `seq` after the results are visible (may be null)
    uint64_t seq;
    int lanes;            // 0: canonical to `result`; 1: device lanes to `result`; 2: peer exchange (below)
    // lanes == 2: the all-reduce is done HERE, over NVLink peer memory. The finishing thread stores this
    // rank's K*8 lanes straight into every peer's exchange buffer (slot [parity][rank]) and raises a
    // per-source sequence flag there, waits until all `world` sources have landed in its own buffer, sums
    // them and publishes the totals (as lanes) to the host-mapped `result` + `flag`. No NCCL launch, no
    // extra kernel: the collective costs one NVLink store/flag round trip inside the round's own launch.
    // Double buffering by the parity of the exchange sequence number `xseq` makes slot reuse safe: a rank
    // can only be one exchange ahead of a peer.
    uint64_t* peer[16];   // exchange buffer of every rank as mapped in THIS process (peer[rank] = own)
    int world, rank;
    uint64_t xseq;
    long long timeout_cycles;
};
constexpr int XCH_SLOT_U64 = 136;                // u64 lanes per (parity, source) slot (a thin round: 8 sums x 17 lanes)
constexpr int XCH_FLAG_BASE = 2 * 16 * XCH_SLOT_U64;  // flags[parity][source] follow the slots
constexpr int XCH_GFLAG_BASE = XCH_FLAG_BASE + 2 * 16;  // gather barrier flags [parity][source]
constexpr size_t XCH_BYTES = (size_t)(XCH_GFLAG_BASE + 2 * 16) * 8;
// The same IPC allocation continues with the GATHER ARENA: once a sharded member's shards are short, every rank
// writes its bound shard straight into every peer's arena (NVLink stores from inside the resident kernel) and all
// ranks finish the remaining rounds on the gathered tables - no kernel exit, no NCCL all-gather. Two halves
// (parity of the context's gather count): a rank can be at most one gather ahead of a peer.
constexpr size_t XCH_ARENA_OFFSET = 65536;                   // bytes from the start of the allocation
constexpr size_t XCH_ARENA_HALF = (size_t)16 << 20;          // bytes per parity half
constexpr size_t XCH_TOTAL_BYTES = XCH_ARENA_OFFSET + 2 * XCH_ARENA_HALF;

template <class F>
__device__ __forceinline__ F ld_elem_cg(const uint64_t* base, size_t idx) {
    F r;
    const uint32_t* p = reinterpret_cast<const uint32_t*>(base) + idx * 8;
    asm volatile("ld.global.cg.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]),
                   "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p));
    return r;
}

// Thread 0 of the finishing block: write the K totals, then (host-mapped mode) raise the flag.
template <int K>
__device__ __forceinline__ void publish_round(const Fr (&tot)[K], const RoundOut& out) {
    if (out.lanes == 2) {
        const int par = (int)(out.xseq & 1);
        const int slot = (par * 16 + out.rank) * XCH_SLOT_U64;
        for (int g = 0; g < out.world; ++g) {
            uint64_t* dst = out.peer[g] + slot;
#pragma unroll
            for (int t = 0; t < K; ++t)
#pragma unroll
                for (int w = 0; w < 8; ++w) dst[t * 8 + w] = tot[t].v[w];
        }
        __threadfence_system();
        for (int g = 0; g < out.world; ++g)
            *(volatile uint64_t*)(out.peer[g] + XCH_FLAG_BASE + par * 16 + out.rank) = out.xseq;
        // wait for every source's lanes of this exchange to land in OUR buffer
        uint64_t* mine = out.peer[out.rank];
        const long long t0 = clock64();
        bool ok = true;
        for (int src = 0; src < out.world && ok; ++src) {
            while (*(volatile uint64_t*)(mine + XCH_FLAG_BASE + par * 16 + src) != out.xseq) {
                if (clock64() - t0 > out.timeout_cycles) {
                    ok = false;
                    break;
                }
            }
        }
        __threadfence_system();
        for (int i = 0; i < K * 8; ++i) {
            uint64_t sum = 0;
            for (int src = 0; src < out.world; ++src)
                sum += *(volatile uint64_t*)(mine + (par * 16 + src) * XCH_SLOT_U64 + i);
            out.result[i] = ok ? sum : ~0ull;
        }
        if (out.flag) {
            __threadfence_system();
            *out.flag = out.seq;
        }
        return;
    }
#pragma unroll
    for (int t = 0; t < K; ++t) {
        if (out.lanes) {
#pragma unroll
            for (int w = 0; w < 8; ++w) out.result[t * 8 + w] = tot[t].v[w];
        } else {
#pragma unroll
            for (int w = 0; w < 4; ++w)
                out.result[t * 4 + w] = (uint64_t)tot[t].v[2 * w] | ((uint64_t)tot[t].v[2 * w + 1] << 32);
        }
    }
    if (out.flag) {
        __threadfence_system();
        *out.flag = out.seq;
    }
}

// Called by every thread of every block after thread 0 holds the block's K sums in acc[].
template <int K>
__device__ __forceinline__ void round_epilogue(Fr (&acc)[K], uint32_t* smem, const RoundOut& out) {
    __shared__ bool is_last;
    if (gridDim.x == 1) {  // latency path: nothing to fold, publish the block's sums directly
        if (threadIdx.x == 0) publish_round<K>(acc, out);
        return;
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int t = 0; t < K; ++t) st_elem(out.partial, (size_t)blockIdx.x * K + t, acc[t]);
        __threadfence();
        unsigned int ticket = atomicAdd(out.counter, 1u);
        is_last = (ticket == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    Fr tot[K];
#pragma unroll
    for (int t = 0; t < K; ++t) {
        tot[t] = Fr::zero();
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x)
            tot[t] = fp_add(tot[t], ld_elem_cg<Fr>(out.partial, (size_t)b * K + t));
    }
    block_sum<K>(tot, smem);
    if (threadIdx.x == 0) {
        *out.counter = 0;
        publish_round<K>(tot, out);
    }
}

constexpr int JB_MAX_TABLES = 8;  // tables of one member: D factors x P terms

struct TablePtrs {
    const uint64_t* in[JB_MAX_TABLES];
    uint64_t* out[JB_MAX_TABLES];
    // WEIGHTED passes (split-eq members): the pair y carries the weight e_out[y >> in_bits] * e_in[y & mask]
    // (TensorEqTable::evaluate_index, crates/jolt-poly/src/split_eq.rs:52-56); both tables are ~sqrt(N) long.
    const uint64_t* e_out;
    const uint64_t* e_in;
    int in_bits;
    // DYN passes (resident kernel): pair indices below static_end are laid out statically (grid-stride); the rest
    // is handed out 32 indices at a time, one warp per claim, from the counter *work (zero at the start of a pass).
    // static_end is a multiple of the grid stride; SIZE_MAX = everything static.
    unsigned int* work;
    size_t static_end;
};

// Fused pass for a sum-of-products member  sum_x sum_{k<P} prod_{j<D} f_{kD+j}(x)  (degree D, T = D*P tables;
// P = 1 is the plain product member; D = 2, P = 2 is the reference's IncClaimReduction summand
// A*RamInc + B*RdInc, crates/jolt-kernels/src/optimized/inc_claim_reduction.rs:146-156):
//   BIND: first fold every table under `s` (writing the bound table), then
//   sweep the BOUND tables for the round polynomial s(t) = sum_y sum_k prod_j (lo_j(y) + t D_j(y)),
//   D_j = hi_j - lo_j. The pass emits K values, in this order:
//     s(0), [s(1) unless SKIP1], s(2), .., s(D-1), s(inf)          (D >= 2)
//     s(0), [s(1) unless SKIP1]                                    (D == 1)
//   where s(inf) = sum_y sum_k prod_j D_j(y) is the leading coefficient: evaluating at infinity instead of
//   t = D needs no lo + t*D advance at all for D = 2 (s(1) uses hi_j directly), the same trade the
//   reference makes in UnivariatePoly::from_evals_toom / the optimized tier's skipped evaluations
//   (jolt-poly/src/univariate.rs:219-, jolt-kernels/src/optimized/support.rs:450-460). With SKIP1
//   the host derives s(1) = previous_claim - s(0). The host rebuilds s(D) (capi.cu, assemble_evals).
// `pairs` = number of y indices = (bound length)/2. Layout:
//   HighToLow, BIND : reads e[y], e[y+P], e[y+2P], e[y+3P] (P = pairs); writes e'[y], e'[y+P] in place
//   LowToHigh, BIND : reads e[4y..4y+3]; writes out[2y], out[2y+1]   (out-of-place)
//   no BIND         : reads the pair only, writes nothing
// The last factor of every product is multiplied in WITHOUT reduction into a 544-bit per-thread
// accumulator kept in SHARED memory (mul_wide_acc_smem; the GPU form of the reference's
// WideAccumulator) and reduced once per BLOCK after the loop. D == 1 has no product and accumulates plain
// field sums. All sums are exact field values, so the reduction order does not matter.
template <int D, bool SKIP1>
struct FusedShape {
    static constexpr int K = SKIP1 ? D : D + 1;  // number of values produced
    // dynamic shared memory: K accumulators x 17 words x BLOCK threads (D > 1) + the block-sum scratch
    __host__ __device__ static constexpr size_t acc_words(int block) { return (D == 1) ? 0 : (size_t)K * 17 * block; }
    __host__ __device__ static constexpr size_t smem_bytes(int block) { return (acc_words(block) + 8 * K * 8) * 4; }
};

// NC: the tables are read-only for the lifetime of the kernel (one launch per round) -> non-coherent loads.
// A resident kernel reads what OTHER blocks wrote in the previous round, so it takes the coherent path.
template <bool NC>
__device__ __forceinline__ Fr ld_tab(const uint64_t* base, size_t idx) {
    return NC ? ld_elem<Fr>(base, idx) : ld_elem_rw<Fr>(base, idx);
}

// The body of a pass: thread `first` .. step `stride` over the pair indices. On return thread 0 of the block
// holds the block's K sums in acc[] and a __syncthreads() has been executed (dsm may be reused).
// dsm: FusedShape<D, SKIP1>::smem_bytes(BLOCK) bytes of dynamic shared memory.
// RAW (D > 1): skip the block's Montgomery reduction and leave the K x 17 integer column sums (u64) in the scratch
// area dsm + acc_words - the resident kernel ships them to the host, which does the O(K) serial reduction far
// faster than one GPU lane can (acc[] is then not written).
// DYN: the tail of the index range is claimed dynamically (TablePtrs::work / static_end): the SMs do not all
// stream at the same rate (measured: the slowest block of a 2^21-pair pass arrives ~20 % after the fastest), and
// a round ends when the LAST block arrives - blocks that are ahead take more of the tail.
template <int D, int P, int ORDER, bool BIND, bool HI4, bool SKIP1, int BLOCK, bool WEIGHTED, bool NC, bool RAW = false,
          bool DYN = false>
__device__ __forceinline__ void fused_pass(const TablePtrs& tp, size_t pairs, const BindScalar& s, uint32_t* dsm,
                                           size_t first, size_t stride, Fr (&acc)[FusedShape<D, SKIP1>::K]) {
    constexpr int K = FusedShape<D, SKIP1>::K;
    constexpr int T = D * P;
    uint32_t* wacc = dsm;                                       // [e][word][tid]
    uint32_t* red = dsm + FusedShape<D, SKIP1>::acc_words(BLOCK);  // block_sum scratch
    const int tid = threadIdx.x;
    Fr sum1[D == 1 ? K : 1];
    if (D == 1) {
#pragma unroll
        for (int e = 0; e < K; ++e) sum1[e] = Fr::zero();
    } else {
#pragma unroll
        for (int e = 0; e < K; ++e)
#pragma unroll
            for (int w = 0; w < 17; ++w) wacc[(e * 17 + w) * BLOCK + tid] = 0;
    }

    // Eval-only passes (no bind) have registers to spare: the NEXT iteration's pair is loaded into registers
    // before the current one is multiplied (software pipelining), so the DRAM latency of an iteration hides
    // behind the previous iteration's arithmetic instead of behind other warps - there are only 16 per SM.
    // (ptxas sinks the L2 prefetch below to the end of the loop body, so on its own it buys no lead time.)
    constexpr bool PIPE = !BIND && P == 1 && (D == 1 || (D == 2 && SKIP1));
    // The index sequence of a thread: first, first + stride, ... while below S (static part), then warp-wide claims.
    const size_t S = DYN ? tp.static_end : (size_t)0;
    bool dyn = false;
    auto claim = [&]() -> size_t {  // warp-uniform: every lane of the warp is in the loop or none is
        unsigned c = 0;
        if ((tid & 31) == 0) c = atomicAdd(tp.work, 1u);
        c = __shfl_sync(0xffffffffu, c, 0);
        return S + (size_t)c * 32 + (tid & 31);
    };
    auto advance = [&](size_t prev) -> size_t {
        if (!DYN) return prev + stride;
        if (!dyn && prev + stride < S) return prev + stride;  // (uniform over the grid: S is a multiple of stride)
        dyn = true;
        return claim();
    };
    size_t ystart = first;
    if (DYN && first >= S && first < pairs) {  // (no static part at all)
        dyn = true;
        ystart = claim();
    }
    Fr nlo[PIPE ? D : 1], nhi[PIPE ? D : 1];
    if (PIPE) {
        const size_t y0 = ystart;
        if (y0 < pairs) {
#pragma unroll
            for (int j = 0; j < D; ++j) {
                if (ORDER == ORDER_HIGH_TO_LOW) {
                    nlo[j] = ld_tab<NC>(tp.in[j], y0);
                    nhi[j] = ld_tab<NC>(tp.in[j], y0 + pairs);
                } else {
                    nlo[j] = ld_tab<NC>(tp.in[j], 2 * y0);
                    nhi[j] = ld_tab<NC>(tp.in[j], 2 * y0 + 1);
                }
            }
        }
    }
    // Two indices of lookahead: y1 is the next iteration's, y2 the one after. Eval-only passes load y1 into registers
    // and prefetch y2's lines into L2; bind passes prefetch y1's lines (ptxas sinks that prefetch to the end of the
    // loop body; prefetching y2 there instead measured 8-13 % SLOWER on the 2^20..2^21-pair rounds, r02 probe).
    auto prefetch_pair = [&](size_t yn) {
        if (yn < pairs) {
#pragma unroll
            for (int j = 0; j < T; ++j) {
                if (ORDER == ORDER_HIGH_TO_LOW) {
                    prefetch_l2(tp.in[j], yn);
                    prefetch_l2(tp.in[j], yn + pairs);
                    if (BIND) {
                        prefetch_l2(tp.in[j], yn + 2 * pairs);
                        prefetch_l2(tp.in[j], yn + 3 * pairs);
                    }
                } else {
                    prefetch_l2(tp.in[j], (BIND ? 4 : 2) * yn);  // 4 (or 2) consecutive elements: one line
                }
            }
        }
    };
    size_t y1 = (ystart < pairs) ? advance(ystart) : pairs;
    for (size_t y = ystart; y < pairs;) {
        const size_t ynext = y1;
        const size_t y2 = (y1 < pairs) ? advance(y1) : pairs;
        prefetch_pair(PIPE ? y2 : y1);
        Fr wgt;
        if (WEIGHTED) {
            const size_t mask = ((size_t)1 << tp.in_bits) - 1;
            wgt = fp_mul(ld_elem<Fr>(tp.e_out, y >> tp.in_bits), ld_elem<Fr>(tp.e_in, y & mask));
        }
#pragma unroll
        for (int k = 0; k < P; ++k) {  // one product term at a time: D tables live in registers
            Fr lo[D], hi[D];
            if (PIPE) {
#pragma unroll
                for (int j = 0; j < D; ++j) {
                    lo[j] = nlo[j];
                    hi[j] = nhi[j];
                }
                const size_t yn = ynext;
                if (yn < pairs) {
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        if (ORDER == ORDER_HIGH_TO_LOW) {
                            nlo[j] = ld_tab<NC>(tp.in[j], yn);
                            nhi[j] = ld_tab<NC>(tp.in[j], yn + pairs);
                        } else {
                            nlo[j] = ld_tab<NC>(tp.in[j], 2 * yn);
                            nhi[j] = ld_tab<NC>(tp.in[j], 2 * yn + 1);
                        }
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < D; ++j) {
                if (PIPE) break;
                const uint64_t* in = tp.in[k * D + j];
                uint64_t* out = tp.out[k * D + j];
                if (BIND) {
                    Fr a, b, c, d;
                    if (ORDER == ORDER_HIGH_TO_LOW) {
                        a = ld_elem_rw<Fr>(in, y);
                        c = ld_elem_rw<Fr>(in, y + 2 * pairs);
                        b = ld_elem_rw<Fr>(in, y + pairs);
                        d = ld_elem_rw<Fr>(in, y + 3 * pairs);
                        lo[j] = bind_pair<HI4>(a, c, s);
                        hi[j] = bind_pair<HI4>(b, d, s);
                        st_elem(out, y, lo[j]);
                        st_elem(out, y + pairs, hi[j]);
                    } else {
                        a = ld_tab<NC>(in, 4 * y);
                        b = ld_tab<NC>(in, 4 * y + 1);
                        c = ld_tab<NC>(in, 4 * y + 2);
                        d = ld_tab<NC>(in, 4 * y + 3);
                        lo[j] = bind_pair<HI4>(a, b, s);
                        hi[j] = bind_pair<HI4>(c, d, s);
                        st_elem(out, 2 * y, lo[j]);
                        st_elem(out, 2 * y + 1, hi[j]);
                    }
                } else {
                    if (ORDER == ORDER_HIGH_TO_LOW) {
                        lo[j] = ld_elem_rw<Fr>(in, y);
                        hi[j] = ld_elem_rw<Fr>(in, y + pairs);
                    } else {
                        lo[j] = ld_tab<NC>(in, 2 * y);
                        hi[j] = ld_tab<NC>(in, 2 * y + 1);
                    }
                }
            }
            if (WEIGHTED) {
                lo[0] = fp_mul(lo[0], wgt);
                hi[0] = fp_mul(hi[0], wgt);
            }
            if (D == 1) {
                sum1[0] = fp_add(sum1[0], lo[0]);
                if (!SKIP1) sum1[K - 1] = fp_add(sum1[K - 1], hi[0]);
            } else {
                int e = 0;
                {  // t = 0
                    Fr prod = lo[0];
#pragma unroll
                    for (int j = 1; j < D - 1; ++j) prod = fp_mul(prod, lo[j]);
                    mul_wide_acc_smem(wacc + (e * 17) * BLOCK + tid, BLOCK, prod.v, lo[D - 1].v);
                    ++e;
                }
                if (!SKIP1) {  // t = 1: lo + D = hi
                    Fr prod = hi[0];
#pragma unroll
                    for (int j = 1; j < D - 1; ++j) prod = fp_mul(prod, hi[j]);
                    mul_wide_acc_smem(wacc + (e * 17) * BLOCK + tid, BLOCK, prod.v, hi[D - 1].v);
                    ++e;
                }
                Fr dlt[D];
#pragma unroll
                for (int j = 0; j < D; ++j) dlt[j] = (D == 2) ? fp_sub_lazy(hi[j], lo[j]) : fp_sub(hi[j], lo[j]);
                if (D > 2) {  // t = 2 .. D-1
                    Fr cur[D];
#pragma unroll
                    for (int j = 0; j < D; ++j) cur[j] = hi[j];
#pragma unroll
                    for (int t = 2; t < D; ++t) {
#pragma unroll
                        for (int j = 0; j < D; ++j) cur[j] = fp_add(cur[j], dlt[j]);
                        Fr prod = cur[0];
#pragma unroll
                        for (int j = 1; j < D - 1; ++j) prod = fp_mul(prod, cur[j]);
                        mul_wide_acc_smem(wacc + (e * 17) * BLOCK + tid, BLOCK, prod.v, cur[D - 1].v);
                        ++e;
                    }
                }
                {  // t = infinity: the leading coefficient prod_j D_j
                    Fr prod = dlt[0];
#pragma unroll
                    for (int j = 1; j < D - 1; ++j) prod = fp_mul(prod, dlt[j]);
                    mul_wide_acc_smem(wacc + (e * 17) * BLOCK + tid, BLOCK, prod.v, dlt[D - 1].v);
                }
            }
        }
        y = y1;
        y1 = y2;
    }
    if (D == 1) {
#pragma unroll
        for (int e = 0; e < K; ++e) acc[e] = sum1[e];
        block_sum<K>(acc, red);
    } else {
        // Block sum of the wide accumulators BEFORE the Montgomery reduction: the K x 17 word columns are summed
        // over the block's threads as plain integers (a column sum is < 2^40; the block total stays far below
        // 2^544: at most P * pairs / gridDim.x products of < 2^512 each), then lane e of warp 0 propagates the carries
        // of value e and reduces ONCE. One reduction per block instead of one per thread: the per-thread
        // reductions were ~13 % of the instructions a pass issued (ncu, profiles/r01b_ncu_fused_round_kernels.md).
        uint64_t* colsum = reinterpret_cast<uint64_t*>(red);  // K * 17 u64 <= the 8 * K * 8 words of scratch
        const int lane = tid & 31, warp = tid >> 5, nwarps = (int)blockDim.x >> 5;
        __syncthreads();
        for (int c = warp; c < K * 17; c += nwarps) {
            uint64_t sacc = 0;
            for (int t = lane; t < (int)blockDim.x; t += 32) sacc += wacc[c * BLOCK + t];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) sacc += __shfl_down_sync(0xffffffffu, sacc, off);
            if (lane == 0) colsum[c] = sacc;
        }
        __syncthreads();
        if (!RAW && warp == 0) {
            Fr mine = Fr::zero();
            if (lane < K) {
                uint32_t Tw[17];
                uint64_t carry = 0;
#pragma unroll
                for (int w = 0; w < 17; ++w) {
                    const uint64_t t = colsum[lane * 17 + w] + carry;
                    Tw[w] = (uint32_t)t;
                    carry = t >> 32;
                }
                mine = reduce_wide17<FrParams>(Tw, 1);
            }
#pragma unroll
            for (int e = 0; e < K; ++e)
#pragma unroll
                for (int w = 0; w < 8; ++w) acc[e].v[w] = __shfl_sync(0xffffffffu, mine.v[w], e);
        }
    }
    __syncthreads();  // scratch is reused by the caller (the last block's fold)
}

// One launch per round: BLOCK threads per block, MINB = resident blocks per SM requested from
// ptxas. WEIGHTED: the sweep is sum_y E(y) prod_j(...) with the split-eq weight E(y) = e_out * e_in folded into
// table 0's pair AFTER the bound values are stored (GruenSplitEqPolynomial, split_eq.rs:159-447: the eq
// polynomial is never materialised or bound as a table; its current variable is a linear factor the host
// multiplies in). Each block writes its sums and the last block folds them (round_epilogue).
template <int D, int P, int ORDER, bool BIND, bool HI4, bool SKIP1, int BLOCK, int MINB, bool WEIGHTED = false>
__global__ void __launch_bounds__(BLOCK, MINB) fused_round_kernel(TablePtrs tp, size_t pairs, BindScalar s, RoundOut out) {
    constexpr int K = FusedShape<D, SKIP1>::K;
    extern __shared__ uint32_t dsm[];
    Fr acc[K];
    fused_pass<D, P, ORDER, BIND, HI4, SKIP1, BLOCK, WEIGHTED, true>(
        tp, pairs, s, dsm, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x, acc);
    round_epilogue<K>(acc, dsm + FusedShape<D, SKIP1>::acc_words(BLOCK), out);
}

// ---- eq-table expansion --------------------------------------------------------------------
// table[x] = scale * prod_i (r_i if bit_i(x) else 1 - r_i), bit_i(x) = bit (n-1-i) of x.
// One block expands EQ_BLOCK_VARS trailing variables from one prefix value:
//   stage 1: the block builds the 2^(nv-3) table of the first nv-3 block variables in shared
//            memory, level by level (1 mul + 1 sub per pair, eq.rs:308-312);
//   stage 2: each thread expands the last 3 variables in registers and writes 8 consecutive
//            outputs (256 B). Total work ~ 1 mul + 1 sub per output, written once: 32 B/output.
constexpr int EQ_BLOCK_VARS = 11;  // 2^11 outputs per block, 256 threads x 8

// The point travels in the kernel-parameter space (<= 11 variables per launch): no staging buffer,
// no host->device copy, no synchronisation on the eq path.
struct EqVars {
    uint32_t r[EQ_BLOCK_VARS][8];  // r[0] = most significant variable of this launch
    uint32_t scale[8];
    int has_scale;
};
__device__ __forceinline__ Fr eq_var(const EqVars& v, int j) {
    Fr x;
#pragma unroll
    for (int w = 0; w < 8; ++w) x.v[w] = v.r[j][w];
    return x;
}

static __global__ void __launch_bounds__(256) eq_expand_kernel(const uint64_t* prefix,  // gridDim.x prefix values (or null: scale)
                                                        const __grid_constant__ EqVars ev, int nv, uint64_t* out) {
    __shared__ uint32_t tab[8 * 256];  // word-major: tab[w*256 + idx] (conflict-free)
    const int tid = threadIdx.x;
    const int reg_vars = nv < 3 ? nv : 3;
    const int smem_vars = nv - reg_vars;  // <= 8
    if (tid == 0) {
        Fr base = Fr::one();
        if (prefix) base = ld_elem_rw<Fr>(prefix, blockIdx.x);
        else if (ev.has_scale) {
#pragma unroll
            for (int w = 0; w < 8; ++w) base.v[w] = ev.scale[w];
        }
#pragma unroll
        for (int w = 0; w < 8; ++w) tab[w * 256] = base.v[w];
    }
    __syncthreads();
    // level j doubles the table: new[2i+1] = old[i]*r_j, new[2i] = old[i] - new[2i+1].
    for (int j = 0; j < smem_vars; ++j) {
        const int cur = 1 << j;
        Fr v, hi;
        if (tid < cur) {
#pragma unroll
            for (int w = 0; w < 8; ++w) v.v[w] = tab[w * 256 + tid];
            hi = fp_mul(v, eq_var(ev, j));
        }
        __syncthreads();
        if (tid < cur) {
            Fr lo = fp_sub(v, hi);
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                tab[w * 256 + 2 * tid] = lo.v[w];
                tab[w * 256 + 2 * tid + 1] = hi.v[w];
            }
        }
        __syncthreads();
    }
    if (tid >= (1 << smem_vars)) return;
    Fr e[8];
#pragma unroll
    for (int w = 0; w < 8; ++w) e[0].v[w] = tab[w * 256 + tid];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        if (j < reg_vars) {  // block-uniform
            Fr rj = eq_var(ev, smem_vars + j);
#pragma unroll
            for (int i = (1 << j) - 1; i >= 0; --i) {
                Fr hi = fp_mul(e[i], rj);
                e[2 * i] = fp_sub(e[i], hi);
                e[2 * i + 1] = hi;
            }
        }
    }
    const int cnt = 1 << reg_vars;
    size_t base_idx = ((size_t)blockIdx.x << nv) + ((size_t)tid << reg_vars);
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (i < cnt) st_elem(out, base_idx + i, e[i]);
}

// Streaming form for n > EQ_BLOCK_VARS: out[(b << 11) | (k << 8) | t] = prefix[b] * low8[t] * eq3[k]
// where low8 is the (unscaled, block-independent) table over the block's last 8 variables, built once
// by eq_expand_kernel, and eq3 the table over its first 3. Each thread forms v = prefix[b] * low8[t]
// (one full product) and expands the three leading variables in registers with the reference's
// doubling step hi = v * r_j, lo = v - hi (eq.rs:308-312) - products by the POINT, so a 125-bit
// challenge point (Montgomery limbs [0,0,lo,hi]) takes the 4-row product: 1 + 7/2 full-product
// equivalents per 8 outputs instead of 8. Every store instruction writes 32 consecutive elements per
// warp (1 KiB, fully coalesced); 32 B of HBM write per output, no reads beyond the 8 KiB low8 table.
// One Montgomery product per output is inherent to an eq table (2^n - 1 products for 2^n leaves), so
// with a full 254-bit point this kernel is bound by the integer pipe (66.8 G mul/s x 32 B = 2.1 TB/s),
// not by HBM.
// CS: streaming (evict-first) stores - the table is written once and consumed by a LATER kernel; keeping 128 MB+ of
// it dirty in L2 only evicts what the consumer wants there (A/B: profiles/r02_eq_store_ab.md).
// Layout: a thread's 8 outputs are 8 KiB apart so that each store instruction covers 1 KiB per warp. The
// alternative, 8 consecutive outputs per thread, writes the same DRAM bytes (2.03 x the table at 2^26 either
// way) and measured 7 % slower (profiles/r02_eq_store_ab.md).
template <bool HI4, bool CS>
__global__ void __launch_bounds__(256) eq_stream_kernel(const uint64_t* prefix, const __grid_constant__ EqVars ev,
                                                        const uint64_t* low8, uint64_t* out) {
    const int tid = threadIdx.x;
    Fr e[8];
    e[0] = fp_mul(ld_elem_rw<Fr>(prefix, blockIdx.x), ld_elem_rw<Fr>(low8, tid));
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const Fr rj = eq_var(ev, j);
#pragma unroll
        for (int i = (1 << j) - 1; i >= 0; --i) {
            Fr hi = HI4 ? fp_mul_hi4(e[i], rj.v + 4) : fp_mul(e[i], rj);
            e[2 * i] = fp_sub(e[i], hi);
            e[2 * i + 1] = hi;
        }
    }
    const size_t base = ((size_t)blockIdx.x << EQ_BLOCK_VARS) + (size_t)tid;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const size_t idx = base + ((size_t)k << 8);
        if (CS) st_elem_cs(out, idx, e[k]);
        else st_elem(out, idx, e[k]);
    }
}

// ---- element-wise helpers (tests + host glue) --------------------------------------------------
// op: 0 add, 1 sub, 2 mul (Montgomery), 3 mul with b's 4 low words zero (hi4 path), 4 neg(a), 5 square(a)
template <class F>
__global__ void vec_op_kernel(const uint64_t* a, const uint64_t* b, uint64_t* o, size_t n, int op) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    F x = ld_elem<F>(a, i), y = ld_elem<F>(b, i), z;
    if (op == 0) z = fp_add(x, y);
    else if (op == 1) z = fp_sub(x, y);
    else if (op == 2) z = fp_mul(x, y);
    else if (op == 3) z = fp_mul_hi4(x, y.v + 4);
    else if (op == 4) z = fp_neg(x);
    else z = fp_sqr(x);
    st_elem(o, i, z);
}

}  // namespace jb
