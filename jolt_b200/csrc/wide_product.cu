// Fused bind + sweep for products of many tables: the round of a product member of 5..8 tables, and of a split-eq
// member of 4..8 tables (restating NaiveSumcheckProver::prove_round, jolt-kernels/src/reference/naive.rs:241-310, and
// the split-eq product of d tables, mles_product_sum.rs, for any d up to 8).
//
// It keeps every contract of fused_pass (poly_kernels.cuh): the same table layout and binds (HighToLow in place,
// LowToHigh out of place into the alternate buffer, eval-only without a bind), the same K values in the same order
//     s(0), [s(1) unless SKIP1], s(2), .., s(D-1), s(inf)
// canonical, folded by the last block and published through RoundOut / round_epilogue. So member_round,
// wait_round_result and assemble_evals consume its output unchanged.
//
// What differs is how a pair index is evaluated. fused_pass multiplies the D factors lo_j + t D_j point by point:
// D - 1 products for each of the K points, ~D^2 per pair index, with lo[D], hi[D], dlt[D] and cur[D] live at once.
// Here the product is a balanced tree of polynomials in t, each known by its values at 0..N-1 and its leading
// coefficient (WPoly<N>):
//   * a leaf is one factor lo + t D (values lo and D: no product);
//   * two children of degrees A and B are stepped to the points 0..A+B-1 by forward differences (additions only: the
//     N-th difference of a degree-N polynomial is the constant N! lead) and multiplied point by point, plus the
//     product of the leads: A + B + 1 products;
//   * at the root the two halves are stepped through the K points and multiplied into the unreduced accumulators.
// Products per pair index (with SKIP1, binds and split-eq weight not counted):
//     D       4    5    6    7    8
//     tree   10   15   20   25   30        (point by point: 12, 20, 30, 42, 56)
// A bind adds 2 products per table (half-width for a 125-bit challenge), the split-eq weight 3.
//
// Bounds. Every factor, tree value and lead is canonical (< p): fp_add, fp_sub and fp_mul reduce fully. The root
// multiplies two canonical values WITHOUT reduction, a < p^2 < 2^508 integer, into a 17-word (544-bit) per-thread
// accumulator in shared memory: a thread may carry up to 2^36 pair indices per round before it could overflow. The
// block's column sums are < 2^32 * 128 < 2^39 per word (u64), and the block total stays < 2^544 for the same reason.
//
// Resources. The accumulators take K x 17 words per thread in shared memory, so the block is 128 threads: at K = 9
// that is 78 KiB per block and two blocks fit an SM (the 256-thread layout of fused_pass would need 157 KiB per block).
// Two blocks of 128 threads leave up to 255 registers per thread, which the two stepped halves at the root (2 x 5
// values at D = 8) and the Montgomery rows need without spilling.
#include <cuda_runtime.h>

#include "member.hpp"

namespace jb {

constexpr int WIDE_BLOCK = 128;
constexpr int WIDE_MINB = 2;

// A polynomial of degree N in t: v[0..N-1] = p(0..N-1), v[N] = its leading coefficient (all canonical).
template <int N>
struct WPoly {
    Fr v[N + 1];
};

__host__ __device__ constexpr unsigned wide_factorial(int n) { return n <= 1 ? 1u : (unsigned)n * wide_factorial(n - 1); }

// x * KK for a small constant KK by doubling and adding (additions only)
template <unsigned KK>
__device__ __forceinline__ Fr mul_small(const Fr& x) {
    if constexpr (KK == 1) {
        return x;
    } else if constexpr (KK % 2 == 0) {
        const Fr h = mul_small<KK / 2>(x);
        return fp_add(h, h);
    } else {
        return fp_add(mul_small<KK - 1>(x), x);
    }
}

// Walks a WPoly<N> through t = 0, 1, 2, ...: d[k] is the k-th forward difference at the current t and d[N] = N! lead is
// constant, so one step is N additions.
template <int N>
struct Stepper {
    Fr d[N + 1];
    __device__ __forceinline__ explicit Stepper(const WPoly<N>& p) {
#pragma unroll
        for (int k = 0; k < N; ++k) d[k] = p.v[k];
#pragma unroll
        for (int lvl = 1; lvl < N; ++lvl)
#pragma unroll
            for (int k = N - 1; k >= lvl; --k) d[k] = fp_sub(d[k], d[k - 1]);
        d[N] = mul_small<wide_factorial(N)>(p.v[N]);
    }
    __device__ __forceinline__ const Fr& value() const { return d[0]; }
    __device__ __forceinline__ void step() {
#pragma unroll
        for (int k = 0; k < N; ++k) d[k] = fp_add(d[k], d[k + 1]);
    }
};

// a * b at 0..A+B-1 and the product of the leads: A + B + 1 products
template <int A, int B>
__device__ __forceinline__ WPoly<A + B> wmul(const WPoly<A>& a, const WPoly<B>& b) {
    WPoly<A + B> r;
    Stepper<A> sa(a);
    Stepper<B> sb(b);
#pragma unroll
    for (int t = 0; t < A + B; ++t) {
        r.v[t] = fp_mul(sa.value(), sb.value());
        if (t + 1 < A + B) {
            sa.step();
            sb.step();
        }
    }
    r.v[A + B] = fp_mul(a.v[A], b.v[B]);
    return r;
}

// the product of factors [LO, LO + N) as a WPoly<N>; leaf(j) yields factor j as a WPoly<1>
template <int LO, int N, class Leaf>
__device__ __forceinline__ WPoly<N> wtree(Leaf& leaf) {
    if constexpr (N == 1) {
        return leaf(LO);
    } else {
        constexpr int L = (N + 1) / 2;
        const WPoly<L> a = wtree<LO, L>(leaf);
        const WPoly<N - L> b = wtree<LO + L, N - L>(leaf);
        return wmul(a, b);
    }
}

// Grid-stride over the pair indices; on return thread 0 holds the block's K sums in acc[] (see fused_pass for the
// layout of dsm: K x 17 accumulator words x BLOCK, then the block-sum scratch).
template <int D, int ORDER, bool BIND, bool HI4, bool SKIP1, bool WEIGHTED>
__device__ __forceinline__ void wide_pass(const TablePtrs& tp, size_t pairs, const BindScalar& s, uint32_t* dsm,
                                          Fr (&acc)[FusedShape<D, SKIP1>::K]) {
    constexpr int K = FusedShape<D, SKIP1>::K;
    constexpr int BLOCK = WIDE_BLOCK;
    constexpr int L = (D + 1) / 2;  // the root's two halves: factors [0, L) and [L, D)
    uint32_t* wacc = dsm;  // [e][word][tid]
    uint32_t* red = dsm + FusedShape<D, SKIP1>::acc_words(BLOCK);
    const int tid = threadIdx.x;
#pragma unroll
    for (int e = 0; e < K; ++e)
#pragma unroll
        for (int w = 0; w < 17; ++w) wacc[(e * 17 + w) * BLOCK + tid] = 0;

    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t y = (size_t)blockIdx.x * blockDim.x + tid; y < pairs; y += stride) {
        const size_t yn = y + stride;
        if (yn < pairs) {  // the next index's lines into L2 (ptxas sinks this to the end of the loop body)
#pragma unroll
            for (int j = 0; j < D; ++j) {
                if (ORDER == ORDER_HIGH_TO_LOW) {
                    prefetch_l2(tp.in[j], yn);
                    prefetch_l2(tp.in[j], yn + pairs);
                    if (BIND) {
                        prefetch_l2(tp.in[j], yn + 2 * pairs);
                        prefetch_l2(tp.in[j], yn + 3 * pairs);
                    }
                } else {
                    prefetch_l2(tp.in[j], (BIND ? 4 : 2) * yn);
                }
            }
        }
        Fr wgt;
        if (WEIGHTED) {
            const size_t mask = ((size_t)1 << tp.in_bits) - 1;
            wgt = fp_mul(ld_elem<Fr>(tp.e_out, y >> tp.in_bits), ld_elem<Fr>(tp.e_in, y & mask));
        }
        // factor j at this pair index: bind (and store) first, then the split-eq weight goes into factor 0
        auto leaf = [&](int j) -> WPoly<1> {
            const uint64_t* in = tp.in[j];
            uint64_t* out = tp.out[j];
            Fr lo, hi;
            if (BIND) {
                if (ORDER == ORDER_HIGH_TO_LOW) {
                    const Fr a = ld_elem_rw<Fr>(in, y), c = ld_elem_rw<Fr>(in, y + 2 * pairs);
                    const Fr b = ld_elem_rw<Fr>(in, y + pairs), d = ld_elem_rw<Fr>(in, y + 3 * pairs);
                    lo = bind_pair<HI4>(a, c, s);
                    hi = bind_pair<HI4>(b, d, s);
                    st_elem(out, y, lo);
                    st_elem(out, y + pairs, hi);
                } else {
                    const Fr a = ld_elem<Fr>(in, 4 * y), b = ld_elem<Fr>(in, 4 * y + 1);
                    const Fr c = ld_elem<Fr>(in, 4 * y + 2), d = ld_elem<Fr>(in, 4 * y + 3);
                    lo = bind_pair<HI4>(a, b, s);
                    hi = bind_pair<HI4>(c, d, s);
                    st_elem(out, 2 * y, lo);
                    st_elem(out, 2 * y + 1, hi);
                }
            } else if (ORDER == ORDER_HIGH_TO_LOW) {
                lo = ld_elem<Fr>(in, y);
                hi = ld_elem<Fr>(in, y + pairs);
            } else {
                lo = ld_elem<Fr>(in, 2 * y);
                hi = ld_elem<Fr>(in, 2 * y + 1);
            }
            if (WEIGHTED && j == 0) {
                lo = fp_mul(lo, wgt);
                hi = fp_mul(hi, wgt);
            }
            WPoly<1> f;
            f.v[0] = lo;
            f.v[1] = fp_sub(hi, lo);
            return f;
        };
        const WPoly<L> a = wtree<0, L>(leaf);
        const WPoly<D - L> b = wtree<L, D - L>(leaf);
        Stepper<L> sa(a);
        Stepper<D - L> sb(b);
        int e = 0;
#pragma unroll
        for (int t = 0; t < D; ++t) {
            if (!(SKIP1 && t == 1)) {
                mul_wide_acc_smem(wacc + (e * 17) * BLOCK + tid, BLOCK, sa.value().v, sb.value().v);
                ++e;
            }
            if (t + 1 < D) {
                sa.step();
                sb.step();
            }
        }
        mul_wide_acc_smem(wacc + (e * 17) * BLOCK + tid, BLOCK, a.v[L].v, b.v[D - L].v);  // s(inf)
    }
    // block sum of the wide accumulators before the Montgomery reduction, as in fused_pass
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
    if (warp == 0) {
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
    __syncthreads();  // the scratch is reused by the last block's fold
}

template <int D, int ORDER, bool BIND, bool HI4, bool SKIP1, bool WEIGHTED>
__global__ void __launch_bounds__(WIDE_BLOCK, WIDE_MINB) wide_round_kernel(TablePtrs tp, size_t pairs, BindScalar s,
                                                                           RoundOut out) {
    constexpr int K = FusedShape<D, SKIP1>::K;
    extern __shared__ uint32_t dsm[];
    Fr acc[K];
    wide_pass<D, ORDER, BIND, HI4, SKIP1, WEIGHTED>(tp, pairs, s, dsm, acc);
    round_epilogue<K>(acc, dsm + FusedShape<D, SKIP1>::acc_words(WIDE_BLOCK), out);
}

}  // namespace jb

namespace jbi {
namespace {

using namespace jb;

template <int D, int ORDER, bool BIND, bool HI4, bool SKIP1, bool WEIGHTED>
int launch_wide(jb_ctx* c, const TablePtrs& tp, size_t pairs, const BindScalar& s, RoundOut out) {
    auto kernel = wide_round_kernel<D, ORDER, BIND, HI4, SKIP1, WEIGHTED>;
    constexpr size_t smem = FusedShape<D, SKIP1>::smem_bytes(WIDE_BLOCK);
    static int per_sm = [&] {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        int nb = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, WIDE_BLOCK, smem) != cudaSuccess || nb < 1) nb = 1;
        return nb;
    }();
    // grid-stride over whole waves of resident blocks; a round of <= 32 pairs runs as one warp
    const size_t need = (pairs + WIDE_BLOCK - 1) / WIDE_BLOCK;
    const size_t resident = (size_t)c->sm_count * per_sm;
    size_t grid = need < resident ? need : resident;
    if (grid < 1) grid = 1;
    constexpr int K = FusedShape<D, SKIP1>::K;
    int st = c->ensure_partial(grid * K);
    if (st != JB_OK) return st;
    out.partial = c->d_partial;
    const int tix = c->timing_begin(BIND ? 0 : 2, pairs, D);
    const unsigned block = pairs <= 32 ? 32u : (unsigned)WIDE_BLOCK;
    kernel<<<(unsigned)grid, block, smem, c->stream>>>(tp, pairs, s, out);
    c->timing_end(tix);
    c->launches++;
    return c->check(cudaGetLastError(), WEIGHTED ? "wide_round_kernel (weighted) launch" : "wide_round_kernel launch");
}

template <int D, int ORDER, bool SKIP1, bool WEIGHTED>
int launch_wide_bind(jb_ctx* c, const TablePtrs& tp, size_t pairs, bool bind, bool hi4, const BindScalar& s,
                     const RoundOut& out) {
    if (!bind) return launch_wide<D, ORDER, false, false, SKIP1, WEIGHTED>(c, tp, pairs, s, out);
    return hi4 ? launch_wide<D, ORDER, true, true, SKIP1, WEIGHTED>(c, tp, pairs, s, out)
               : launch_wide<D, ORDER, true, false, SKIP1, WEIGHTED>(c, tp, pairs, s, out);
}

template <int D>
int launch_wide_plain(jb_ctx* c, int order, bool skip1, const TablePtrs& tp, size_t pairs, bool bind, bool hi4,
                      const BindScalar& s, const RoundOut& out) {
    if (order == JB_HIGH_TO_LOW)
        return skip1 ? launch_wide_bind<D, ORDER_HIGH_TO_LOW, true, false>(c, tp, pairs, bind, hi4, s, out)
                     : launch_wide_bind<D, ORDER_HIGH_TO_LOW, false, false>(c, tp, pairs, bind, hi4, s, out);
    return skip1 ? launch_wide_bind<D, ORDER_LOW_TO_HIGH, true, false>(c, tp, pairs, bind, hi4, s, out)
                 : launch_wide_bind<D, ORDER_LOW_TO_HIGH, false, false>(c, tp, pairs, bind, hi4, s, out);
}

// split-eq passes always derive s(1) from the claim (SKIP1)
template <int D>
int launch_wide_weighted(jb_ctx* c, int order, const TablePtrs& tp, size_t pairs, bool bind, bool hi4,
                         const BindScalar& s, const RoundOut& out) {
    return order == JB_HIGH_TO_LOW ? launch_wide_bind<D, ORDER_HIGH_TO_LOW, true, true>(c, tp, pairs, bind, hi4, s, out)
                                   : launch_wide_bind<D, ORDER_LOW_TO_HIGH, true, true>(c, tp, pairs, bind, hi4, s, out);
}

}  // namespace

int launch_wide_round(jb_ctx* c, int m, int order, bool skip1, bool weighted, const TablePtrs& tp, size_t pairs, bool bind,
                      bool hi4, const BindScalar& s, const RoundOut& out) {
    if (weighted) {
        switch (m) {
            case 4: return launch_wide_weighted<4>(c, order, tp, pairs, bind, hi4, s, out);
            case 5: return launch_wide_weighted<5>(c, order, tp, pairs, bind, hi4, s, out);
            case 6: return launch_wide_weighted<6>(c, order, tp, pairs, bind, hi4, s, out);
            case 7: return launch_wide_weighted<7>(c, order, tp, pairs, bind, hi4, s, out);
            case 8: return launch_wide_weighted<8>(c, order, tp, pairs, bind, hi4, s, out);
            default: return c->fail(JB_ERR_UNSUPPORTED, "eq member: m must be 1..8");
        }
    }
    switch (m) {
        case 5: return launch_wide_plain<5>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        case 6: return launch_wide_plain<6>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        case 7: return launch_wide_plain<7>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        case 8: return launch_wide_plain<8>(c, order, skip1, tp, pairs, bind, hi4, s, out);
        default: return c->fail(JB_ERR_UNSUPPORTED, "member: m must be 1..8");
    }
}

}  // namespace jbi
