// BN254 G1 multi-scalar multiplication (Pippenger bucket method) for sm_100a.
// Replaces JoltGroup::msm (crates/jolt-crypto/src/ec/group.rs:70, impl ec/bn254/mod.rs:195-212 ->
// ark_ec::VariableBaseMSM::msm_bigint) and therefore kzg_commit (crates/jolt-hyperkzg/src/kzg.rs:15-27).
// The result is defined by value: sum_i [s_i] P_i with s_i the canonical integer of the scalar
// (into_bigint, mod.rs:208); any schedule is admissible (specs/clean-slate-prover.md:565-571).
//
// Pipeline (all on the context's stream, integer pipes only - there is no dense contraction here):
//   1. digits     : scalar -> canonical (one Montgomery product) -> signed base-2^c digits
//                   d_w in [-2^(c-1), 2^(c-1)], + per-(window, bucket) histogram (global REDs)
//   2. scan       : exclusive prefix of the histogram -> bucket offsets and task offsets (3 small kernels)
//   3. scatter    : point indices (with the digit's sign) into bucket order (one atomic each)
//   4. accumulate : one thread per task (a <= max(64, cnt/64)-point chunk of one bucket): XYZZ += +-P
//                   (mixed add, 8M + 2S) - the hot kernel; split buckets are folded by a combine pass
//   5. segments   : per (window, 16-bucket segment) running sums -> sum_b weight(b) * B_b
//   6. windows    : per-window tree sum of the segment results, then 2^(c w) by doubling
//   7. final      : sum of the window points -> Jacobian (X, Y, Z)
// Affine bases live on the device for the lifetime of the SRS handle (HyperKZGProverSetup::g1_powers,
// crates/jolt-hyperkzg/src/scheme.rs:60-66): the per-call `into_affine` of the reference
// (mod.rs:205) becomes a one-time normalisation at upload.
#include <cuda_runtime.h>

#include <cstring>
#include <vector>

#include "ctx.hpp"
#include "ec.cuh"
#include "small_scalar.cuh"

using namespace jb;

namespace {

// buckets per reduction segment: one thread walks a segment (2 general additions per bucket) and then multiplies the
// segment's plain sum by its first bucket number (double-and-add, ~330 products): the multiplication is per SEGMENT, so
// short segments cost work (measured at 2^20 / 2^24 terms, precomputed SRS: 8 buckets 0.88 / 3.76 ms, 16 buckets
// 0.55 / 2.38 ms).
int msm_seg_size(int buckets) {
    return buckets >= (1 << 21) ? 64 : 16;  // 2^24 terms (2^21 buckets): 16 / 32 / 64 = 40.6 / 40.0 / 39.7 ms per MSM; 2^20 terms: 3.17 / 3.26 / 3.61
}

struct MsmPlan {
    int c;        // window bits
    int W;        // windows
    int B;        // buckets per window = 2^(c-1)
    int T;        // segments per window
};

// `bits`: width of the scalars' magnitudes (254 for Fr, 8..128 for the small-scalar kinds).
MsmPlan plan_with(int c, int bits = 254) {
    MsmPlan p;
    p.c = c;
    p.W = (bits + c - 1) / c;
    if (bits - (p.W - 1) * c > c - 1) p.W += 1;  // top window: data < 2^(c-1), so data + carry <= 2^(c-1) = B
    p.B = 1 << (c - 1);
    p.T = (p.B + msm_seg_size(p.B) - 1) / msm_seg_size(p.B);
    return p;
}

// Shared-bucket plan for an SRS with precomputed 2^(c w) P_i: one bucket set for all windows, so the
// window can be much wider (fewer windows = fewer bucket additions) and the 2^(c w) doubling chains and
// per-window reductions disappear. c is fixed when the table is built.
int shared_window_for(size_t srs_len) {
    int lg = 0;
    while (((size_t)1 << (lg + 1)) <= srs_len) ++lg;
    // only windows whose top digit is well populated (254 mod c large): 15 -> 14 bits, 16 -> 14, 17 -> 16,
    // 20 -> 14, 22 -> 12; a near-empty top window would pile n/4 points into each of four buckets
    if (lg >= 24) return 22;
    if (lg >= 20) return 20;
    if (lg >= 18) return 17;
    if (lg >= 16) return 16;
    return 15;
}

// Window size by a small cost model (in mixed-add equivalents): W*n bucket additions, 2.8 per bucket for
// the running-sum reduction, and the serial tail of the sparsely populated top window (254 mod c bits):
// its buckets hold n / 2^(bits-1) points each and are cut into at most 64 chunks, so one thread walks
// max(64, cnt/64) points while the rest of the machine (~5 G adds/s vs ~7 M adds/s per thread) waits.
// Small-scalar kinds (bits < 254) search every window size: a u8 column wants ONE 9-bit window, a u64
// column five 13-bit ones, whatever n is.
MsmPlan plan_for(size_t n, int bits = 254) {
    int lg = 0;
    while (((size_t)1 << (lg + 1)) <= n) ++lg;
    int c0 = lg - 4;  // ~ 2^5 points per bucket
    double best = 0;
    int best_c = 0;
    const bool small = bits < 254;
    for (int c = small ? 4 : c0 - 2; c <= (small ? 16 : c0 + 2); ++c) {
        if (c < 4 || c > 16) continue;
        MsmPlan p = plan_with(c, bits);
        int top_bits = bits - (p.W - 1) * c;
        if (top_bits < 1) top_bits = 1;
        double cnt_top = (double)n / (double)((size_t)1 << (top_bits - 1));
        double chunk = cnt_top / 64.0 < 64.0 ? 64.0 : cnt_top / 64.0;
        if (small && (double)n / (double)p.B / 64.0 > chunk) chunk = (double)n / (double)p.B / 64.0;
        double cost = (double)p.W * (double)n + 2.8 * (double)p.W * (double)p.B + 750.0 * chunk;
        if (best_c == 0 || cost < best) {
            best = cost;
            best_c = c;
        }
    }
    if (best_c == 0) best_c = c0 < 4 ? 4 : 16;
    return plan_with(best_c, bits);
}

// ---- 1. digits ----------------------------------------------------------------------------------
// `kind`: SK_FR = Montgomery Fr limbs; otherwise a primitive integer column (small_scalar.cuh) whose
// magnitude is cut into digits and whose sign flips every digit (msm_u8 .. msm_i128 of the arkworks fork,
// as called from crates/jolt-prover-legacy/src/msm/mod.rs:27-150).
// AGG: equal slots within a warp are counted by ONE atomic (match.any) - witness columns are skewed
// (binary, one-hot, constants: millions of points in one bucket), and same-address atomics serialise.
// Halving rows (HyperKZG's folded polynomials, packed back to back: lengths 2^(h-1), 2^(h-2), .., 2): term g of the
// packed buffer belongs to row r = the number of leading ones of g as an h-bit number, at column g minus the row's
// offset 2^h - 2^(h-r) - i.e. the low h - r - 1 bits of g.
__device__ __forceinline__ int halving_row(unsigned g, int h) { return __clz(~(g << (32 - h))); }
__device__ __forceinline__ unsigned halving_col(unsigned g, int h) { return g & ((1u << (h - halving_row(g, h) - 1)) - 1u); }

// row_w: 0 for one MSM over n terms; otherwise the n terms are n / row_w ROWS of row_w scalars, every row against the
// same bases[0 .. row_w) and with its own (shared-window) bucket set: slot = row * B + bucket (jb_msm_g1_rows).
template <bool AGG>
__global__ void __launch_bounds__(256) msm_digits_kernel(const void* scalars, int kind, const uint64_t* bases, size_t n, int c,
                                                         int W, int B, int shared, uint32_t* digits, unsigned int* hist,
                                                         size_t row_w, int halving) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n;
    if (!AGG && !valid) return;
    Fr k = Fr::zero();
    uint32_t flip = 0;
    bool skip = true;
    if (valid) {
        if (kind == SK_FR) {
            k = fp_from_mont(ld_elem<Fr>((const uint64_t*)scalars, i));  // canonical integer limbs
        } else {
            if (ld_small(scalars, i, kind, k.v)) flip = 0x80000000u;
        }
        // identity bases contribute nothing
        const size_t bi = halving ? halving_col((unsigned)i, halving) : row_w ? i % row_w : i;
        skip = ld_elem<Fq>(bases, 2 * bi).is_zero() && ld_elem<Fq>(bases, 2 * bi + 1).is_zero();
    }
    const size_t row_slot = !valid ? 0 : halving ? (size_t)halving_row((unsigned)i, halving) * (size_t)B
                                        : row_w ? (i / row_w) * (size_t)B : 0;
    uint32_t carry = 0;
    const uint32_t mask = (1u << c) - 1u;
    const int lane = threadIdx.x & 31;
    for (int w = 0; w < W; ++w) {
        int bit = w * c;
        int word = bit >> 5, off = bit & 31;
        uint32_t d = 0;
        if (word < 8) {
            d = k.v[word] >> off;
            if (off + c > 32 && word + 1 < 8) d |= k.v[word + 1] << (32 - off);
        }
        d = (d & mask) + carry;
        uint32_t enc = 0;
        if (d > (uint32_t)B) {  // d in (2^(c-1), 2^c]: use d - 2^c < 0 and carry one up
            uint32_t neg = (1u << c) - d;  // |d - 2^c| in [0, 2^(c-1))
            carry = 1;
            if (neg) enc = neg | 0x80000000u;
        } else {
            carry = 0;
            if (d) enc = d;
        }
        if (skip) enc = 0;
        if (enc) enc ^= flip;
        if (valid) digits[(size_t)w * n + i] = enc;
        const size_t slot = (shared ? row_slot : (size_t)w * B) + ((enc & 0x7fffffffu) - 1);
        if (AGG) {
            const unsigned m = __ballot_sync(0xffffffffu, enc != 0);
            if (enc) {
                const unsigned peers = __match_any_sync(m, (unsigned)slot);
                if (lane == __ffs(peers) - 1) atomicAdd(&hist[slot], (unsigned)__popc(peers));
            }
        } else {
            if (enc) atomicAdd(&hist[slot], 1u);
        }
    }
}

// ---- 2. exclusive scans (one block; the histogram is at most 17 * 2^15 counters): point offsets per
//         bucket AND task offsets per bucket. A bucket's list is cut into q_b <= MSM_MAX_CHUNKS tasks of
//         L_b = max(MSM_CHUNK, ceil(cnt_b / MSM_MAX_CHUNKS)) points, so no thread ever walks more than
//         max(MSM_CHUNK, cnt/64) points: this bounds the skew of short top windows, small scalars and
//         adversarially repeated digits, and evens out the lanes of a warp. ------------------------------
constexpr unsigned MSM_CHUNK = 64;
constexpr unsigned MSM_MAX_CHUNKS = 64;

// q = min(64, ceil(cnt / 64)) chunks of ceil(cnt / q) points: equal-sized chunks keep the lanes of a warp
// in step (a 96-point bucket is 2 x 48, not 64 + 32).
// maxq = MSM_MAX_CHUNKS for field scalars; the small-scalar kinds (a one-hot or binary column puts every
// point into ONE bucket) raise it to MSM_MAX_CHUNKS_SMALL and fold wide buckets with a block per bucket.
constexpr unsigned MSM_MAX_CHUNKS_SMALL = 16384;
// `maxq` carries the task plan: the chunk cap in its low 16 bits, log2 of the smallest chunk above them (0 = MSM_CHUNK).
// Field-scalar MSMs use 128-point chunks: at 2^24 terms with a 22-bit window a bucket holds ~96 points, and 64-point chunks
// made two tasks, a 256-byte partial and a combine pass out of almost every bucket.
__host__ __device__ __forceinline__ unsigned plan_cap(unsigned maxq) { return maxq & 0xffffu; }
__host__ __device__ __forceinline__ unsigned plan_chunk(unsigned maxq) { return (maxq >> 16) ? 1u << (maxq >> 16) : MSM_CHUNK; }
__device__ __forceinline__ unsigned chunk_count(unsigned cnt, unsigned maxq) {
    if (!cnt) return 0;
    const unsigned ch = plan_chunk(maxq), cap = plan_cap(maxq);
    unsigned q = (cnt + ch - 1) / ch;
    return q > cap ? cap : q;
}
__device__ __forceinline__ unsigned chunk_len(unsigned cnt, unsigned maxq) {
    unsigned q = chunk_count(cnt, maxq);
    return q ? (cnt + q - 1) / q : 1;
}

// Three-kernel exclusive scan of (cnt, chunk_count(cnt)) with coalesced access: (a) each block of 1024
// threads scans 4096 counters (4 per thread, one 128-bit load) and emits its two totals, (b) one block
// scans the block totals, (c) the block bases are added. The histogram is zeroed on the way (it becomes
// the scatter cursor).
constexpr int SCAN_PER_BLOCK = 4096;

__device__ __forceinline__ void block_exclusive_scan2(unsigned int& a, unsigned int& b, unsigned int* sm_a, unsigned int* sm_b,
                                                      unsigned int& total_a, unsigned int& total_b) {
    // a, b: per-thread sums in; exclusive prefix over the block's threads out
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned int ia = a, ib = b;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        unsigned int ta = __shfl_up_sync(0xffffffffu, ia, off), tb = __shfl_up_sync(0xffffffffu, ib, off);
        if (lane >= off) { ia += ta; ib += tb; }
    }
    if (lane == 31) { sm_a[warp] = ia; sm_b[warp] = ib; }
    __syncthreads();
    if (warp == 0) {
        unsigned int wa = sm_a[lane], wb = sm_b[lane];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            unsigned int ta = __shfl_up_sync(0xffffffffu, wa, off), tb = __shfl_up_sync(0xffffffffu, wb, off);
            if (lane >= off) { wa += ta; wb += tb; }
        }
        sm_a[lane] = wa;
        sm_b[lane] = wb;
    }
    __syncthreads();
    total_a = sm_a[31];
    total_b = sm_b[31];
    unsigned int base_a = warp ? sm_a[warp - 1] : 0, base_b = warp ? sm_b[warp - 1] : 0;
    a = base_a + ia - a;  // exclusive
    b = base_b + ib - b;
    __syncthreads();
}

__global__ void __launch_bounds__(1024) msm_scan_local_kernel(unsigned int* hist, unsigned int* offsets, unsigned int* toff,
                                                              size_t total, unsigned int* block_sums, unsigned maxq) {
    __shared__ unsigned int sm_a[32], sm_b[32];
    const size_t base = (size_t)blockIdx.x * SCAN_PER_BLOCK + (size_t)threadIdx.x * 4;
    unsigned int c[4] = {0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (base + k < total) c[k] = hist[base + k];
    unsigned int q[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) q[k] = chunk_count(c[k], maxq);
    unsigned int sa = c[0] + c[1] + c[2] + c[3], sb = q[0] + q[1] + q[2] + q[3], ta, tb;
    block_exclusive_scan2(sa, sb, sm_a, sm_b, ta, tb);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (base + k < total) {
            offsets[base + k] = sa;
            toff[base + k] = sb;
            hist[base + k] = 0;
        }
        sa += c[k];
        sb += q[k];
    }
    if (threadIdx.x == 0) {
        block_sums[2 * blockIdx.x] = ta;
        block_sums[2 * blockIdx.x + 1] = tb;
    }
}

// nblocks <= 1024 (total <= 4 Mi counters)
__global__ void __launch_bounds__(1024) msm_scan_blocks_kernel(unsigned int* block_sums, int nblocks, unsigned int* offsets,
                                                               unsigned int* toff, size_t total) {
    __shared__ unsigned int sm_a[32], sm_b[32];
    unsigned int a = threadIdx.x < nblocks ? block_sums[2 * threadIdx.x] : 0;
    unsigned int b = threadIdx.x < nblocks ? block_sums[2 * threadIdx.x + 1] : 0;
    unsigned int ta, tb;
    block_exclusive_scan2(a, b, sm_a, sm_b, ta, tb);
    if (threadIdx.x < nblocks) {
        block_sums[2 * threadIdx.x] = a;
        block_sums[2 * threadIdx.x + 1] = b;
    }
    if (threadIdx.x == 0) {
        offsets[total] = ta;
        toff[total] = tb;
    }
}

__global__ void __launch_bounds__(1024) msm_scan_apply_kernel(unsigned int* offsets, unsigned int* toff, size_t total,
                                                              const unsigned int* block_sums) {
    const unsigned int ba = block_sums[2 * blockIdx.x], bb = block_sums[2 * blockIdx.x + 1];
    const size_t base = (size_t)blockIdx.x * SCAN_PER_BLOCK + (size_t)threadIdx.x * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (base + k < total) {
            offsets[base + k] += ba;
            toff[base + k] += bb;
        }
}

// task -> bucket map (a bucket writes its <= 64 task slots) AND the order in which the accumulation walks the tasks:
// by chunk length, longest first (a counting sort on min(len, 255)). One thread owns one task, so a warp is as slow
// as its longest chunk: in bucket order the lengths of neighbouring tasks are Poisson-distributed (2^20 terms with a
// 20-bit window: mean 26, the longest of 32 is ~41 - a third of the lanes idle); in length order every warp walks
// equal chunks and the long ones start first.
constexpr int MSM_LEN_BINS = 256;
__device__ __forceinline__ int task_len_bin(unsigned cnt, unsigned maxq) {
    const unsigned len = chunk_len(cnt, maxq);
    return MSM_LEN_BINS - 1 - (int)(len < (unsigned)(MSM_LEN_BINS - 1) ? len : (unsigned)(MSM_LEN_BINS - 1));
}
// Both kernels run a fixed grid; block g owns the contiguous bucket range [g * per, (g + 1) * per) and counts in shared
// memory, so the 256 global counters see one atomic per (block, non-empty bin) instead of one per warp and bin.
constexpr int MSM_TASK_BLOCKS = 592;
__global__ void __launch_bounds__(256) msm_len_hist_kernel(const unsigned int* offsets, const unsigned int* toff, size_t nbuckets,
                                                           unsigned maxq, unsigned int* len_hist) {
    __shared__ unsigned int cnt_s[MSM_LEN_BINS];
    cnt_s[threadIdx.x] = 0;
    __syncthreads();
    const size_t per = (nbuckets + gridDim.x - 1) / gridDim.x;
    const size_t b0 = (size_t)blockIdx.x * per, b1 = b0 + per < nbuckets ? b0 + per : nbuckets;
    for (size_t b = b0 + threadIdx.x; b < b1; b += blockDim.x) {
        const unsigned q = toff[b + 1] - toff[b];
        if (q) atomicAdd(&cnt_s[task_len_bin(offsets[b + 1] - offsets[b], maxq)], q);
    }
    __syncthreads();
    if (cnt_s[threadIdx.x]) atomicAdd(&len_hist[threadIdx.x], cnt_s[threadIdx.x]);
}
// len_hist: [0, 256) task counts per bin (read), [256, 512) cursors (zero on entry)
__global__ void __launch_bounds__(256) msm_tasks_kernel(const unsigned int* offsets, const unsigned int* toff, size_t nbuckets,
                                                        unsigned maxq, unsigned int* len_hist, uint32_t* task_bucket,
                                                        uint32_t* order) {
    __shared__ unsigned int bin_base[MSM_LEN_BINS], cnt_s[MSM_LEN_BINS], tmp[MSM_LEN_BINS];
    const int k = threadIdx.x;
    {   // exclusive scan of the 256 bin counts (Hillis-Steele in shared memory)
        const unsigned v = len_hist[k];
        tmp[k] = v;
        cnt_s[k] = 0;
        __syncthreads();
        for (int off = 1; off < MSM_LEN_BINS; off <<= 1) {
            const unsigned add = k >= off ? tmp[k - off] : 0u;
            __syncthreads();
            tmp[k] += add;
            __syncthreads();
        }
        bin_base[k] = tmp[k] - v;  // start of bin k in `order`
    }
    __syncthreads();
    const size_t per = (nbuckets + gridDim.x - 1) / gridDim.x;
    const size_t b0 = (size_t)blockIdx.x * per, b1 = b0 + per < nbuckets ? b0 + per : nbuckets;
    for (size_t b = b0 + k; b < b1; b += blockDim.x) {  // this block's tasks per bin
        const unsigned q = toff[b + 1] - toff[b];
        if (q) atomicAdd(&cnt_s[task_len_bin(offsets[b + 1] - offsets[b], maxq)], q);
    }
    __syncthreads();
    if (cnt_s[k]) bin_base[k] += atomicAdd(&len_hist[MSM_LEN_BINS + k], cnt_s[k]);  // this block's share of bin k
    cnt_s[k] = 0;
    __syncthreads();
    for (size_t b = b0 + k; b < b1; b += blockDim.x) {
        const unsigned t0 = toff[b], q = toff[b + 1] - t0;
        if (!q) continue;
        const int bin = task_len_bin(offsets[b + 1] - offsets[b], maxq);
        const unsigned pos = bin_base[bin] + atomicAdd(&cnt_s[bin], q);
        for (unsigned j = 0; j < q; ++j) {
            task_bucket[t0 + j] = (uint32_t)b;
            order[pos + j] = t0 + j;
        }
    }
}

// ---- 3. scatter -----------------------------------------------------------------------------------
// `shared`: all windows feed one bucket set and the entry addresses the precomputed table row of its
// window (w * stride + i); otherwise one bucket set per window and the entry is the point index.
template <bool AGG>
__global__ void __launch_bounds__(256) msm_scatter_kernel(const uint32_t* digits, size_t n, int W, int B, int shared,
                                                          size_t stride, const unsigned int* offsets, unsigned int* cursor,
                                                          uint32_t* sorted, size_t row_w, int halving, int mode,
                                                          unsigned range_shift) {
    // mode 0: every window in this thread. The positions are random within the destination, and a random 4-byte
    // store dirties a 32-byte sector: once the destination (4 B x windows x terms) outgrows the L2, the scatter runs at
    // the DRAM's sector rate (6.6 ms for 2^24 terms). So big MSMs order the work in TIME by destination region, one
    // grid row (blockIdx.y) per region, so that the region being filled stays in the L2 until its sectors are complete:
    // mode 1 (one bucket set per window): region = window; mode 2 (one shared bucket set): region = a bucket range
    // (slot >> range_shift); every row re-reads the digits (coalesced, cheap) and keeps its own entries.
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n;
    if (!AGG && !valid) return;
    const int lane = threadIdx.x & 31;
    const size_t row_slot = !valid ? 0 : halving ? (size_t)halving_row((unsigned)i, halving) * (size_t)B
                                        : row_w ? (i / row_w) * (size_t)B : 0;
    const size_t col = !valid ? 0 : halving ? halving_col((unsigned)i, halving) : row_w ? i % row_w : i;  // index into the bases / a table row
    const int w_lo = mode == 1 ? (int)blockIdx.y : 0, w_hi = mode == 1 ? (int)blockIdx.y + 1 : W;
    if (!AGG) {
        // digit -> atomic on the bucket's cursor -> store is a dependent chain of L2 round trips (ncu: long_scoreboard 86 %
        // with one window at a time); the windows of a term are independent, so eight of them are put in flight together:
        // all the digit loads, then all the atomics and offset loads, then the stores.
        constexpr int SW = 8;
        for (int w0 = w_lo; w0 < w_hi; w0 += SW) {
            uint32_t enc[SW];
            size_t slot[SW];
#pragma unroll
            for (int j = 0; j < SW; ++j) enc[j] = (w0 + j < w_hi) ? __ldcs(&digits[(size_t)(w0 + j) * n + i]) : 0u;  // streaming: leave the L2 to the destination
#pragma unroll
            for (int j = 0; j < SW; ++j) {
                slot[j] = (shared ? row_slot : (size_t)(w0 + j) * B) + ((enc[j] & 0x7fffffffu) - 1);
                if (mode == 2 && enc[j] && (unsigned)(slot[j] >> range_shift) != blockIdx.y) enc[j] = 0;
            }
            unsigned int pos[SW], off[SW];
#pragma unroll
            for (int j = 0; j < SW; ++j) {
                pos[j] = off[j] = 0;
                if (enc[j]) {
                    pos[j] = atomicAdd(&cursor[slot[j]], 1u);
                    off[j] = offsets[slot[j]];
                }
            }
#pragma unroll
            for (int j = 0; j < SW; ++j)
                if (enc[j]) sorted[off[j] + pos[j]] = (uint32_t)(shared ? (size_t)(w0 + j) * stride + col : col) | (enc[j] & 0x80000000u);
        }
    } else
    for (int w = w_lo; w < w_hi; ++w) {
        uint32_t enc = valid ? __ldcs(&digits[(size_t)w * n + i]) : 0u;
        const size_t slot = (shared ? row_slot : (size_t)w * B) + ((enc & 0x7fffffffu) - 1);
        if (mode == 2 && enc && (unsigned)(slot >> range_shift) != blockIdx.y) enc = 0;
        // one atomic per distinct slot in the warp; lanes take consecutive positions in lane order
        const unsigned m = __ballot_sync(0xffffffffu, enc != 0);
        if (!enc) continue;
        const unsigned peers = __match_any_sync(m, (unsigned)slot);
        const int leader = __ffs(peers) - 1;
        unsigned int base = 0;
        if (lane == leader) base = atomicAdd(&cursor[slot], (unsigned)__popc(peers));
        base = __shfl_sync(peers, base, leader);
        const unsigned int pos = offsets[slot] + base + (unsigned)__popc(peers & ((1u << lane) - 1u));
        sorted[pos] = (uint32_t)(shared ? (size_t)w * stride + col : col) | (enc & 0x80000000u);
    }
}

// ---- 4. bucket accumulation: the hot kernel. One thread per task (a chunk of one bucket's list). A
//         single-chunk bucket is written straight to `buckets`; chunks of a split bucket go to `partial`
//         and are folded by msm_combine_kernel. --------------------------------------------------------
__global__ void __launch_bounds__(128) msm_accumulate_kernel(const uint64_t* bases, const uint32_t* sorted,
                                                             const unsigned int* offsets, const unsigned int* toff,
                                                             const uint32_t* task_bucket, const uint32_t* order,
                                                             size_t nbuckets, uint64_t* buckets, uint64_t* partial,
                                                             unsigned maxq) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= toff[nbuckets]) return;
    const size_t t = order[k];  // tasks in length order (msm_tasks_kernel)
    const uint32_t b = task_bucket[t];
    const unsigned int base = offsets[b], cnt = offsets[b + 1] - base;
    const unsigned int len = chunk_len(cnt, maxq), j = (unsigned int)t - toff[b];
    unsigned int lo = base + j * len;
    unsigned int hi = lo + len < base + cnt ? lo + len : base + cnt;
    XYZZ acc = XYZZ::inf();
    // The gather is a dependent random 64-byte read per addition: fetch point k+1 while adding point k
    // (the addresses come from the index list, not from the running sum).
    uint32_t e_next = 0;
    Fq nx = Fq::zero(), ny = Fq::zero();
    auto fetch = [&](unsigned int at) {
        e_next = sorted[at];
        nx = ld_elem<Fq>(bases, 2 * (size_t)(e_next & 0x7fffffffu));
        ny = ld_elem<Fq>(bases, 2 * (size_t)(e_next & 0x7fffffffu) + 1);
    };
    if (lo < hi) fetch(lo);
    for (unsigned int i = lo; i < hi; ++i) {
        const uint32_t e = e_next;
        const Fq px = nx, py = ny;
        if (i + 1 < hi) fetch(i + 1);
        xyzz_add_affine(acc, px, py, (e >> 31) != 0);
    }
    if (toff[b + 1] - toff[b] == 1) st_xyzz(buckets, b, acc);
    else st_xyzz(partial, t, acc);
}

// empty buckets -> identity; split buckets -> sum of their chunk partials
__global__ void __launch_bounds__(128) msm_combine_kernel(const unsigned int* toff, size_t nbuckets, const uint64_t* partial,
                                                          uint64_t* buckets) {
    size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbuckets) return;
    unsigned int t0 = toff[b], t1 = toff[b + 1];
    if (t1 - t0 == 1 || t1 - t0 > MSM_MAX_CHUNKS) return;  // wide buckets: msm_combine_wide_kernel
    XYZZ acc = XYZZ::inf();
    for (unsigned int t = t0; t < t1; ++t) xyzz_add(acc, ld_xyzz(partial, t));
    st_xyzz(buckets, b, acc);
}

// ---- 5. segment sums: G = sum_{b in segment} (b + 1) * B_b ---------------------------------------------
__global__ void __launch_bounds__(128) msm_segment_kernel(const uint64_t* buckets, int W, int B, int T, int seg_size,
                                                          uint64_t* seg_out) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)W * T) return;
    int w = (int)(t / T), seg = (int)(t % T);
    int lo = seg * seg_size;
    int hi = lo + seg_size < B ? lo + seg_size : B;
    XYZZ run = XYZZ::inf(), acc = XYZZ::inf();
    for (int b = hi - 1; b >= lo; --b) {
        XYZZ bk = ld_xyzz(buckets, (size_t)w * B + b);
        xyzz_add(run, bk);
        xyzz_add(acc, run);
    }
    // acc = sum (b - lo + 1) B_b ; add lo * run (double-and-add, lo < 2^23)
    if (lo && !run.is_inf()) {
        XYZZ m = XYZZ::inf();
        for (int bit = 23; bit >= 0; --bit) {
            xyzz_double(m);
            if ((lo >> bit) & 1) xyzz_add(m, run);
        }
        xyzz_add(acc, m);
    }
    st_xyzz(seg_out, t, acc);
}

// block-wide tree sum of XYZZ points through shared memory (word-major: conflict-free)
__device__ __forceinline__ void smem_put(uint32_t* sm, int tid, const XYZZ& p) {
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        sm[(0 * 8 + w) * 256 + tid] = p.x.v[w];
        sm[(1 * 8 + w) * 256 + tid] = p.y.v[w];
        sm[(2 * 8 + w) * 256 + tid] = p.zz.v[w];
        sm[(3 * 8 + w) * 256 + tid] = p.zzz.v[w];
    }
}
__device__ __forceinline__ XYZZ smem_get(const uint32_t* sm, int tid) {
    XYZZ p;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        p.x.v[w] = sm[(0 * 8 + w) * 256 + tid];
        p.y.v[w] = sm[(1 * 8 + w) * 256 + tid];
        p.zz.v[w] = sm[(2 * 8 + w) * 256 + tid];
        p.zzz.v[w] = sm[(3 * 8 + w) * 256 + tid];
    }
    return p;
}

// Buckets cut into more than MSM_MAX_CHUNKS chunks (small-scalar kinds only): one block per bucket, a
// strided pass over its partials and a shared-memory tree.
__global__ void __launch_bounds__(256) msm_combine_wide_kernel(const unsigned int* toff, const uint64_t* partial,
                                                               uint64_t* buckets) {
    __shared__ uint32_t sm[32 * 256];
    const size_t b = blockIdx.x;
    const int tid = threadIdx.x;
    const unsigned int t0 = toff[b], t1 = toff[b + 1];
    if (t1 - t0 <= MSM_MAX_CHUNKS) return;  // uniform over the block
    XYZZ acc = XYZZ::inf();
    for (unsigned int t = t0 + tid; t < t1; t += 256) xyzz_add(acc, ld_xyzz(partial, t));
    smem_put(sm, tid, acc);
    __syncthreads();
    for (int half = 128; half > 0; half >>= 1) {
        if (tid < half) {
            XYZZ o = smem_get(sm, tid + half);
            xyzz_add(acc, o);
            smem_put(sm, tid, acc);
        }
        __syncthreads();
    }
    if (tid == 0) st_xyzz(buckets, b, acc);
}

// ---- 6. per-window sum of the segment points: a multi-block tree (each block folds 2048 points of one
//         window into one), repeated until one point per window is left; then the 2^(c w) doublings ----
// in: [W][count] points, out: [W][gridDim.x] points
__global__ void __launch_bounds__(256) msm_tree_sum_kernel(const uint64_t* in, int count, uint64_t* out) {
    __shared__ uint32_t sm[32 * 256];
    const int w = blockIdx.y, tid = threadIdx.x;
    const size_t base = (size_t)w * count;
    XYZZ acc = XYZZ::inf();
    for (int k = blockIdx.x * 2048 + tid; k < count && k < (blockIdx.x + 1) * 2048; k += 256) xyzz_add(acc, ld_xyzz(in, base + k));
    smem_put(sm, tid, acc);
    __syncthreads();
    for (int half = 128; half > 0; half >>= 1) {
        if (tid < half) {
            XYZZ o = smem_get(sm, tid + half);
            xyzz_add(acc, o);
            smem_put(sm, tid, acc);
        }
        __syncthreads();
    }
    if (tid == 0) st_xyzz(out, (size_t)w * gridDim.x + blockIdx.x, acc);
}

// win[w] *= 2^(c w)   (one thread per window; absent on the shared-bucket path)
__global__ void __launch_bounds__(32) msm_window_shift_kernel(uint64_t* win, int W, int c) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W || w == 0) return;
    XYZZ acc = ld_xyzz(win, w);
    for (int k = 0; k < c * w; ++k) xyzz_double(acc);
    st_xyzz(win, w, acc);
}

// ---- 7. final: sum of the W window points -> Jacobian (X Z'^2-scaled): Z = ZZ*ZZZ ------------------------
__global__ void __launch_bounds__(32) msm_final_kernel(const uint64_t* win, int W, uint64_t* out_xyz) {
    __shared__ uint32_t sm[32 * 256];
    const int tid = threadIdx.x;
    XYZZ acc = XYZZ::inf();
    for (int k = tid; k < W; k += 32) xyzz_add(acc, ld_xyzz(win, k));  // W can reach 64 for small windows
    smem_put(sm, tid, acc);
    __syncwarp();
    for (int half = 16; half > 0; half >>= 1) {
        if (tid < half) {
            XYZZ o = smem_get(sm, tid + half);
            xyzz_add(acc, o);
            smem_put(sm, tid, acc);
        }
        __syncwarp();
    }
    if (tid == 0) {
        // x = X/ZZ, y = Y/ZZZ. With Z = ZZ*ZZZ: X_j = x Z^2 = X ZZ ZZZ^2, Y_j = y Z^3 = Y ZZ^3 ZZZ^2.
        Fq X, Y, Z;
        if (acc.is_inf()) {
            X = Fq::one();
            Y = Fq::one();
            Z = Fq::zero();
        } else {
            Fq zzz2 = fp_sqr(acc.zzz);
            Fq zz2 = fp_sqr(acc.zz);
            X = fp_mul(fp_mul(acc.x, acc.zz), zzz2);
            Y = fp_mul(fp_mul(acc.y, fp_mul(zz2, acc.zz)), zzz2);
            Z = fp_mul(acc.zz, acc.zzz);
        }
        st_elem(out_xyz, 0, X);
        st_elem(out_xyz, 1, Y);
        st_elem(out_xyz, 2, Z);
    }
}

// rows mode: every bucket set is one row's MSM; win[r] (XYZZ) -> Jacobian, one thread per row
__global__ void __launch_bounds__(128) msm_rows_out_kernel(const uint64_t* win, size_t rows, uint64_t* out_xyz) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const XYZZ acc = ld_xyzz(win, r);
    Fq X = Fq::one(), Y = Fq::one(), Z = Fq::zero();
    if (!acc.is_inf()) {
        Fq zzz2 = fp_sqr(acc.zzz);
        Fq zz2 = fp_sqr(acc.zz);
        X = fp_mul(fp_mul(acc.x, acc.zz), zzz2);
        Y = fp_mul(fp_mul(acc.y, fp_mul(zz2, acc.zz)), zzz2);
        Z = fp_mul(acc.zz, acc.zzz);
    }
    st_elem(out_xyz, 3 * r, X);
    st_elem(out_xyz, 3 * r + 1, Y);
    st_elem(out_xyz, 3 * r + 2, Z);
}

// ---- binary columns: msm_binary (the `all(s <= 1)` arm of VariableBaseMSM::msm / msm_u8,
//      crates/jolt-prover-legacy/src/msm/mod.rs:35-47, 96-106). The result is the plain sum of the selected bases: no
//      digits, no sort - every thread walks its own 16-flag groups and adds the selected bases into ONE XYZZ
//      accumulator (complete mixed additions: repeated / opposite bases are handled), then the existing tree folds
//      the per-thread partials. ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) u8_max_kernel(const uint8_t* v, size_t n, unsigned int* out_max) {
    const size_t T = (size_t)gridDim.x * blockDim.x, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned int m = 0;
    const size_t groups = n / 16;
    for (size_t g = t; g < groups; g += T) {
        const uint4 q = ((const uint4*)v)[g];
        m = __vmaxu4(m, __vmaxu4(__vmaxu4(q.x, q.y), __vmaxu4(q.z, q.w)));
    }
    for (size_t i = groups * 16 + t; i < n; i += T) m = __vmaxu4(m, (unsigned int)v[i]);
    m = max(max(m & 0xffu, (m >> 8) & 0xffu), max((m >> 16) & 0xffu, m >> 24));
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out_max, m);
}

__global__ void __launch_bounds__(128) msm_select_sum_kernel(const uint8_t* flags, const uint64_t* bases, size_t n,
                                                             uint64_t* partial) {
    const size_t T = (size_t)gridDim.x * blockDim.x, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    XYZZ acc = XYZZ::inf();
    const size_t groups = (n + 15) / 16;
    for (size_t g = t; g < groups; g += T) {
        const size_t i0 = g * 16;
        uint32_t mask = 0;
        if (i0 + 16 <= n) {
            const uint4 q = ((const uint4*)flags)[g];
            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                mask |= ((w[k] & 1u) | ((w[k] >> 7) & 2u) | ((w[k] >> 14) & 4u) | ((w[k] >> 21) & 8u)) << (4 * k);
        } else {
            for (size_t i = i0; i < n; ++i) mask |= (uint32_t)(flags[i] & 1u) << (i - i0);
        }
        while (mask) {
            const int j = __ffs(mask) - 1;
            mask &= mask - 1;
            const Fq px = ld_elem<Fq>(bases, 2 * (i0 + j)), py = ld_elem<Fq>(bases, 2 * (i0 + j) + 1);
            if (px.is_zero() && py.is_zero()) continue;  // identity base
            xyzz_add_affine(acc, px, py, false);
        }
    }
    st_xyzz(partial, t, acc);
}

// ---- SRS helpers ------------------------------------------------------------------------------------------
// Jacobian (X, Y, Z) -> affine (x, y) = (X/Z^2, Y/Z^3); Z == 0 -> identity (0, 0). One inversion per thread.
__global__ void __launch_bounds__(128) jacobian_to_affine_kernel(const uint64_t* xyz, size_t n, uint64_t* xy) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fq X = ld_elem<Fq>(xyz, 3 * i), Y = ld_elem<Fq>(xyz, 3 * i + 1), Z = ld_elem<Fq>(xyz, 3 * i + 2);
    Fq x = Fq::zero(), y = Fq::zero();
    if (!Z.is_zero()) {
        Fq zi = fq_inverse(Z);
        Fq zi2 = fp_sqr(zi);
        x = fp_mul(X, zi2);
        y = fp_mul(Y, fp_mul(zi2, zi));
    }
    st_elem(xy, 2 * i, x);
    st_elem(xy, 2 * i + 1, y);
}

// bases[i] = (i + 1) * base, affine. Each thread seeds (start + 1) * base by double-and-add, then
// walks GEN_RUN consecutive multiples; one Fermat inversion per emitted point (one-off SRS work).
constexpr int GEN_RUN = 32;
__global__ void __launch_bounds__(128) gen_multiples_kernel(const uint64_t* base_xy, size_t n, uint64_t* out_xy) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t start = t * GEN_RUN;
    if (start >= n) return;
    Fq bx = ld_elem_rw<Fq>(base_xy, 0), by = ld_elem_rw<Fq>(base_xy, 1);
    XYZZ acc = XYZZ::inf();
    uint64_t k = start + 1;
    for (int bit = 40; bit >= 0; --bit) {
        xyzz_double(acc);
        if ((k >> bit) & 1) xyzz_add_affine(acc, bx, by, false);
    }
    for (int j = 0; j < GEN_RUN && start + j < n; ++j) {
        Fq x = Fq::zero(), y = Fq::zero();
        if (!acc.is_inf()) {
            Fq i3 = fq_inverse(acc.zzz);
            Fq tz = fp_mul(acc.zz, i3);  // ZZ/ZZZ = 1/Z
            x = fp_mul(acc.x, fp_sqr(tz));
            y = fp_mul(acc.y, i3);
        }
        st_elem(out_xy, 2 * (start + j), x);
        st_elem(out_xy, 2 * (start + j) + 1, y);
        xyzz_add_affine(acc, bx, by, false);
    }
}

// table[w * n + i] = 2^(c w) * P_i (affine), w < W. One thread per base: c doublings per window in XYZZ,
// one Fermat inversion per emitted point (one-off SRS work, like the reference's setup).
__global__ void __launch_bounds__(128) precompute_windows_kernel(const uint64_t* xy, size_t n, int c, int W, uint64_t* table) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fq px = ld_elem<Fq>(xy, 2 * i), py = ld_elem<Fq>(xy, 2 * i + 1);
    st_elem(table, 2 * i, px);
    st_elem(table, 2 * i + 1, py);
    const bool inf = px.is_zero() && py.is_zero();
    XYZZ acc;
    acc.x = px;
    acc.y = py;
    acc.zz = inf ? Fq::zero() : Fq::one();
    acc.zzz = acc.zz;
    for (int w = 1; w < W; ++w) {
        for (int k = 0; k < c; ++k) xyzz_double(acc);
        Fq x = Fq::zero(), y = Fq::zero();
        if (!acc.is_inf()) {
            Fq i3 = fq_inverse(acc.zzz);
            Fq tz = fp_mul(acc.zz, i3);
            x = fp_mul(acc.x, fp_sqr(tz));
            y = fp_mul(acc.y, i3);
        }
        st_elem(table, 2 * ((size_t)w * n + i), x);
        st_elem(table, 2 * ((size_t)w * n + i) + 1, y);
    }
}

// out = sum of `count` Jacobian points (X, Y, Z; Z == 0 is the identity) -> Jacobian. One warp.
__global__ void __launch_bounds__(32) jacobian_sum_kernel(const uint64_t* pts, int count, uint64_t* out_xyz) {
    __shared__ uint32_t sm[32 * 256];
    const int tid = threadIdx.x;
    XYZZ acc = XYZZ::inf();
    for (int k = tid; k < count; k += 32) {
        Fq X = ld_elem_rw<Fq>(pts, 3 * (size_t)k), Y = ld_elem_rw<Fq>(pts, 3 * (size_t)k + 1), Z = ld_elem_rw<Fq>(pts, 3 * (size_t)k + 2);
        if (Z.is_zero()) continue;
        XYZZ p;  // (X, Y, Z) Jacobian == (X, Y, Z^2, Z^3) XYZZ
        p.x = X;
        p.y = Y;
        p.zz = fp_sqr(Z);
        p.zzz = fp_mul(p.zz, Z);
        xyzz_add(acc, p);
    }
    smem_put(sm, tid, acc);
    __syncwarp();
    for (int half = 16; half > 0; half >>= 1) {
        if (tid < half) {
            XYZZ o = smem_get(sm, tid + half);
            xyzz_add(acc, o);
            smem_put(sm, tid, acc);
        }
        __syncwarp();
    }
    if (tid == 0) {
        Fq X = Fq::one(), Y = Fq::one(), Z = Fq::zero();
        if (!acc.is_inf()) {
            Fq zzz2 = fp_sqr(acc.zzz), zz2 = fp_sqr(acc.zz);
            X = fp_mul(fp_mul(acc.x, acc.zz), zzz2);
            Y = fp_mul(fp_mul(acc.y, fp_mul(zz2, acc.zz)), zzz2);
            Z = fp_mul(acc.zz, acc.zzz);
        }
        st_elem(out_xyz, 0, X);
        st_elem(out_xyz, 1, Y);
        st_elem(out_xyz, 2, Z);
    }
}

bool canonical_q(const uint64_t* a) {
    static const uint64_t Q[4] = {0x3c208c16d87cfd47ULL, 0x97816a916871ca8dULL, 0xb85045b68181585dULL,
                                  0x30644e72e131a029ULL};
    for (int i = 3; i >= 0; --i)
        if (a[i] != Q[i]) return a[i] < Q[i];
    return false;
}

using Guard = CtxGuard;

// `srs`: the resident bases; terms are bases[offset .. offset + n).
// rows > 1 (jb_msm_g1_rows): n = rows * row_w terms, row r = scalars[r * row_w ..) against bases[0 .. row_w); the
// small table (8-bit shared windows) must cover row_w; out_xyz receives rows x 12 limbs.
// halving = h > 0: the rows are the h - 1 packed polynomials of lengths 2^(h-1) .. 2 (n = 2^h - 2, rows = h - 1).
int msm_device(jb_ctx* c, const Srs& srs, size_t offset, const void* d_scalars, size_t n, uint64_t* out_xyz,
               int kind = SK_FR, size_t rows = 1, int halving = 0) {
    const int bits = small_kind_bits(kind);
    const bool by_rows = rows > 1;
    const size_t row_w = by_rows && !halving ? n / rows : 0;
    // (a row's bucket holds at most row_w * W points: 64 chunks bound the walk without the block-per-bucket pass)
    // (128-point chunks only where there is parallelism to spare: a 4096-term MSM over the 128-bucket table wants
    // its 2048 short tasks, not 1024 long ones)
    const unsigned maxq = (kind == SK_FR || by_rows) ? (MSM_MAX_CHUNKS | (kind == SK_FR && !by_rows && n >= ((size_t)1 << 18) ? 7u << 16 : 0u))
                                                     : MSM_MAX_CHUNKS_SMALL;
    // shared-bucket path when the SRS carries precomputed windows and the MSM is large enough for the
    // wide window's bucket reduction (2^(c-1) buckets) to be in the noise
    // Small MSMs (the tail of HyperKZG's intermediate commitments, verifier-sized MSMs) use a second, tiny
    // table with 8-bit windows over the first bases: 128 buckets, no doubling chain - latency, not work.
    constexpr size_t small_max = 4096;  // largest MSM served by the 8-bit-window table
    const bool use_small = by_rows || (srs.pre_small != nullptr && n <= small_max && offset + n <= srs.pre_small_len);
    const bool use_big = !use_small && srs.pre != nullptr && n >= ((size_t)1 << (srs.pre_c - 4));
    const bool shared = use_small || use_big;
    const MsmPlan p = use_small ? plan_with(8, bits) : use_big ? plan_with(srs.pre_c, bits) : plan_for(n, bits);
    const size_t pre_stride = use_small ? srs.pre_small_len : srs.n;       // row w starts at w * stride
    const uint64_t* d_bases = srs.xy + 8 * offset;                          // digits: identity test, per-window path: gather
    const uint64_t* d_gather = use_small ? srs.pre_small + 8 * offset : use_big ? srs.pre + 8 * offset : d_bases;
    const int Weff = by_rows ? (int)rows : shared ? 1 : p.W;  // bucket sets
    const size_t nb = (size_t)Weff * p.B;
    // bucket offsets, task offsets, the scatter cursor and the histogram are 32-bit: W * n sorted entries must stay
    // below 2^32 (n ~ 2^28 with 16 windows would wrap the exclusive scan and read wrong ranges - silently)
    const size_t entries = (size_t)p.W * n;
    if (entries >= ((size_t)1 << 32) || nb + entries / MSM_CHUNK + 1 >= ((size_t)1 << 32))
        return c->fail(JB_ERR_UNSUPPORTED, "msm: windows x terms must be < 2^32 (split the call)");
    // upper bound on tasks: every bucket at most cnt/MSM_CHUNK + 1 chunks
    const size_t max_tasks = nb + entries / MSM_CHUNK + 1;
    uint32_t *digits = nullptr, *sorted = nullptr, *task_bucket = nullptr, *order = nullptr;
    unsigned int* len_hist = nullptr;
    unsigned int *hist = nullptr, *offsets = nullptr, *toff = nullptr, *block_sums = nullptr;
    const unsigned scan_blocks = (unsigned)((nb + SCAN_PER_BLOCK - 1) / SCAN_PER_BLOCK);  // <= 512 (c <= 22)
    uint64_t *buckets = nullptr, *partial = nullptr, *seg = nullptr, *win = nullptr, *d_out = nullptr;
    uint64_t *tree_a = nullptr, *tree_b = nullptr;
    const size_t tree_pts = (size_t)Weff * ((p.T + 2047) / 2048) + 1;
    int st = c->dev_alloc((void**)&digits, (size_t)p.W * n * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&sorted, entries * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&hist, nb * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&offsets, (nb + 1) * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&toff, (nb + 1) * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&block_sums, 2 * 1024 * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&task_bucket, max_tasks * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&order, max_tasks * 4);
    if (st == JB_OK) st = c->dev_alloc((void**)&len_hist, 2 * MSM_LEN_BINS * 4);
    if (st == JB_OK) st = c->check(cudaMemsetAsync(len_hist, 0, 2 * MSM_LEN_BINS * 4, c->stream), "msm memset");
    if (st == JB_OK) st = c->dev_alloc((void**)&buckets, nb * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&partial, max_tasks * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&seg, (size_t)Weff * p.T * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&win, (size_t)Weff * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&tree_a, tree_pts * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&tree_b, tree_pts * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&d_out, 96 * rows);
    if (st == JB_OK) st = c->check(cudaMemsetAsync(hist, 0, nb * 4, c->stream), "msm memset");
    if (st == JB_OK) {
        unsigned g = (unsigned)((n + 255) / 256);
        const bool agg = kind != SK_FR;
        if (agg)
            msm_digits_kernel<true><<<g, 256, 0, c->stream>>>(d_scalars, kind, d_bases, n, p.c, p.W, p.B, shared ? 1 : 0, digits, hist, row_w, halving);
        else
            msm_digits_kernel<false><<<g, 256, 0, c->stream>>>(d_scalars, kind, d_bases, n, p.c, p.W, p.B, shared ? 1 : 0, digits, hist, row_w, halving);
        msm_scan_local_kernel<<<scan_blocks, 1024, 0, c->stream>>>(hist, offsets, toff, nb, block_sums, maxq);
        msm_scan_blocks_kernel<<<1, 1024, 0, c->stream>>>(block_sums, (int)scan_blocks, offsets, toff, nb);
        msm_scan_apply_kernel<<<scan_blocks, 1024, 0, c->stream>>>(offsets, toff, nb, block_sums);
        {   // scatter, ordered in time by destination region once the destination outgrows the L2 (see the kernel)
            int mode = 0, regions = 1;
            unsigned range_shift = 0;
            if (!by_rows && entries >= ((size_t)1 << 25)) {
                if (!shared) {
                    mode = 1;
                    regions = p.W;
                } else if (p.c - 1 >= 6) {
                    mode = 2;
                    const int rl = 2;  // log2(regions); measured at 2^24 terms, 12 windows: 1 / 2 / 4 / 8 / 16 regions = 41.7 / 40.5 / 39.2 / 40.6 / 44.8 ms per MSM
                    regions = 1 << rl;
                    range_shift = (unsigned)(p.c - 1) - (unsigned)rl;  // nb = 2^(c-1) buckets
                }
            }
            const dim3 sg(g, (unsigned)regions);
            if (agg)
                msm_scatter_kernel<true><<<sg, 256, 0, c->stream>>>(digits, n, p.W, p.B, shared ? 1 : 0, pre_stride, offsets, hist, sorted, row_w, halving, mode, range_shift);
            else
                msm_scatter_kernel<false><<<sg, 256, 0, c->stream>>>(digits, n, p.W, p.B, shared ? 1 : 0, pre_stride, offsets, hist, sorted, row_w, halving, mode, range_shift);
        }
        int tix = c->timing_begin(4, n, p.c);  // (window bits) for the bench's roofline
        msm_len_hist_kernel<<<MSM_TASK_BLOCKS, 256, 0, c->stream>>>(offsets, toff, nb, maxq, len_hist);
        msm_tasks_kernel<<<MSM_TASK_BLOCKS, 256, 0, c->stream>>>(offsets, toff, nb, maxq, len_hist, task_bucket, order);
        c->launches++;
        msm_accumulate_kernel<<<(unsigned)((max_tasks + 127) / 128), 128, 0, c->stream>>>(d_gather, sorted, offsets, toff, task_bucket,
                                                                                          order, nb, buckets, partial, maxq);
        c->timing_end(tix);
        msm_combine_kernel<<<(unsigned)((nb + 127) / 128), 128, 0, c->stream>>>(toff, nb, partial, buckets);
        if (plan_cap(maxq) > MSM_MAX_CHUNKS) {
            msm_combine_wide_kernel<<<(unsigned)nb, 256, 0, c->stream>>>(toff, partial, buckets);
            c->launches++;
        }
        msm_segment_kernel<<<(unsigned)(((size_t)Weff * p.T + 127) / 128), 128, 0, c->stream>>>(buckets, Weff, p.B, p.T, msm_seg_size(p.B), seg);
        {   // tree-sum the T segment points of every bucket set, ping-ponging between two scratch buffers
            const uint64_t* src = seg;
            int count = p.T;
            uint64_t* dst = count > 2048 ? tree_a : win;
            while (true) {
                const int blocks = (count + 2047) / 2048;
                msm_tree_sum_kernel<<<dim3(blocks, Weff), 256, 0, c->stream>>>(src, count, blocks == 1 ? win : dst);
                c->launches++;
                if (blocks == 1) break;
                src = dst;
                count = blocks;
                dst = (dst == tree_a) ? tree_b : tree_a;
            }
            if (!shared) {
                msm_window_shift_kernel<<<(Weff + 31) / 32, 32, 0, c->stream>>>(win, Weff, p.c);
                c->launches++;
            }
        }
        if (by_rows) msm_rows_out_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, c->stream>>>(win, rows, d_out);
        else msm_final_kernel<<<1, 32, 0, c->stream>>>(win, Weff, d_out);
        c->launches += 10;
        st = c->check(cudaGetLastError(), "msm kernels");
    }
    if (by_rows) {
        if (st == JB_OK) st = c->check(cudaMemcpyAsync(out_xyz, d_out, 96 * rows, cudaMemcpyDeviceToHost, c->stream), "msm rows D2H");
        if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "msm sync");
    } else {
        if (st == JB_OK) st = c->check(cudaMemcpyAsync(c->h_small, d_out, 96, cudaMemcpyDeviceToHost, c->stream), "msm D2H");
        if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "msm sync");
        if (st == JB_OK) std::memcpy(out_xyz, c->h_small, 96);
    }
    c->dev_free(digits);
    c->dev_free(sorted);
    c->dev_free(task_bucket);
    c->dev_free(order);
    c->dev_free(len_hist);
    c->dev_free(hist);
    c->dev_free(offsets);
    c->dev_free(toff);
    c->dev_free(block_sums);
    c->dev_free(buckets);
    c->dev_free(partial);
    c->dev_free(seg);
    c->dev_free(win);
    c->dev_free(tree_a);
    c->dev_free(tree_b);
    c->dev_free(d_out);
    return st;
}

// The small-MSM table: 8-bit shared windows (2^(8 w) * P_i, 32 rows) over the first bases - at least `want` of them,
// by default the first <= 2^15 (<= 66 MiB). Serves MSMs of <= 4096 terms (the tail of a HyperKZG open) and the
// row-batched MSMs of jb_msm_g1_rows.
int build_small_table(jb_ctx* c, Srs& s, size_t want) {
    const MsmPlan ps = plan_with(8);
    size_t small_len = s.n < ((size_t)1 << 15) ? s.n : ((size_t)1 << 15);
    if (want > small_len) small_len = want;
    if (small_len > s.n) small_len = s.n;
    if (s.pre_small && s.pre_small_len >= small_len) return JB_OK;
    uint64_t* tab = nullptr;
    int st = c->dev_alloc((void**)&tab, (size_t)ps.W * small_len * 64);
    if (st != JB_OK) return st;
    precompute_windows_kernel<<<(unsigned)((small_len + 127) / 128), 128, 0, c->stream>>>(s.xy, small_len, ps.c, ps.W, tab);
    c->launches++;
    st = c->check(cudaGetLastError(), "precompute_windows (small) launch");
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "precompute sync");
    if (st != JB_OK) {
        c->dev_free(tab);
        return st;
    }
    if (s.pre_small) c->dev_free(s.pre_small);
    s.pre_small = tab;
    s.pre_small_len = small_len;
    return JB_OK;
}

void identity_xyz(uint64_t out[12]);

// msm_binary on the device: `d_flags` = n bytes (0 / 1) already resident. Returns the Jacobian sum of the selected bases.
int msm_binary_device(jb_ctx* c, const Srs& srs, size_t offset, const uint8_t* d_flags, size_t n, uint64_t out_xyz[12]) {
    const unsigned blocks = 148 * 8;  // 1184 blocks x 128 threads: every thread owns ~n / 2^17 groups
    const size_t T = (size_t)blocks * 128;
    uint64_t *partial = nullptr, *tree_a = nullptr, *tree_b = nullptr, *d_out = nullptr;
    int st = c->dev_alloc((void**)&partial, T * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&tree_a, ((T + 2047) / 2048 + 1) * 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&tree_b, 128);
    if (st == JB_OK) st = c->dev_alloc((void**)&d_out, 96);
    if (st == JB_OK) {
        int tix = c->timing_begin(4, n, 1);
        msm_select_sum_kernel<<<blocks, 128, 0, c->stream>>>(d_flags, srs.xy + 8 * offset, n, partial);
        c->timing_end(tix);
        const int b1 = (int)((T + 2047) / 2048);
        msm_tree_sum_kernel<<<dim3(b1, 1), 256, 0, c->stream>>>(partial, (int)T, tree_a);
        msm_tree_sum_kernel<<<dim3(1, 1), 256, 0, c->stream>>>(tree_a, b1, tree_b);  // b1 = 74 <= 2048
        msm_final_kernel<<<1, 32, 0, c->stream>>>(tree_b, 1, d_out);
        c->launches += 4;
        st = c->check(cudaGetLastError(), "msm_binary kernels");
    }
    if (st == JB_OK) st = c->check(cudaMemcpyAsync(c->h_small, d_out, 96, cudaMemcpyDeviceToHost, c->stream), "msm D2H");
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "msm sync");
    if (st == JB_OK) std::memcpy(out_xyz, c->h_small, 96);
    c->dev_free(partial);
    c->dev_free(tree_a);
    c->dev_free(tree_b);
    c->dev_free(d_out);
    return st;
}

void identity_xyz(uint64_t out[12]) {
    // Montgomery one for X and Y, Z = 0 (G1Projective::zero() is (1, 1, 0))
    static const uint64_t ONE_Q[4] = {0xd35d438dc58f0d9dULL, 0x0a78eb28f5c70b3dULL, 0x666ea36f7879462cULL,
                                      0x0e0a77c19a07df2fULL};
    std::memcpy(out, ONE_Q, 32);
    std::memcpy(out + 4, ONE_Q, 32);
    std::memset(out + 8, 0, 32);
}

}  // namespace

void jb_ctx::msm_release() {}

// HyperKZG open (hyperkzg.cu): the commitments of the h - 1 folded polynomials of lengths 2^(h-1) .. 2, packed back to
// back on the device, in ONE pass of the pipeline over (polynomial, bucket) sets of the 8-bit-window table (the tail of an
// open is 15 MSMs of <= 2^15 terms: launch latency, not work). Returns JB_ERR_UNSUPPORTED when the SRS has no small table
// covering 2^(h-1) bases (the caller then commits them one by one). out_xyz: (h - 1) x 12 limbs.
int jb::msm_halving_rows_device(jb_ctx* c, jb_srs h_srs, const uint64_t* d_scalars, int h, uint64_t* out_xyz) {
    if (!c || !d_scalars || !out_xyz || h < 3 || h > 20) return JB_ERR_UNSUPPORTED;
    Guard g(c);
    auto it = c->srs.find(h_srs);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    const Srs& srs = it->second;
    if (!srs.pre_small || srs.pre_small_len < ((size_t)1 << (h - 1))) return JB_ERR_UNSUPPORTED;
    return msm_device(c, srs, 0, d_scalars, ((size_t)1 << h) - 2, out_xyz, SK_FR, (size_t)(h - 1), h);
}

extern "C" {

int jb_srs_upload_affine(jb_ctx* c, const uint64_t* xy, size_t n, jb_srs* out) {
    if (!c || !out || (n && !xy)) return JB_ERR_INVALID;
    Guard g(c);
    for (size_t i = 0; i < n * 2; ++i)
        if (!canonical_q(xy + 4 * i)) return c->fail(JB_ERR_INVALID, "srs: coordinate limbs not canonical (>= q)");
    Srs s;
    s.n = n;
    int st = c->dev_alloc((void**)&s.xy, (n ? n : 1) * 64);
    if (st != JB_OK) return st;
    if (n) {
        st = c->check(cudaMemcpyAsync(s.xy, xy, n * 64, cudaMemcpyHostToDevice, c->stream), "srs H2D");
        if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "srs H2D sync");
        if (st != JB_OK) {
            c->dev_free(s.xy);
            return st;
        }
    }
    *out = c->next_id++;
    c->srs[*out] = s;
    return JB_OK;
}

int jb_srs_upload_jacobian(jb_ctx* c, const uint64_t* xyz, size_t n, jb_srs* out) {
    if (!c || !out || (n && !xyz)) return JB_ERR_INVALID;
    Guard g(c);
    for (size_t i = 0; i < n * 3; ++i)
        if (!canonical_q(xyz + 4 * i)) return c->fail(JB_ERR_INVALID, "srs: coordinate limbs not canonical (>= q)");
    Srs s;
    s.n = n;
    uint64_t* d_xyz = nullptr;
    int st = c->dev_alloc((void**)&s.xy, (n ? n : 1) * 64);
    if (st != JB_OK) return st;
    if (n) {
        st = c->dev_alloc((void**)&d_xyz, n * 96);
        if (st == JB_OK) st = c->check(cudaMemcpyAsync(d_xyz, xyz, n * 96, cudaMemcpyHostToDevice, c->stream), "srs H2D");
        if (st == JB_OK) {
            jacobian_to_affine_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(d_xyz, n, s.xy);
            c->launches++;
            st = c->check(cudaGetLastError(), "jacobian_to_affine launch");
        }
        if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "srs sync");
        if (d_xyz) c->dev_free(d_xyz);
        if (st != JB_OK) {
            c->dev_free(s.xy);
            return st;
        }
    }
    *out = c->next_id++;
    c->srs[*out] = s;
    return JB_OK;
}

int jb_srs_generate_multiples(jb_ctx* c, const uint64_t base_xy[8], size_t n, jb_srs* out) {
    if (!c || !out || !base_xy || n == 0) return JB_ERR_INVALID;
    Guard g(c);
    if (!canonical_q(base_xy) || !canonical_q(base_xy + 4)) return c->fail(JB_ERR_INVALID, "srs: base limbs not canonical");
    Srs s;
    s.n = n;
    uint64_t* d_base = nullptr;
    int st = c->dev_alloc((void**)&s.xy, n * 64);
    if (st == JB_OK) st = c->dev_alloc((void**)&d_base, 64);
    if (st == JB_OK) st = c->check(cudaMemcpyAsync(d_base, base_xy, 64, cudaMemcpyHostToDevice, c->stream), "srs base H2D");
    if (st == JB_OK) {
        size_t threads = (n + GEN_RUN - 1) / GEN_RUN;
        gen_multiples_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, c->stream>>>(d_base, n, s.xy);
        c->launches++;
        st = c->check(cudaGetLastError(), "gen_multiples launch");
    }
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "srs generate sync");
    if (d_base) c->dev_free(d_base);
    if (st != JB_OK) {
        if (s.xy) c->dev_free(s.xy);
        return st;
    }
    *out = c->next_id++;
    c->srs[*out] = s;
    return JB_OK;
}

int jb_srs_precompute(jb_ctx* c, jb_srs h, int window_bits) {
    if (!c) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    Srs& s = it->second;
    if (s.pre) return JB_OK;
    if (s.n == 0) return c->fail(JB_ERR_INVALID, "srs precompute: empty srs");
    const int cbits = window_bits > 0 ? window_bits : shared_window_for(s.n);
    if (cbits < 8 || cbits > 24) return c->fail(JB_ERR_INVALID, "srs precompute: window bits must be in 8..24");
    const MsmPlan p = plan_with(cbits);
    if ((size_t)p.W * s.n >= ((size_t)1 << 31)) return c->fail(JB_ERR_UNSUPPORTED, "srs precompute: windows * bases must be < 2^31");
    int st = c->dev_alloc((void**)&s.pre, (size_t)p.W * s.n * 64);
    if (st != JB_OK) return st;  // JB_ERR_OOM: the caller keeps the plain per-window path
    precompute_windows_kernel<<<(unsigned)((s.n + 127) / 128), 128, 0, c->stream>>>(s.xy, s.n, p.c, p.W, s.pre);
    c->launches++;
    st = c->check(cudaGetLastError(), "precompute_windows launch");
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "precompute sync");
    if (st != JB_OK) {
        c->dev_free(s.pre);
        s.pre = nullptr;
        return st;
    }
    s.pre_c = p.c;
    s.pre_W = p.W;
    build_small_table(c, s, 0);  // optional: the plain path stays without it
    return JB_OK;
}

int jb_srs_len(jb_ctx* c, jb_srs h, size_t* n) {
    if (!c || !n) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    *n = it->second.n;
    return JB_OK;
}

int jb_srs_download_affine(jb_ctx* c, jb_srs h, uint64_t* out_xy, size_t n) {
    if (!c || !out_xy) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    if (n > it->second.n) return c->fail(JB_ERR_INVALID, "srs download: n exceeds length");
    int st = c->check(cudaMemcpyAsync(out_xy, it->second.xy, n * 64, cudaMemcpyDeviceToHost, c->stream), "srs D2H");
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "srs D2H sync");
    return st;
}

int jb_srs_free(jb_ctx* c, jb_srs h) {
    if (!c) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    c->dev_free(it->second.xy);
    if (it->second.pre) c->dev_free(it->second.pre);
    if (it->second.pre_small) c->dev_free(it->second.pre_small);
    c->srs.erase(it);
    return JB_OK;
}

int jb_msm_g1(jb_ctx* c, jb_srs h, size_t offset, const uint64_t* scalars, size_t n, uint64_t out_xyz[12]) {
    if (!c || !out_xyz || (n && !scalars)) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    if (offset + n > it->second.n) return c->fail(JB_ERR_LENGTH, "msm: bases/scalars length mismatch");
    if (n == 0) {
        identity_xyz(out_xyz);
        return JB_OK;
    }
    if (n >= ((size_t)1 << 31)) return c->fail(JB_ERR_UNSUPPORTED, "msm: n must be < 2^31");
    uint64_t* d_s = nullptr;
    int st = c->dev_alloc((void**)&d_s, n * 32);
    if (st != JB_OK) return st;
    st = c->check(cudaMemcpyAsync(d_s, scalars, n * 32, cudaMemcpyHostToDevice, c->stream), "msm scalars H2D");
    if (st == JB_OK) st = msm_device(c, it->second, offset, d_s, n, out_xyz);
    c->dev_free(d_s);
    return st;
}

int jb_msm_g1_small(jb_ctx* c, jb_srs h, size_t offset, const void* scalars, size_t n, int kind, uint64_t out_xyz[12]) {
    if (!c || !out_xyz || (n && !scalars)) return JB_ERR_INVALID;
    if (kind < SK_U8 || kind > SK_LAST) return c->fail(JB_ERR_INVALID, "msm_small: unknown scalar kind");
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    if (offset + n > it->second.n) return c->fail(JB_ERR_LENGTH, "msm: bases/scalars length mismatch");
    if (n == 0) {
        identity_xyz(out_xyz);
        return JB_OK;
    }
    if (n >= ((size_t)1 << 31)) return c->fail(JB_ERR_UNSUPPORTED, "msm: n must be < 2^31");
    void* d_s = nullptr;
    const size_t bytes = n * (size_t)small_kind_bytes(kind);
    int st = c->dev_alloc(&d_s, bytes);
    if (st != JB_OK) return st;
    st = c->check(cudaMemcpyAsync(d_s, scalars, bytes, cudaMemcpyHostToDevice, c->stream), "msm small scalars H2D");
    // The reference's dispatch for u8 / bool columns (msm/mod.rs:35-47, 96-106): all zero -> identity, all <= 1 ->
    // msm_binary, else msm_u8. One pass over the bytes decides (the reference's par_iter().all()); below 2^14 terms
    // the general path is launch-latency either way.
    unsigned int vmax = 2;
    if (st == JB_OK && kind == SK_U8 && n >= ((size_t)1 << 14)) {
        unsigned int* d_max = nullptr;
        st = c->dev_alloc((void**)&d_max, 4);
        if (st == JB_OK) st = c->check(cudaMemsetAsync(d_max, 0, 4, c->stream), "msm max memset");
        if (st == JB_OK) {
            u8_max_kernel<<<148 * 4, 256, 0, c->stream>>>((const uint8_t*)d_s, n, d_max);
            c->launches++;
            st = c->check(cudaMemcpyAsync(c->h_small, d_max, 4, cudaMemcpyDeviceToHost, c->stream), "msm max D2H");
        }
        if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "msm max sync");
        if (st == JB_OK) std::memcpy(&vmax, c->h_small, 4);
        if (d_max) c->dev_free(d_max);
    }
    if (st == JB_OK) {
        if (vmax == 0) identity_xyz(out_xyz);
        else if (vmax == 1) st = msm_binary_device(c, it->second, offset, (const uint8_t*)d_s, n, out_xyz);
        else st = msm_device(c, it->second, offset, d_s, n, out_xyz, kind);
    }
    c->dev_free(d_s);
    return st;
}

int jb_msm_g1_batch(jb_ctx* c, jb_srs h, size_t count, const void* const* scalars, const size_t* lens, const int* kinds,
                    uint64_t* out_xyz) {
    if (!c || (count && (!scalars || !lens || !kinds || !out_xyz))) return JB_ERR_INVALID;
    size_t srs_n = 0;
    {
        Guard g(c);
        auto it = c->srs.find(h);
        if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
        srs_n = it->second.n;
        for (size_t k = 0; k < count; ++k) {
            if (kinds[k] < SK_FR || kinds[k] > SK_LAST) return c->fail(JB_ERR_INVALID, "batch_msm: unknown scalar kind");
            if (lens[k] > srs_n) return c->fail(JB_ERR_LENGTH, "batch_msm: a column is longer than the base set");
            if (lens[k] && !scalars[k]) return c->fail(JB_ERR_INVALID, "batch_msm: null column");
        }
    }
    for (size_t k = 0; k < count; ++k) {
        const int st = kinds[k] == SK_FR ? jb_msm_g1(c, h, 0, (const uint64_t*)scalars[k], lens[k], out_xyz + 12 * k)
                                         : jb_msm_g1_small(c, h, 0, scalars[k], lens[k], kinds[k], out_xyz + 12 * k);
        if (st != JB_OK) return st;
    }
    return JB_OK;
}

int jb_msm_g1_rows(jb_ctx* c, jb_srs h, const void* scalars, size_t rows, size_t row_width, int kind, uint64_t* out_xyz) {
    if (!c || (rows && row_width && (!scalars || !out_xyz)) || (rows && !out_xyz)) return JB_ERR_INVALID;
    if (kind < SK_FR || kind > SK_LAST) return c->fail(JB_ERR_INVALID, "msm_rows: unknown scalar kind");
    if (rows == 0) return JB_OK;
    if (row_width == 0) {
        for (size_t r = 0; r < rows; ++r) identity_xyz(out_xyz + 12 * r);
        return JB_OK;
    }
    const size_t esz = kind == SK_FR ? 32 : (size_t)small_kind_bytes(kind);
    if (rows == 1)
        return kind == SK_FR ? jb_msm_g1(c, h, 0, (const uint64_t*)scalars, row_width, out_xyz)
                             : jb_msm_g1_small(c, h, 0, scalars, row_width, kind, out_xyz);
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    if (row_width > it->second.n) return c->fail(JB_ERR_LENGTH, "msm: bases/scalars length mismatch");
    int st = build_small_table(c, it->second, row_width);
    if (st != JB_OK) return st;
    // rows per pass: 32-bit offsets (entries < 2^28 keeps the workspace near 2 GiB) and <= 4 Mi histogram counters
    const MsmPlan p = plan_with(8, small_kind_bits(kind));
    size_t per = ((size_t)1 << 28) / ((size_t)p.W * row_width);
    if (per > 32768) per = 32768;
    if (per < 2) per = 2;
    if ((size_t)p.W * row_width * per >= ((size_t)1 << 31)) return c->fail(JB_ERR_UNSUPPORTED, "msm_rows: row too wide (use jb_msm_g1_batch)");
    for (size_t r0 = 0; r0 < rows && st == JB_OK; r0 += per) {
        size_t cnt = rows - r0 < per ? rows - r0 : per;
        const char* src = (const char*)scalars + r0 * row_width * esz;
        if (cnt == 1) {  // a lone last row: the single-MSM path (by_rows needs >= 2 rows)
            void* d1 = nullptr;
            st = c->dev_alloc(&d1, row_width * esz);
            if (st == JB_OK) st = c->check(cudaMemcpyAsync(d1, src, row_width * esz, cudaMemcpyHostToDevice, c->stream), "msm rows H2D");
            if (st == JB_OK) st = msm_device(c, it->second, 0, d1, row_width, out_xyz + 12 * r0, kind);
            if (d1) c->dev_free(d1);
            continue;
        }
        void* d_s = nullptr;
        st = c->dev_alloc(&d_s, cnt * row_width * esz);
        if (st == JB_OK) st = c->check(cudaMemcpyAsync(d_s, src, cnt * row_width * esz, cudaMemcpyHostToDevice, c->stream), "msm rows H2D");
        if (st == JB_OK) st = msm_device(c, it->second, 0, d_s, cnt * row_width, out_xyz + 12 * r0, kind, cnt);
        if (d_s) c->dev_free(d_s);
    }
    return st;
}

int jb_msm_g1_device(jb_ctx* c, jb_srs h, size_t offset, const uint64_t* d_scalars, size_t n, uint64_t out_xyz[12]) {
    if (!c || !out_xyz || (n && !d_scalars)) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    if (offset + n > it->second.n) return c->fail(JB_ERR_LENGTH, "msm: bases/scalars length mismatch");
    if (n == 0) {
        identity_xyz(out_xyz);
        return JB_OK;
    }
    if (n >= ((size_t)1 << 31)) return c->fail(JB_ERR_UNSUPPORTED, "msm: n must be < 2^31");
    return msm_device(c, it->second, offset, d_scalars, n, out_xyz);
}

// Multi-GPU MSM (SURVEY 8e): the terms are partitioned across ranks (each rank holds its own bases and
// scalars), every rank runs a full Pippenger on its share, ONE all-gather moves the G partial points
// (96 B each - EC addition is not an NCCL reduction) and every rank adds them. Same value on all ranks.
int jb_msm_g1_sharded(jb_ctx* c, jb_srs h, size_t offset, const uint64_t* scalars, size_t n, uint64_t out_xyz[12]) {
    if (!c || !out_xyz) return JB_ERR_INVALID;
    if (!c->nccl_comm) return c->fail(JB_ERR_INVALID, "sharded msm: no communicator (jb_comm_init)");
    uint64_t local[12];
    int st = jb_msm_g1(c, h, offset, scalars, n, local);
    if (st != JB_OK) return st;
    Guard g(c);
    uint64_t *d_mine = nullptr, *d_all = nullptr, *d_out = nullptr;
    st = c->dev_alloc((void**)&d_mine, 96);
    if (st == JB_OK) st = c->dev_alloc((void**)&d_all, 96 * (size_t)c->world);
    if (st == JB_OK) st = c->dev_alloc((void**)&d_out, 96);
    std::memcpy(c->h_small, local, 96);
    if (st == JB_OK) st = c->check(cudaMemcpyAsync(d_mine, c->h_small, 96, cudaMemcpyHostToDevice, c->stream), "sharded msm H2D");
    if (st == JB_OK) st = c->comm_allgather(d_mine, d_all, 12);
    if (st == JB_OK) {
        jacobian_sum_kernel<<<1, 32, 0, c->stream>>>(d_all, c->world, d_out);
        c->launches++;
        st = c->check(cudaGetLastError(), "jacobian_sum launch");
    }
    if (st == JB_OK) st = c->check(cudaMemcpyAsync(c->h_small, d_out, 96, cudaMemcpyDeviceToHost, c->stream), "sharded msm D2H");
    if (st == JB_OK) st = c->check(cudaStreamSynchronize(c->stream), "sharded msm sync");
    if (st == JB_OK) std::memcpy(out_xyz, c->h_small, 96);
    c->dev_free(d_mine);
    c->dev_free(d_all);
    c->dev_free(d_out);
    return st;
}

int jb_msm_g1_table(jb_ctx* c, jb_srs h, size_t offset, jb_table scalars, size_t n, uint64_t out_xyz[12]) {
    if (!c || !out_xyz) return JB_ERR_INVALID;
    Guard g(c);
    auto it = c->srs.find(h);
    if (it == c->srs.end()) return c->fail(JB_ERR_INVALID, "unknown srs handle");
    Table* t = c->find(scalars);
    if (!t) return c->fail(JB_ERR_INVALID, "unknown table handle");
    if (n > t->len || offset + n > it->second.n) return c->fail(JB_ERR_LENGTH, "msm: bases/scalars length mismatch");
    if (n == 0) {
        identity_xyz(out_xyz);
        return JB_OK;
    }
    if (n >= ((size_t)1 << 31)) return c->fail(JB_ERR_UNSUPPORTED, "msm: n must be < 2^31");
    return msm_device(c, it->second, offset, t->buf, n, out_xyz);
}

}  // extern "C"
