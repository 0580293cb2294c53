// runs.cuh -- frame-dedup fast path of the input projection and its weight gradient (SURVEY.md 8f.1).
//
// The production encoder (ToSpikes with tau = 0.02, datasets.py:21, :72-86) emits rasters whose frames repeat over
// long runs of time steps (periods are 1 or n_steps-1: at most three distinct frames per sample).  Consecutive equal
// frames (b, t-1) == (b, t) have equal input currents, so
//   forward : I_in is computed for the first row of every run only (compact rows) and copied to the rest of the run;
//   backward: dW_in = sum_r x_r^T gI_r = sum_runs x_run^T (sum_{r in run} gI_r)   -- the contraction shrinks from
//             B*T rows to the number of runs; dW_rec still contracts over all rows (the spike trace does not repeat).
// Which rows repeat is data: the encoder records it (changed[b][t], k_encode), k_frame_runs turns it into the run
// table below, and every kernel of both variants (dedup and dense) is launched and gated on the table's `ok` word
// on the DEVICE, so the choice needs no host synchronisation and the step stays capturable in one CUDA graph.
//
// Run table (int32): [0] n_rows (number of runs in the batch)  [1] ok (1: n_rows <= cap, use the dedup kernels)
//                    [2] cap  [3] 0   [4 .. 4+B*T) compact row of every dense row b*T+t
//                    then rep[cap] = first dense row of each run, then len[cap] = its length.
#pragma once
#include "common.cuh"

namespace snnk {

constexpr int kRunHdr = kRunHdrInts;
__host__ __device__ inline int run_cap(long long BT)
{
    long long c = (BT / 4 + 127) / 128 * 128;
    return (int)(c < 128 ? 128 : c);
}
// + one scratch word per sample behind the run lengths (run counts between the two kernels of the parallel build)
__host__ __device__ inline size_t run_table_ints(long long B, long long T)
{
    return (size_t)kRunHdr + (size_t)(B * T) + 2 * (size_t)run_cap(B * T) + (size_t)B;
}

// One CTA of 32 warps.  (1) ballots over the change flags count the runs of every sample; (2) block scan of the counts
// -> first compact row of every sample (in shared memory up to kRunSmemB samples, else in the table's own run-length
// area, cap >= B ints, which is written last); (3) compact row of every step by a ballot prefix, and the first rows;
// (4) run lengths from consecutive first rows.  The kernel is a chain of dependent global round trips, so each phase
// issues all its loads before the first ballot.  A geometry whose scratch does not fit is marked not ok (dense kernels).
constexpr int kRunSmemB = 4096;
constexpr int kRunMaskB = 1024;
__global__ void __launch_bounds__(1024) k_frame_runs(int B, int T, const unsigned char* __restrict__ changed,
                                                    int* __restrict__ table)
{
    __shared__ int s_base[kRunSmemB];
    __shared__ int s_warp[32];
    __shared__ unsigned s_flag[kRunMaskB * 4];   // ballot words of the change flags (T <= 128, B <= kRunMaskB): phase 3
                                                 // then needs no second trip to global memory
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = blockDim.x, nwarp = nthr >> 5;
    const int cap = run_cap((long long)B * T);
    int* row2c = table + kRunHdr;
    int* rep = row2c + (size_t)B * T;
    int* len = rep + cap;
    int* base = B <= kRunSmemB ? s_base : len;
    if (B > kRunSmemB && cap < B) {
        if (tid == 0) { table[0] = B * T; table[1] = 0; table[2] = cap; table[3] = 0; }
        return;
    }
    constexpr int kBatch = 8;
    const bool cached = T <= 128 && B <= kRunMaskB;
    for (int b0 = warp * kBatch; b0 < B; b0 += nwarp * kBatch) {     // kBatch samples per pass, chunk by chunk
        int n[kBatch];
#pragma unroll
        for (int q = 0; q < kBatch; ++q) n[q] = 0;
        for (int t0 = 0; t0 < T; t0 += 32) {
            const int t = t0 + lane;
            bool f[kBatch];
#pragma unroll
            for (int q = 0; q < kBatch; ++q)
                f[q] = b0 + q < B && t < T && (t == 0 || changed[(size_t)(b0 + q) * T + t] != 0);
#pragma unroll
            for (int q = 0; q < kBatch; ++q) {
                const unsigned m = __ballot_sync(0xffffffffu, f[q]);
                n[q] += __popc(m);
                if (cached && lane == 0 && b0 + q < B) s_flag[(b0 + q) * 4 + (t0 >> 5)] = m;
            }
        }
#pragma unroll
        for (int q = 0; q < kBatch; ++q)
            if (lane == q && b0 + q < B) base[b0 + q] = n[q];
    }
    __syncthreads();
    // exclusive scan of the counts: contiguous chunk per thread, warp shuffle scan, scan of the 32 warp totals
    const int per = (B + nthr - 1) / nthr;
    const int lo = min(tid * per, B), hi = min(lo + per, B);
    int mine = 0;
    for (int b = lo; b < hi; ++b) mine += base[b];
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = lane < nwarp ? s_warp[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += v;
        }
        s_warp[lane] = w;      // inclusive totals
    }
    __syncthreads();
    const int total = s_warp[nwarp - 1];
    int run = incl - mine + (warp > 0 ? s_warp[warp - 1] : 0);
    for (int b = lo; b < hi; ++b) { const int n = base[b]; base[b] = run; run += n; }
    __syncthreads();
    for (int b0 = warp * kBatch; b0 < B; b0 += nwarp * kBatch) {     // kBatch samples per pass, chunk by chunk
        int r[kBatch];
#pragma unroll
        for (int q = 0; q < kBatch; ++q) r[q] = (b0 + q < B ? base[b0 + q] : 0) - 1;
        for (int t0 = 0; t0 < T; t0 += 32) {
            const int t = t0 + lane;
            bool f[kBatch];
            unsigned mw[kBatch];
            if (cached) {
#pragma unroll
                for (int q = 0; q < kBatch; ++q) {
                    mw[q] = b0 + q < B ? s_flag[(b0 + q) * 4 + (t0 >> 5)] : 0u;
                    f[q] = (mw[q] >> lane) & 1u;
                }
            } else {
#pragma unroll
                for (int q = 0; q < kBatch; ++q)
                    f[q] = b0 + q < B && t < T && (t == 0 || changed[(size_t)(b0 + q) * T + t] != 0);
            }
#pragma unroll
            for (int q = 0; q < kBatch; ++q) {
                const unsigned m = cached ? mw[q] : __ballot_sync(0xffffffffu, f[q]);
                const int r_t = r[q] + __popc(m & (0xffffffffu >> (31 - lane)));
                if (b0 + q < B && t < T) {
                    row2c[(size_t)(b0 + q) * T + t] = r_t;
                    if (f[q] && r_t < cap) rep[r_t] = (b0 + q) * T + t;
                }
                r[q] += __popc(m);
            }
        }
    }
    __syncthreads();
    const int n = min(total, cap);
    for (int r = tid; r < n; r += nthr) {
        const int row = rep[r], b = row / T;
        const int nxt = (r + 1 < n && rep[r + 1] / T == b) ? rep[r + 1] : (b + 1) * T;
        len[r] = nxt - row;     // (the last stored run of an overfull table may be cut short: the table is not ok then)
    }
    if (tid == 0) {
        table[0] = total;
        table[1] = total <= cap ? 1 : 0;
        table[2] = cap;
        table[3] = 0;
    }
}

// ---- parallel build for T <= 128 (the reference's T = 100): the single-CTA kernel above executes ~64 k warp
// instructions on ONE SM (12 us); here a warp owns a sample, 8 samples per CTA, two launches.
//   k_frame_counts: ballots of the change flags -> run count of every sample (scratch words behind the table)
//   k_frame_fill  : every CTA sums the counts of the samples before its own (B small integers), then writes compact
//                   rows, first rows and run lengths of its samples straight from the ballot words; the CTA that owns
//                   the last sample writes the header.
__global__ void __launch_bounds__(256) k_frame_counts(int B, int T, const unsigned char* __restrict__ changed,
                                                     int* __restrict__ counts)
{
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    bool f[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int t = 32 * c + lane;
        f[c] = t < T && (t == 0 || changed[(size_t)b * T + t] != 0);
    }
    int n = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) n += __popc(__ballot_sync(0xffffffffu, f[c]));
    if (lane == 0) counts[b] = n;
}

__global__ void __launch_bounds__(256) k_frame_fill(int B, int T, const unsigned char* __restrict__ changed,
                                                   const int* __restrict__ counts, int* __restrict__ table)
{
    __shared__ int s_red[8];
    __shared__ int s_cnt[8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b0 = blockIdx.x * 8, b = b0 + warp;
    const int cap = run_cap((long long)B * T);
    int* row2c = table + kRunHdr;
    int* rep = row2c + (size_t)B * T;
    int* len = rep + cap;
    // this sample's flags (issued before the prefix sum: independent loads)
    bool f[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        const int t = 32 * c + lane;
        f[c] = b < B && t < T && (t == 0 || changed[(size_t)b * T + t] != 0);
    }
    // runs of all samples before this CTA's first one
    int part = 0;
    for (int q = tid; q < b0; q += 256) part += counts[q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) { s_red[warp] = part; s_cnt[warp] = b < B ? counts[b] : 0; }
    __syncthreads();
    int base = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) base += s_red[w];
    for (int w = 0; w < warp; ++w) base += s_cnt[w];
    unsigned m[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) m[c] = __ballot_sync(0xffffffffu, f[c]);
    if (b < B) {
        int r = base - 1;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int t = 32 * c + lane;
            const int r_t = r + __popc(m[c] & (0xffffffffu >> (31 - lane)));
            if (t < T) {
                row2c[(size_t)b * T + t] = r_t;
                if (f[c] && r_t < cap) {
                    // length of the run that starts here: distance to the next flag of this sample, or to T
                    unsigned rest = lane < 31 ? (m[c] & (0xffffffffu << (lane + 1))) : 0u;
                    int nxt = T;
                    if (rest) nxt = 32 * c + __ffs(rest) - 1;
                    else {
#pragma unroll
                        for (int c2 = 3; c2 >= 0; --c2)
                            if (c2 > c && m[c2]) nxt = 32 * c2 + __ffs(m[c2]) - 1;
                    }
                    rep[r_t] = b * T + t;
                    len[r_t] = nxt - t;
                }
            }
            r += __popc(m[c]);
        }
        if (b == B - 1 && lane == 0) {
            const int total = base + s_cnt[warp];
            table[0] = total;
            table[1] = total <= cap ? 1 : 0;
            table[2] = cap;
            table[3] = 0;
        }
    }
}

// X_u[r] = X[rep[r]] for r < n_rows; rows up to the next multiple of 32 are zero-filled (the weight-gradient GEMM
// contracts over whole 32-row blocks).  CTAs stride over the compact rows, N/4 float4 per row.
__global__ void __launch_bounds__(256) k_gather_rows(const float* __restrict__ X, const int* __restrict__ table, int BT,
                                                    int N, float* __restrict__ Xu)
{
    // header and the first-row index of this CTA's first compact row are independent loads (the index is inside the
    // table whatever n_rows is): two dependent round trips instead of four on a latency-bound kernel
    const int* rep = table + kRunHdr + BT;
    const int ok = table[1], n_rows = table[0], cap = table[2];
    int first = (int)blockIdx.x < cap ? rep[blockIdx.x] : 0;
    if (ok != 1) return;
    const int n_pad = (n_rows + 31) & ~31;
    for (int r = blockIdx.x; r < n_pad; r += gridDim.x) {
        float4* dst = reinterpret_cast<float4*>(Xu + (size_t)r * N);
        if (r < n_rows) {
            const int row = r == (int)blockIdx.x ? first : rep[r];
            const float4* src = reinterpret_cast<const float4*>(X + (size_t)row * N);
            for (int i = threadIdx.x; i < N / 4; i += blockDim.x) dst[i] = __ldg(src + i);
        } else {
            for (int i = threadIdx.x; i < N / 4; i += blockDim.x) dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

// The same gather for the projection: X_u is written as the K-major, 128B-swizzled shared-memory tiles the tensor pipe
// consumes ([row tile of 128][k-block of 32][row][32 floats], 16-byte chunks permuted by chunk ^ (row & 7), k padded
// with zeros to Kpad), so that the projection kernel fetches an A tile with ONE contiguous 16 KB bulk copy instead of
// a tensor-map box of 128 strided 128-byte rows.
__global__ void __launch_bounds__(256) k_gather_rows_tiled(const float* __restrict__ X, const int* __restrict__ table,
                                                          int BT, int N, int Kpad, float* __restrict__ Xt)
{
    const int* rep = table + kRunHdr + BT;
    const int ok = table[1], n_rows = table[0], cap = table[2];
    int first = (int)blockIdx.x < cap ? rep[blockIdx.x] : 0;      // independent of the header loads (see k_gather_rows)
    if (ok != 1) return;
    const int kblocks = Kpad / 32;
    for (int r = blockIdx.x; r < n_rows; r += gridDim.x) {
        const int row = r == (int)blockIdx.x ? first : rep[r];
        const float4* src = reinterpret_cast<const float4*>(X + (size_t)row * N);
        const int mt = r >> 7, rr = r & 127;
        for (int c4 = threadIdx.x; c4 < Kpad / 4; c4 += blockDim.x) {
            const float4 v = 4 * c4 < N ? __ldg(src + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
            const int kb = c4 >> 3, c = c4 & 7;
            float* tile = Xt + ((size_t)mt * kblocks + kb) * (128 * 32);
            reinterpret_cast<float4*>(tile + rr * 32)[c ^ (rr & 7)] = v;
        }
    }
}

// The run sums of gI (compact rows of the dW_in contraction) are produced by the BPTT sweep itself: recur_bwd.cuh.

}  // namespace snnk
