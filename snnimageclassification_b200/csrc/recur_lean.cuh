// recur_lean.cuh -- the forward recurrence of the HEADLINE geometry with a minimal step.
//
// k_recur_fwd (recur_fwd.cuh) serves every layer type, row count and input variant with one step loop; at batch 256
// that loop is bound by the in-order issue of its 169 instructions per warp-step, of which 64 are the recurrent
// sum (ncu, profiles/r02_*: one warp per scheduler, no second warp to switch to -- DESIGN.md section 3).  This
// kernel is the same arithmetic in the same order (bit-identical outputs) for the case that matters most --
// recurrent LIF / ALIF, H = 128, one row per CTA, T * H * 4 <= 64 KB -- with everything that is not the step taken out
// of the loop:
//   * the row's whole input current (T x H floats) sits in shared memory before the loop starts -- ONE bulk copy of
//     the contiguous block for dense input, or the compact rows of the frame-dedup variant expanded per step by plain
//     loads in the prologue -- so a step reads its current with one LDS at an incrementing address: no ring, no
//     mbarrier wait, no compact-row lookup, no uniform-register traffic in the loop;
//   * trace pointers advance by H per step instead of being rebuilt from (b, t, i);
//   * the double-buffer parity of the spike vector is compile-time (two steps per loop iteration);
//   * layer type and trace output are template parameters.
// The recurrent matrix is staged through shared memory in two halves (32 KB) so that two CTAs still fit an SM.
// k_recur_bwd_lean below is the matching BPTT sweep, and k_train_lean runs forward, head and sweep of a row in one CTA.
#pragma once
#include <type_traits>

#include "recur_bwd.cuh"
#include "recur_fwd.cuh"
#include "gemm_bits.cuh"   // fence_proxy_async_smem

namespace snnk {

template <int H>
constexpr size_t lean_fwd_smem_bytes(int T, int O)
{
    return sizeof(float) * (size_t)(2 * H) + sizeof(uint32_t) * (size_t)((T * (H / 32) + 3) & ~3) +
           sizeof(float) * (size_t)((H * 12 + T * kOMax + 3) & ~3) + sizeof(float) * (size_t)T * H +
           sizeof(float) * (size_t)(H / 2) * H + sizeof(uint64_t) * 2;
}

// rows [half * H/2, (half+1) * H/2) of the staged matrix -> the matching half of the column-blocked register file
template <int H>
__device__ __forceinline__ void load_w_cb_half(float (&w)[H], const float* __restrict__ s_half, int i, int half)
{
    const int g = i & 3, c0 = i & ~3;
#pragma unroll
    for (int ci = 0; ci < 4; ++ci)
#pragma unroll
        for (int j = 0; j < H / 16; ++j)
            if ((j >= H / 32) == (half != 0)) {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    w[(ci * (H / 16) + j) * 4 + e] = s_half[(16 * (j - half * (H / 32)) + 4 * g + e) * H + c0 + ci];
            }
}

// Tail of the lean forward kernel (one row per CTA): the same sums in the same order as fwd_tail / head_tail, laid out
// for a CTA that owns ONE row (ncu: the shared tail was 30 % of this kernel).
//   * readout sums s[t][c] = sum_j Z_t[j] W_out[j][c], ascending j: thread = time step, walking the SET bits of its
//     four spike words only (adding nothing for a silent neuron is what the predicated add of fwd_tail does too) and
//     adding the neuron's row of W_out (three LDS.128 from rows padded to 12 floats) to its ten running sums;
//   * the scan over t per class reads eight sums ahead of its own stores;
//   * the head: one warp, lane = class -- exponentials and log-probabilities in parallel, the sum of exponentials in
//     class order as k_head_nll forms it.
constexpr int kLeanOP = 12;     // row pitch of the readout matrix in shared memory (O <= 12)

// Returns, to thread c < O, the first arg-max step of class c (tstar); -1 to the other threads.
template <int H>
__device__ __forceinline__ int fwd_tail_lean(const FwdParams& p, const uint32_t* s_mask, const float* s_wout, float* s_s,
                                             float* s_logit, int b, int tid)
{
    int ts = -1;
    constexpr int W32 = H / 32;
    const int T = p.T, O = p.O;
    for (int idx = tid; idx < T * W32; idx += H) p.zbits[(size_t)b * T * W32 + idx] = s_mask[idx];
    for (int t = tid; t < T; t += H) {
        float sum[kLeanOP];
#pragma unroll
        for (int c = 0; c < kLeanOP; ++c) sum[c] = 0.f;
#pragma unroll
        for (int wd = 0; wd < W32; ++wd) {
            uint32_t m = s_mask[t * W32 + wd];
            while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1;
                const float4* wr = reinterpret_cast<const float4*>(s_wout + (wd * 32 + l) * kLeanOP);
#pragma unroll
                for (int q = 0; q < kLeanOP / 4; ++q) {
                    const float4 w4 = wr[q];
                    sum[4 * q + 0] = __fadd_rn(sum[4 * q + 0], w4.x);
                    sum[4 * q + 1] = __fadd_rn(sum[4 * q + 1], w4.y);
                    sum[4 * q + 2] = __fadd_rn(sum[4 * q + 2], w4.z);
                    sum[4 * q + 3] = __fadd_rn(sum[4 * q + 3], w4.w);
                }
            }
        }
#pragma unroll
        for (int c = 0; c < kLeanOP; ++c)
            if (c < O) s_s[t * O + c] = sum[c];
    }
    __syncthreads();
    // y_t = kappa y_{t-1} + s_t + b (spiking_layers.py:407) and the first maximum over time (snn.py:228)
    if (tid < O) {
        const int c = tid;
        const float bc = __ldg(p.b_out + c);
        float yv = 0.f, mx = 0.f;
        int mt = 0;
        for (int t0 = 0; t0 < T; t0 += 8) {
            float sv[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) sv[q] = (t0 + q < T) ? s_s[(t0 + q) * O + c] : 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int t = t0 + q;
                if (t < T) {
                    yv = __fadd_rn(__fadd_rn(__fmul_rn(p.kappa, yv), sv[q]), bc);
                    s_s[t * O + c] = yv;
                    if (t == 0 || yv > mx) { mx = yv; mt = t; }
                }
            }
        }
        p.logits[(size_t)b * O + c] = mx;
        p.tstar[(size_t)b * O + c] = mt;
        s_logit[c] = mx;
        ts = mt;
    }
    __syncthreads();
    for (int idx = tid; idx < T * O; idx += H) p.y[(size_t)b * T * O + idx] = s_s[idx];
    return ts;
}

// Returns, to thread c < O, the row's dL/dlogits of class c (when p.g_logits is set); 0 to the other threads.
__device__ __forceinline__ float head_tail_lean(const FwdParams& p, const float* s_logit, int* s_hd, double* s_hp, int b, int tid,
                                                int nthr)
{
    constexpr long long kIgnore = -100;
    const int O = p.O, B = p.B;
    const int n_valid = s_hd[0];
    const bool bad = s_hd[1] != 0;
    const int lane = tid & 31;
    float g_row = 0.f;
    if (tid < 32) {
        const float lg = lane < O ? s_logit[lane] : -INFINITY;
        float mx = lg;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float e = lane < O ? expf(lg - mx) : 0.f;
        float se = 0.f;
        for (int c = 0; c < O; ++c) se += __shfl_sync(0xffffffffu, e, c);       // class order, as k_head_nll
        const float lse = logf(se);
        const float lp = (lg - mx) - lse;
        const long long lab = p.labels[b];
        const bool row_ok = lab >= 0 && lab < O, row_bad = !row_ok && lab != kIgnore;
        if (lane < O) {
            if (p.logp) p.logp[(size_t)b * O + lane] = lp;
            if (p.g_logits) {
                float g = row_ok ? __fdiv_rn(expf(lp) - (lane == lab ? 1.0f : 0.0f), (float)n_valid) : 0.0f;
                if (row_bad) g = __int_as_float(0x7fc00000);
                p.g_logits[(size_t)b * O + lane] = g;
                g_row = g;
            }
        }
        const float nll = -__shfl_sync(0xffffffffu, lp, row_ok ? (int)lab : 0);
        if (lane == 0) {
            p.part_nll[b] = row_ok ? nll : 0.f;
            __threadfence();
            s_hd[2] = atomicAdd(p.ticket, 1u) == gridDim.x - 1;
        }
    }
    __syncthreads();
    if (s_hd[2]) {      // the last CTA to finish: the loss (block-uniform branch)
        __threadfence();
        for (int vw = tid >> 5; vw < 8; vw += nthr >> 5) {
            double acc = 0.0;
            for (int bb = vw * 32 + lane; bb < B; bb += 256) acc += (double)__ldcg(p.part_nll + bb);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) s_hp[vw] = acc;
        }
        __syncthreads();
        if (tid == 0) {
            double sum = 0.0;
            for (int q = 0; q < 8; ++q) sum += s_hp[q];
            const float lossf = bad ? __int_as_float(0x7fc00000) : (float)(sum / (double)n_valid);
            *p.loss = lossf;
            *p.ticket = 0u;
            if (p.mailbox) {
                const unsigned int seq = *p.mail_counter + 1u;
                *p.mail_counter = seq;
                *reinterpret_cast<volatile unsigned long long*>(p.mailbox) =
                    (static_cast<unsigned long long>(seq) << 32) | __float_as_uint(lossf);
                __threadfence_system();
            }
        }
    }
    return g_row;
}

// Dynamic shared memory of the lean forward kernel (lean_fwd_smem_bytes)
template <int H>
struct LeanFwdSmem {
    float* s_z;         // [2][H] spike vector of the previous / current step
    uint32_t* s_mask;   // [T][W32] spike words of the row
    float* s_wout;      // [H][12]: rows of W_out padded with zeros
    float* s_s;         // [T][O] (tail); compact rows of the steps (prologue)
    float* s_cur;       // [T][H] input current of the row
    float* s_w;         // [H/2][H] staging of the recurrent matrix
    uint64_t* s_bar;    // [0] weights, [1] input current
    __device__ __forceinline__ LeanFwdSmem(unsigned char* raw, int T)
    {
        s_z = reinterpret_cast<float*>(raw);
        s_mask = reinterpret_cast<uint32_t*>(s_z + 2 * H);
        s_wout = reinterpret_cast<float*>(s_mask + ((T * (H / 32) + 3) & ~3));
        s_s = s_wout + H * kLeanOP;
        s_cur = s_wout + ((H * kLeanOP + T * kOMax + 3) & ~3);
        s_w = s_cur + (size_t)T * H;
        s_bar = reinterpret_cast<uint64_t*>(s_w + (H / 2) * H);
    }
};

// Prologue of the lean forward (one row per CTA): W_eff in registers (column-blocked), the row's input current in s_cur,
// W_out in s_wout, the initial state, and the head's count of valid rows.  FENCE_W: this thread's reads of the staging
// area are also ordered before async-proxy writes that the caller issues there after the closing barrier.
template <int H, bool ALIF, bool FENCE_W>
__device__ __forceinline__ void lean_fwd_prologue(const FwdParams& p, const LeanFwdSmem<H>& sm, int* s_hd, float (&w)[H],
                                                  float& beta, float& v, float& a, float& zp)
{
    const int T = p.T, O = p.O;
    const int i = threadIdx.x;
    const int b = blockIdx.x;
    float* const s_z = sm.s_z;
    float* const s_wout = sm.s_wout;
    float* const s_s = sm.s_s;
    float* const s_cur = sm.s_cur;
    float* const s_w = sm.s_w;
    uint64_t* const s_bar = sm.s_bar;

    const bool compact = p.run_table != nullptr && p.run_table[1] == 1;
    constexpr uint32_t kHalfBytes = (uint32_t)((H / 2) * H * sizeof(float));
    if (i == 0) {
        s_hd[0] = s_hd[1] = s_hd[2] = 0;
        tc::mbar_init(s_bar, 1);
        tc::mbar_init(s_bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        tc::mbar_expect_tx(s_bar, kHalfBytes);
        tc::bulk_g2s(s_w, p.W_eff, kHalfBytes, s_bar);
    }
    // The row's input current: the contiguous T x H block (dense), or -- frame-dedup variant -- the sample's compact rows,
    // consecutive rows of I_u (at most T of them), by one bulk copy to the START of the buffer; spread over the steps below.
    // Launched as a programmatic dependent of the projection (p.pdl) everything above and below runs while the
    // projection may still be writing I_in / I_u: the copy is issued last, behind griddepcontrol.wait.
    int cp_first = 0, cp_last = 0;
    if (i == 0 && compact) {
        const int* r2c = p.run_table + kRunHdrInts + (size_t)b * T;
        cp_first = __ldg(r2c);
        cp_last = __ldg(r2c + T - 1);
    }
    auto issue_current = [&]() {      // thread 0 only
        if (p.pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
        if (!compact) {
            const uint32_t bytes = (uint32_t)((size_t)T * H * sizeof(float));
            tc::mbar_expect_tx(s_bar + 1, bytes);
            tc::bulk_g2s(s_cur, p.I_in + (size_t)b * T * H, bytes, s_bar + 1);
        } else {
            const uint32_t bytes = (uint32_t)((size_t)(cp_last - cp_first + 1) * H * sizeof(float));
            tc::mbar_expect_tx(s_bar + 1, bytes);
            tc::bulk_g2s(s_cur, p.I_u + (size_t)cp_first * H, bytes, s_bar + 1);
        }
    };
    if (i == 0 && !p.pdl) issue_current();
    int* s_r2c = reinterpret_cast<int*>(s_s);      // [T] compact row of every step, relative to the sample's first (prologue only)
    if (compact) {
        const int* r2c = p.run_table + kRunHdrInts + (size_t)b * T;
        const int first = __ldg(r2c);
        for (int t = i; t < T; t += H) s_r2c[t] = __ldg(r2c + t) - first;
    }
    __syncthreads();
    if (p.labels) head_count(p, s_hd, i, H);

    tc::mbar_wait(s_bar, 0);
    load_w_cb_half<H>(w, s_w, i, 0);
    // The second half is written into the same staging area by the ASYNC proxy, the reads above went through the generic
    // proxy: without this proxy fence the copy can overtake them (observed: one or two wrong rows per launch of 256 with
    // two CTAs per SM, none with one -- a barrier alone does not order the two proxies).
    tc::fence_proxy_async_smem();
    __syncthreads();                               // everybody is done with the first half
    if (i == 0) {
        tc::mbar_expect_tx(s_bar, kHalfBytes);
        tc::bulk_g2s(s_w, p.W_eff + (size_t)(H / 2) * H, kHalfBytes, s_bar);
    }
    beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
    v = p.V0 ? p.V0[(size_t)b * H + i] : 0.f;
    a = p.a0 ? p.a0[(size_t)b * H + i] : 0.f;
    zp = p.Z0 ? p.Z0[(size_t)b * H + i] : 0.f;
    s_z[H + i] = zp;                               // step 0 reads buffer 1
    for (int idx = i; idx < H * kLeanOP; idx += H) {
        const int j = idx / kLeanOP, c = idx - j * kLeanOP;
        s_wout[idx] = c < O ? __ldg(p.W_out + j * O + c) : 0.f;
    }
    tc::mbar_wait(s_bar, 1);
    load_w_cb_half<H>(w, s_w, i, 1);
    if constexpr (FENCE_W) tc::fence_proxy_async_smem();
    if (i == 0 && p.pdl) issue_current();
    tc::mbar_wait(s_bar + 1, 0);
    if (compact) {
        // step t takes compact row s_r2c[t] <= t (the table never advances by more than one row per step), so walking t
        // DOWNWARDS in place never overwrites a compact row a smaller t still needs; thread i only touches column i
        // (eight steps are read before any of them is written: the loads of a batch are independent of its stores)
        for (int t0 = T - 1; t0 >= 0; t0 -= 8) {
            float cv[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) cv[q] = (t0 - q >= 0) ? s_cur[s_r2c[t0 - q] * H + i] : 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (t0 - q >= 0) s_cur[(t0 - q) * H + i] = cv[q];
        }
    }
    __syncthreads();
}

// What a forward step leaves in memory besides the spike words: nothing, the traces V, Z (and a), or -- for the fused
// training kernel -- Z and, in the step's own input-current slot, sigma'_t = surrogate'(V_t, threshold_t), the only
// thing the reverse sweep of a LIF / ALIF layer needs from V and a.
constexpr int kLeanOutNone = 0, kLeanOutTraces = 1, kLeanOutSweep = 2;

// One step of the lean forward for neuron i = threadIdx.x; BUF = buffer of s_z the step WRITES (it reads the other one).
template <int H, bool ALIF, int OUT, int SURR, int BUF>
__device__ __forceinline__ void lean_fwd_step(const FwdParams& p, const float (&w)[H], float* s_z, float*& curp,
                                              uint32_t*& maskp, size_t& tro, float& v, float& a, float& zp, float beta)
{
    constexpr int W32 = H / 32;
    const int i = threadIdx.x, lane = i & 31;
    float* const slot = curp;
    const float cur = *curp;
    curp += H;
    const float rec = dot_rec16_cb<H>(w, reinterpret_cast<const float4*>(s_z + (BUF ? 0 : H)), i & 3);
    // V' = (alpha V + I_in + I_rec) (1 - Z.detach())     spiking_layers.py:169/239
    const float t1 = __fmul_rn(p.alpha, v);
    const float t2 = __fadd_rn(t1, cur);
    const float t3 = __fadd_rn(t2, rec);
    const float vn = __fmul_rn(t3, __fsub_rn(1.0f, zp));
    float thr = p.theta;
    if constexpr (ALIF) {
        a = __fadd_rn(__fmul_rn(p.rho, a), zp);                    // :240
        thr = __fadd_rn(p.theta, __fmul_rn(beta, a));              // :241
    }
    const float zn = vn >= thr ? 1.0f : 0.0f;                      // spike_funcs.py:27-28
    s_z[BUF * H + i] = zn;
    if constexpr (OUT == kLeanOutTraces) {
        p.V[tro] = vn;
        p.Z[tro] = zn;
        if constexpr (ALIF) p.a[tro] = a;
        tro += H;
    }
    if constexpr (OUT == kLeanOutSweep) {
        *slot = surrogate_grad<SURR>(p.gamma, vn, thr);     // slot t is read by this thread only, and already was
        p.Z[tro] = zn;
        tro += H;
    }
    const unsigned m = __ballot_sync(0xffffffffu, zn != 0.f);
    if (lane == 0) *maskp = m;
    maskp += W32;
    v = vn;
    zp = zn;
    __syncthreads();
}

template <int H, bool ALIF, bool TRACES>
__global__ void __launch_bounds__(H, 256 / H) k_recur_fwd_lean(const FwdParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int T = p.T;
    const int i = threadIdx.x, warp = i >> 5;
    const int b = blockIdx.x;                                                       // one row per CTA
    const LeanFwdSmem<H> sm(smem_raw, T);
    __shared__ int s_hd[4];
    __shared__ double s_hp[8];
    __shared__ float s_logit[kOMax];

    float w[H];
    float beta, v, a, zp;
    lean_fwd_prologue<H, ALIF, false>(p, sm, s_hd, w, beta, v, a, zp);

    float* curp = sm.s_cur + i;
    uint32_t* maskp = sm.s_mask + warp;
    size_t tro = (size_t)b * T * H + i;
    constexpr int OUT = TRACES ? kLeanOutTraces : kLeanOutNone;
    int t = 0;
    for (; t + 1 < T; t += 2) {
        lean_fwd_step<H, ALIF, OUT, 0, 0>(p, w, sm.s_z, curp, maskp, tro, v, a, zp, beta);
        lean_fwd_step<H, ALIF, OUT, 0, 1>(p, w, sm.s_z, curp, maskp, tro, v, a, zp, beta);
    }
    if (t < T) lean_fwd_step<H, ALIF, OUT, 0, 0>(p, w, sm.s_z, curp, maskp, tro, v, a, zp, beta);
    __syncthreads();

    fwd_tail_lean<H>(p, sm.s_mask, sm.s_wout, sm.s_s, s_logit, b, i);
    if (p.labels) head_tail_lean(p, s_logit, s_hd, s_hp, b, i, H);
}

// ---- backward -------------------------------------------------------------------------------------------------------
// k_recur_bwd (recur_bwd.cuh) with the same treatment for the training step of the headline geometry: recurrent LIF /
// ALIF, H = 128, one row per CTA, sparse seeds from the fused head (g_logits, tstar), no seeds on V / Z.  Same arithmetic
// in the same order.  The saved traces still stream through the bulk-copy ring (V and a of a whole row are 100 KB: two
// CTAs would no longer fit an SM), but the ring is walked as chunk x step loops with the eight steps of a chunk
// unrolled: ring offsets, the parity of the gI double buffer and the chunk-boundary test are compile-time, the
// pointers into the adjoint rows / spike words / gI advance by constants, the previous step's spike word is carried in
// a register, and layer type, surrogate, plane split and run sums are template parameters -- the 269 instructions of a
// step of the general kernel contain ~70 of uniform-datapath bookkeeping and branches (profiles/r02_*).
// OP: readout width padded to whole float4 (12 for ten classes): columns >= O of the adjoint rows and of W_out are zero,
// so leaving them out of the two FMA chains changes nothing but the instruction count.
// Frame-dedup variant: the run of step t = i and of step i - 1, and the run of the row's last step.
__device__ __forceinline__ void lean_run_rows(const int* run_table, int T, int b, int i, int& rc_t, int& rc_p, int& crow)
{
    const int* rc = run_table + kRunHdrInts + (size_t)b * T;
    if (i < T) {
        rc_t = __ldg(rc + i);
        if (i > 0) rc_p = __ldg(rc + i - 1);
    }
    crow = __ldg(rc + T - 1);
}

// Frame-dedup variant: the row's run-start bits, and (CTA 0) zeros in the tail of the last 32-row block of the run sums
__device__ __forceinline__ void lean_run_starts(const BwdParams& p, uint32_t* s_start, int rc_t, int rc_p, int i)
{
    const int T = p.T, TW = (T + 31) >> 5;
    if (i < TW) s_start[i] = 0u;
    __syncthreads();
    // bit t of the word: step t is the first of its run of equal input frames
    if (i < T && (i == 0 || rc_t != rc_p)) atomicOr(s_start + (i >> 5), 1u << (i & 31));
    if (blockIdx.x == 0) {   // the weight-gradient GEMM contracts whole 32-row blocks: zero the tail of the last one
        const int n_rows = p.run_table[0], n_pad = (n_rows + 31) & ~31;
        for (int idx = i; idx < (n_pad - n_rows) * 128; idx += 128) {
            p.Gu_hi[(size_t)n_rows * 128 + idx] = 0.f;
            p.Gu_lo[(size_t)n_rows * 128 + idx] = 0.f;
        }
    }
}

// readout adjoint scan gy_t = seed_t + kappa gy_{t+1}  (spiking_layers.py:407 backwards) and db: the seed of a class
// sits at one step (its arg-max over time), so the chain runs in registers -- the same two operations per step as
// the general kernel's scan over shared memory -- and fills the class's whole column, padding columns with zeros
__device__ __forceinline__ void lean_gy_scan(const BwdParams& p, float* s_gy, float seed, int ts, int i)
{
    const int T = p.T, O = p.O;
    if (i < kOMax) {
        float g = 0.f, sum = 0.f;
        for (int t = T - 1; t >= 0; --t) {
            g = __fadd_rn(t == ts ? seed : 0.f, __fmul_rn(p.kappa, g));
            s_gy[t * kOMax + i] = g;
            sum += g;
        }
        if (i < O) p.part_db[(size_t)blockIdx.x * O + i] = sum;
    }
}

// One reverse step t of the lean sweep for neuron i = threadIdx.x.  PAR = t & 1 (the buffer gI_t is written to; gI_{t+1}
// is read from the other one); sigma() yields sigma'_t.
template <int OP, bool PLANES, bool RUNS, int PAR, class Sigma>
__device__ __forceinline__ void lean_bwd_step(const BwdParams& p, int t, const float (&w)[128], const float (&wo)[OP],
                                              float (&dwo)[OP], float* s_g, const uint32_t* s_start, bool run_sums,
                                              const float4*& gyp, const uint32_t*& mkp, uint32_t& mword, float& gv,
                                              float& racc, uint32_t& sbits, int& crow, size_t& tro, Sigma&& sigma)
{
    constexpr int H = 128, W32 = H / 32;
    const int i = threadIdx.x, lane = i & 31;
    const int b = blockIdx.x;
    float gy[OP];
#pragma unroll
    for (int q = 0; q < OP / 4; ++q) {
        const float4 g4 = gyp[q];
        gy[4 * q + 0] = g4.x; gy[4 * q + 1] = g4.y; gy[4 * q + 2] = g4.z; gy[4 * q + 3] = g4.w;
    }
    gyp -= kOMax / 4;
    const float zt = (float)((mword >> lane) & 1u);
    float zprev;
    if (t > 0) {
        mkp -= W32;
        mword = *mkp;
        zprev = (float)((mword >> lane) & 1u);
    } else {
        zprev = p.Z0 ? __ldg(p.Z0 + (size_t)b * H + i) : 0.f;
    }
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < OP; ++c) {
        s = fmaf(gy[c], wo[c], s);               // gy_t W_out^T
        dwo[c] = fmaf(zt, gy[c], dwo[c]);        // dW_out += Z_t^T gy_t
    }
    s = __fadd_rn(s, dot_rec16_cb<H>(w, reinterpret_cast<const float4*>(s_g + (PAR ? 0 : H)), i & 3));   // gI_{t+1} (W_rec . M)^T
    const float sg = sigma();
    const float carry = __fmul_rn(__fmul_rn(p.alpha, gv), __fsub_rn(1.0f, zt));
    const float g = __fadd_rn(__fmul_rn(s, sg), carry);
    gv = g;
    const float gi = __fmul_rn(g, __fsub_rn(1.0f, zprev));
    if (PLANES) {   // tensor-core mode: exact two-plane tf32 split for the weight-gradient GEMM
        const float hi = __uint_as_float(__float_as_uint(gi) & 0xFFFFE000u);
        p.gI[tro] = hi;
        p.gI_lo[tro] = __fsub_rn(gi, hi);
    } else {
        p.gI[tro] = gi;
    }
    tro -= H;
    s_g[PAR * H + i] = gi;
    if (RUNS && run_sums) {   // sum of gI over the run of equal input frames this step belongs to
        racc = __fadd_rn(racc, gi);
        if (t == p.T - 1 || (t & 31) == 31) sbits = s_start[t >> 5];
        if ((sbits >> (t & 31)) & 1u) {
            const float hi = __uint_as_float(__float_as_uint(racc) & 0xFFFFE000u);
            p.Gu_hi[(size_t)crow * H + i] = hi;
            p.Gu_lo[(size_t)crow * H + i] = __fsub_rn(racc, hi);
            racc = 0.f;
            --crow;
        }
    }
    __syncthreads();
}

template <bool ALIF, int SURR, bool PLANES, bool RUNS, int OP>
__global__ void __launch_bounds__(128, 2) k_recur_bwd_lean(const BwdParams p)
{
    constexpr int H = 128, W32 = H / 32;
    static_assert(OP % 4 == 0 && OP <= kOMax, "readout padding");
    static_assert(kChunk % 2 == 0, "compile-time parity of the gI double buffer");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int T = p.T, O = p.O;
    const int i = threadIdx.x, warp = i >> 5;
    const int b = blockIdx.x;

    // Everything the prologue needs from global memory is requested FIRST, into registers: the weight staging below
    // (64 KB through shared memory, which the loop buffers alias) then overlaps those round trips instead of
    // preceding six of them one after the other (ncu: 15 % of the general kernel was prologue).
    const bool run_sums = RUNS && p.run_table != nullptr && p.run_table[1] == 1;
    uint32_t zw[4];                                        // spike words i, i+H, ... of the row (T * W32 <= 4 H)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int idx = i + q * H;
        zw[q] = idx < T * W32 ? __ldg(p.zbits + (size_t)b * T * W32 + idx) : 0u;
    }
    int rc_t = 0, rc_p = -1, crow = 0;                     // run of step t = i and of step i-1; run of the last step
    if (run_sums) lean_run_rows(p.run_table, T, b, i, rc_t, rc_p, crow);
    float seed = 0.f;                                      // thread c < O: the seed of class c at its arg-max step
    int ts = -1;
    if (i < O) {
        const float scale = p.g_scale ? __ldg(p.g_scale) : 1.0f;
        ts = __ldg(p.tstar + (size_t)b * O + i);
        seed = __fmul_rn(__ldg(p.g_logits + (size_t)b * O + i), scale);
    }
    float wo[OP], dwo[OP];
#pragma unroll
    for (int c = 0; c < OP; ++c) {
        wo[c] = c < O ? __ldg(p.W_out + (size_t)i * O + c) : 0.f;
        dwo[c] = 0.f;
    }
    const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;

    float w[H];
    {
        float* s_t = reinterpret_cast<float*>(smem_raw);                        // [H][H], aliases the loop buffers
        uint64_t* wbar = reinterpret_cast<uint64_t*>(s_t + H * H);
        if (i == 0) {
            tc::mbar_init(wbar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            tc::mbar_expect_tx(wbar, (uint32_t)(H * H * sizeof(float)));
            tc::bulk_g2s(s_t, p.W_effT, (uint32_t)(H * H * sizeof(float)), wbar);
        }
        __syncthreads();
        tc::mbar_wait(wbar, 0);
        load_w_cb<H>(w, s_t, i);
        tc::fence_proxy_async_smem();      // the ring's bulk copies (async proxy) land in this area later
        __syncthreads();
        if (i == 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(tc::smem_u32(wbar)) : "memory");
    }

    float* s_g = reinterpret_cast<float*>(smem_raw);                       // [2][H]
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_g + 2 * H);           // [T][W32]
    float* s_gy = reinterpret_cast<float*>(s_mask + ((T * W32 + 3) & ~3)); // [T][kOMax], 16-B aligned
    float* s_v = s_gy + T * kOMax;                                         // [kRing][kChunk][H]
    float* s_a = s_v + kRing * kChunk * H;
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_a + kRing * kChunk * H);
    uint32_t* s_start = reinterpret_cast<uint32_t*>(s_bar + kRing);        // [ceil(T/32)] run-start bits

    const int nchunks = (T + kChunk - 1) / kChunk;
    auto issue_chunk = [&](int k) {
        const int slot = k % kRing, t0 = (nchunks - 1 - k) * kChunk;
        const uint32_t bytes = (uint32_t)(min(kChunk, T - t0) * H * sizeof(float));
        tc::mbar_expect_tx(s_bar + slot, bytes * (ALIF ? 2 : 1));
        const size_t g = ((size_t)b * T + t0) * H;
        tc::bulk_g2s(s_v + (slot * kChunk) * H, p.V + g, bytes, s_bar + slot);
        if (ALIF) tc::bulk_g2s(s_a + (slot * kChunk) * H, p.a + g, bytes, s_bar + slot);
    };
    if (i == 0) {
        for (int s = 0; s < kRing; ++s) tc::mbar_init(s_bar + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int k = 0; k < kRing && k < nchunks; ++k) issue_chunk(k);
    }

    for (int idx = i; idx < 2 * H; idx += H) s_g[idx] = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (i + q * H < T * W32) s_mask[i + q * H] = zw[q];
    if (run_sums) lean_run_starts(p, s_start, rc_t, rc_p, i);
    lean_gy_scan(p, s_gy, seed, ts, i);
    __syncthreads();

    float gv = 0.f, racc = 0.f;
    uint32_t sbits = 0u;
    size_t tro = ((size_t)b * T + (T - 1)) * H + i;
    const float4* gyp = reinterpret_cast<const float4*>(s_gy + (T - 1) * kOMax);
    const uint32_t* mkp = s_mask + (T - 1) * W32 + warp;
    uint32_t mword = *mkp;                                 // spike word of step t (carried: it is step t+1's "previous")
    // one step.  PAR = t & 1 (the buffer gI_t is written to; gI_{t+1} is read from the other one)
    auto step = [&](int t, const float* vrow, const float* arow, auto par_tag) {
        constexpr int PAR = decltype(par_tag)::value;
        const float vt = vrow[i];
        const float at = ALIF ? arow[i] : 0.f;
        lean_bwd_step<OP, PLANES, RUNS, PAR>(p, t, w, wo, dwo, s_g, s_start, run_sums, gyp, mkp, mword, gv, racc, sbits,
                                             crow, tro, [&] {
                                                 float thr = p.theta;
                                                 if (ALIF) thr = __fadd_rn(p.theta, __fmul_rn(beta, at));
                                                 return surrogate_grad<SURR>(p.gamma, vt, thr);
                                             });
    };

    for (int k = 0; k < nchunks; ++k) {
        const int slot = k % kRing, t0 = (nchunks - 1 - k) * kChunk;
        // every thread has passed the barrier of the last step of chunk k-1: its slot can be refilled
        if (i == 0 && k >= 1 && k - 1 + kRing < nchunks) issue_chunk(k - 1 + kRing);
        tc::mbar_wait(s_bar + slot, (k / kRing) & 1);
        const float* vs = s_v + (slot * kChunk) * H;
        const float* as = s_a + (slot * kChunk) * H;
        if (T - t0 >= kChunk) {
#pragma unroll
            for (int tt = kChunk - 1; tt >= 0; --tt) {
                if (tt & 1) step(t0 + tt, vs + tt * H, as + tt * H, std::integral_constant<int, 1>{});
                else step(t0 + tt, vs + tt * H, as + tt * H, std::integral_constant<int, 0>{});
            }
        } else {
            for (int tt = T - t0 - 1; tt >= 0; --tt) {
                if (tt & 1) step(t0 + tt, vs + tt * H, as + tt * H, std::integral_constant<int, 1>{});
                else step(t0 + tt, vs + tt * H, as + tt * H, std::integral_constant<int, 0>{});
            }
        }
    }
#pragma unroll
    for (int c = 0; c < OP; ++c)
        if (c < O) p.part_wout[((size_t)blockIdx.x * H + i) * O + c] = dwo[c];
}

// ---- forward, head and BPTT sweep of a row in one CTA ----------------------------------------------------------------
// k_recur_fwd_lean with its head, then k_recur_bwd_lean<.., kLeanOP> in LIF mode, in the CTA that owns the row: the
// row's dL/dlogits depends on that row alone (every CTA counts n_valid in its prologue), so no CTA waits for another
// and the sweep needs no second launch.  Same arithmetic in the same order as the two kernels (bit-identical results):
//   * the forward overwrites step t's slot of the row's input current, which it reads once at step t, with sigma'_t of
//     the V_t and threshold it just computed, and stores Z (the weight-gradient GEMM reads it) but neither V nor a: the
//     reverse loop reads sigma'_t from shared memory where k_recur_bwd_lean streams V and a back through its ring;
//   * the spike words, W_out, tstar and the seeds stay on chip;
//   * W_effT goes through the forward's weight staging area in two halves: the first while the forward loop runs,
//     the second behind the tail.
// Shared memory is the forward kernel's (lean_fwd_smem_bytes): s_g aliases s_z and s_gy the tail's s_s.
template <bool ALIF, int SURR, bool PLANES, bool RUNS>
__global__ void __launch_bounds__(128, 2) k_train_lean(const FwdParams p, const BwdParams q)
{
    constexpr int H = 128, W32 = H / 32, OP = kLeanOP;
    constexpr uint32_t kHalfBytes = (uint32_t)((H / 2) * H * sizeof(float));
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int T = p.T, O = p.O;
    const int i = threadIdx.x, warp = i >> 5;
    const int b = blockIdx.x;
    const LeanFwdSmem<H> sm(smem_raw, T);
    __shared__ int s_hd[4];
    __shared__ double s_hp[8];
    __shared__ float s_logit[kOMax];
    __shared__ uint32_t s_start[4];                        // run-start bits of the row (T <= 128)

    const bool run_sums = RUNS && q.run_table != nullptr && q.run_table[1] == 1;
    int rc_t = 0, rc_p = -1, crow = 0;                     // run of step t = i and of step i-1; run of the last step
    if (run_sums) lean_run_rows(q.run_table, T, b, i, rc_t, rc_p, crow);
    const float scale = __ldg(q.g_scale);

    float w[H];
    float beta, v, a, zp;
    lean_fwd_prologue<H, ALIF, true>(p, sm, s_hd, w, beta, v, a, zp);
    if (i == 0) {
        tc::mbar_expect_tx(sm.s_bar, kHalfBytes);
        tc::bulk_g2s(sm.s_w, q.W_effT, kHalfBytes, sm.s_bar);
    }

    float* curp = sm.s_cur + i;
    uint32_t* maskp = sm.s_mask + warp;
    size_t tro = (size_t)b * T * H + i;
    int t = 0;
    for (; t + 1 < T; t += 2) {
        lean_fwd_step<H, ALIF, kLeanOutSweep, SURR, 0>(p, w, sm.s_z, curp, maskp, tro, v, a, zp, beta);
        lean_fwd_step<H, ALIF, kLeanOutSweep, SURR, 1>(p, w, sm.s_z, curp, maskp, tro, v, a, zp, beta);
    }
    if (t < T) lean_fwd_step<H, ALIF, kLeanOutSweep, SURR, 0>(p, w, sm.s_z, curp, maskp, tro, v, a, zp, beta);
    __syncthreads();

    // the forward's weights are dead: first half of W_effT into registers, the second half's copy overlaps the tail
    tc::mbar_wait(sm.s_bar, 0);
    load_w_cb_half<H>(w, sm.s_w, i, 0);
    tc::fence_proxy_async_smem();
    __syncthreads();
    if (i == 0) {
        tc::mbar_expect_tx(sm.s_bar, kHalfBytes);
        tc::bulk_g2s(sm.s_w, q.W_effT + (size_t)(H / 2) * H, kHalfBytes, sm.s_bar);
    }
    const int ts = fwd_tail_lean<H>(p, sm.s_mask, sm.s_wout, sm.s_s, s_logit, b, i);
    const float g_row = head_tail_lean(p, s_logit, s_hd, s_hp, b, i, H);
    const float seed = i < O ? __fmul_rn(g_row, scale) : 0.f;     // thread c < O: the seed of class c at step ts

    float wo[OP], dwo[OP];
#pragma unroll
    for (int c = 0; c < OP; ++c) {
        wo[c] = sm.s_wout[i * kLeanOP + c];               // zero for c >= O
        dwo[c] = 0.f;
    }
    float* s_g = sm.s_z;                                   // [2][H]
    float* s_gy = sm.s_s;                                  // [T][kOMax]
    for (int idx = i; idx < 2 * H; idx += H) s_g[idx] = 0.f;
    if (run_sums) lean_run_starts(q, s_start, rc_t, rc_p, i);
    lean_gy_scan(q, s_gy, seed, ts, i);
    tc::mbar_wait(sm.s_bar, 1);
    load_w_cb_half<H>(w, sm.s_w, i, 1);
    __syncthreads();

    float gv = 0.f, racc = 0.f;
    uint32_t sbits = 0u;
    size_t gro = ((size_t)b * T + (T - 1)) * H + i;
    const float4* gyp = reinterpret_cast<const float4*>(s_gy + (T - 1) * kOMax);
    const uint32_t* mkp = sm.s_mask + (T - 1) * W32 + warp;
    uint32_t mword = *mkp;                                 // spike word of step t (carried: it is step t+1's "previous")
    const float* sgp = sm.s_cur + (size_t)(T - 1) * H + i;
    auto step = [&](int tt, auto par_tag) {
        constexpr int PAR = decltype(par_tag)::value;
        lean_bwd_step<OP, PLANES, RUNS, PAR>(q, tt, w, wo, dwo, s_g, s_start, run_sums, gyp, mkp, mword, gv, racc, sbits,
                                             crow, gro, [&] { return *sgp; });
        sgp -= H;
    };
    t = T - 1;
    if (!(t & 1)) step(t--, std::integral_constant<int, 0>{});
    for (; t > 0; t -= 2) {
        step(t, std::integral_constant<int, 1>{});
        step(t - 1, std::integral_constant<int, 0>{});
    }
#pragma unroll
    for (int c = 0; c < OP; ++c)
        if (c < O) q.part_wout[((size_t)b * H + i) * O + c] = dwo[c];
}

}  // namespace snnk
