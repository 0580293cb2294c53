// recur_bwd.cuh -- K3: persistent fused reverse-time BPTT.
//
// Replaces what autograd does for batch_loss.backward() (src/modules/snn.py:413) over the graph the
// forward loop builds: per step, MmBackward for the readout and recurrent matmuls, the surrogate
// backward (src/modules/spike_funcs.py:59-62 FastSigmoid, :75-79 Phi), and the Mul/Add backwards of
// spiking_layers.py:169/239.  The reset factor is detached (:169) and the spike threshold receives no
// gradient (spike_funcs.py:62/79), so the adaptation variable and beta are outside the sweep.
//
//   gy_t = seed_t + kappa gy_{t+1}
//   gZ_t = gy_t W_out^T + gI_{t+1} (W_rec . M)^T               [+ seed on Z]
//   gV_t = gZ_t sigma'(V_t, A_t) + alpha gV_{t+1} (1 - Z_t)    [+ seed on V]
//   gI_t = gV_t (1 - Z_{t-1})
//
// (Izhikevich, MODE = 2: the coupled (gV, gu) recurrence stated in the kernel body.)
//
// Same ownership as the forward kernel: one CTA = R batch rows, thread i = neuron i, the ROWS of the
// masked recurrent matrix register-resident and column-blocked over lane quads (dot_rec16_cb on the
// transpose), gI_{t+1} read from shared memory, one __syncthreads per step.  dW_out and db are
// accumulated in registers / a pre-scan and leave as per-CTA partials (summed in a fixed order by
// k_finalize_grads, so results are run-to-run deterministic); dW_in and dW_rec are contractions over
// (batch x time) and belong to the weight-gradient GEMM (K4).  With a frame-run table the sweep also
// leaves the sum of gI over every run of equal input frames (compact rows of the dW_in contraction).
#pragma once
#include "common.cuh"
#include "gemm_tc.cuh"
#include "recur_fwd.cuh"   // kChunk, kRing

namespace snnk {

template <int H, int R>
constexpr size_t bwd_smem_bytes(int T, bool rec)
{
    // the spike-word region is padded to 16 bytes: s_gy behind it is read with float4 loads
    size_t loop = sizeof(float) * (size_t)(2 * R * H) + sizeof(uint32_t) * (size_t)((R * T * (H / 32) + 3) & ~3) +
                  sizeof(float) * (size_t)(R * T * kOMax) + 2 * sizeof(float) * (size_t)(kRing * R * kChunk * H) +
                  sizeof(uint64_t) * kRing + sizeof(int) * (size_t)(R * T);   // + compact row of every step (run sums)
    size_t stage = rec ? sizeof(float) * (size_t)H * H + 16 : 0;   // weight staging + its mbarrier, prologue only
    return loop > stage ? loop : stage;
}

// MODE: 0 LIF, 1 ALIF, 2 Izhikevich; SURR: 0 FastSigmoid, 1 Phi, 2 sigma' trace -- compile-time for the same reason as
// in k_recur_fwd.  With the trace, LIF / ALIF run MODE 0 with sigma' in the V slot; Izhikevich streams sigma' from `a`.
template <int H, int R, bool REC, int MODE = 1, int SURR = 0>
__global__ void __launch_bounds__(H, 256 / H) k_recur_bwd(const BwdParams p)
{
    constexpr bool IZH = MODE == 2, ALIF = MODE == 1;
    constexpr bool TWO = ALIF || (IZH && SURR == kSurrTrace);   // a second trace streams beside V
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int W32 = H / 32;
    const int T = p.T, O = p.O, B = p.B;
    const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
    const int b0 = blockIdx.x * R;
    const int nvalid = min(R, B - b0);

    // row i of W_rec (.) rec_mask = column i of its transpose (k_prep_rec), staged by ONE bulk copy through shared
    // memory (the staging area aliases the loop buffers, which are initialised afterwards)
    float w[REC ? H : 16];
    if constexpr (REC) {
        float* s_t = reinterpret_cast<float*>(smem_raw);                        // [H][H]
        uint64_t* wbar = reinterpret_cast<uint64_t*>(s_t + H * H);
        if (i == 0) {
            tc::mbar_init(wbar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            tc::mbar_expect_tx(wbar, (uint32_t)(H * H * sizeof(float)));
            tc::bulk_g2s(s_t, p.W_effT, (uint32_t)(H * H * sizeof(float)), wbar);
        }
        __syncthreads();
        tc::mbar_wait(wbar, 0);
        load_w_cb<REC ? H : 16>(w, s_t, i);
        // the ring's bulk copies (async proxy) will land in this area: order the generic-proxy reads above before them
        // (a barrier alone does not order the two proxies; recur_lean.cuh has the observed failure)
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (i == 0) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(tc::smem_u32(wbar)) : "memory");
    }

    float* s_g = reinterpret_cast<float*>(smem_raw);                       // [2][R][H]
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(s_g + 2 * R * H);       // [R][T][W32]
    float* s_gy = reinterpret_cast<float*>(s_mask + ((R * T * W32 + 3) & ~3));   // [R][T][kOMax], 16-B aligned
    float* s_v = s_gy + R * T * kOMax;                                           // [kRing][R][kChunk][H]  V trace ring
    float* s_a = s_v + kRing * R * kChunk * H;                                   // [kRing][R][kChunk][H]  a / sigma' ring
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_a + kRing * R * kChunk * H); // [kRing]
    uint32_t* s_start = reinterpret_cast<uint32_t*>(s_bar + kRing);              // [R][ceil(T/32)] run-start bits
    const bool run_sums = p.run_table != nullptr && p.run_table[1] == 1;
    const int TW = (T + 31) >> 5;

    // The saved traces are streamed backwards in time through the ring by 1-D bulk async copies; chunk k (in
    // processing order) covers forward chunk nchunks-1-k.  Thread 0 only.
    const int nchunks = (T + kChunk - 1) / kChunk;
    auto issue_chunk = [&](int k) {
        const int slot = k % kRing, t0 = (nchunks - 1 - k) * kChunk;
        const uint32_t bytes = (uint32_t)(min(kChunk, T - t0) * H * sizeof(float));
        tc::mbar_expect_tx(s_bar + slot, bytes * nvalid * (TWO ? 2 : 1));
        for (int r = 0; r < nvalid; ++r) {
            const size_t g = ((size_t)(b0 + r) * T + t0) * H;
            tc::bulk_g2s(s_v + ((slot * R + r) * kChunk) * H, p.V + g, bytes, s_bar + slot);
            if (TWO) tc::bulk_g2s(s_a + ((slot * R + r) * kChunk) * H, p.a + g, bytes, s_bar + slot);
        }
    };
    if (i == 0) {   // the staging area above aliases the ring: the first copies start only now
        for (int s = 0; s < kRing; ++s) tc::mbar_init(s_bar + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int k = 0; k < kRing && k < nchunks; ++k) issue_chunk(k);
    }

    float wo[kOMax], dwo[kOMax];
#pragma unroll
    for (int c = 0; c < kOMax; ++c) {
        wo[c] = c < O ? __ldg(p.W_out + (size_t)i * O + c) : 0.f;
        dwo[c] = 0.f;
    }
    const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;

    for (int idx = i; idx < 2 * R * H; idx += H) s_g[idx] = 0.f;
    for (int idx = i; idx < R * T * kOMax; idx += H) s_gy[idx] = 0.f;
    for (int idx = i; idx < R * T * W32; idx += H) {
        const int r = idx / (T * W32), rem = idx - r * (T * W32);
        s_mask[idx] = (b0 + r < B) ? __ldg(p.zbits + (size_t)(b0 + r) * T * W32 + rem) : 0u;
    }
    if (run_sums) {
        // bit t of a row's word: step t is the first of its run of equal input frames (its compact row differs from t-1's)
        for (int idx = i; idx < R * TW; idx += H) s_start[idx] = 0u;
        __syncthreads();
        for (int idx = i; idx < nvalid * T; idx += H) {
            const int r = idx / T, t = idx - r * T;
            const int* rc = p.run_table + kRunHdrInts + (size_t)(b0 + r) * T;
            if (t == 0 || __ldg(rc + t) != __ldg(rc + t - 1)) atomicOr(s_start + r * TW + (t >> 5), 1u << (t & 31));
        }
        if (blockIdx.x == 0) {   // the weight-gradient GEMM contracts whole 32-row blocks: zero the tail of the last one
            const int n_rows = p.run_table[0], n_pad = (n_rows + 31) & ~31;
            for (int idx = i; idx < (n_pad - n_rows) * H; idx += H) {
                p.Gu_hi[(size_t)n_rows * H + idx] = 0.f;
                p.Gu_lo[(size_t)n_rows * H + idx] = 0.f;
            }
        }
    }
    __syncthreads();
    if (p.g_y) {
        for (int idx = i; idx < R * T * O; idx += H) {
            const int r = idx / (T * O), rem = idx - r * (T * O);
            const int t = rem / O, c = rem - t * O;
            if (b0 + r < B) s_gy[(r * T + t) * kOMax + c] = __ldg(p.g_y + (size_t)(b0 + r) * T * O + rem);
        }
    } else {
        const float scale = p.g_scale ? __ldg(p.g_scale) : 1.0f;
        for (int idx = i; idx < R * O; idx += H) {
            const int r = idx / O, c = idx - r * O;
            if (b0 + r < B) {
                const int ts = __ldg(p.tstar + (size_t)(b0 + r) * O + c);
                s_gy[(r * T + ts) * kOMax + c] = __fmul_rn(__ldg(p.g_logits + (size_t)(b0 + r) * O + c), scale);
            }
        }
    }
    __syncthreads();
    // readout adjoint scan gy_t = seed_t + kappa gy_{t+1}  (spiking_layers.py:407 backwards) and db
    for (int idx = i; idx < R * O; idx += H) {
        const int r = idx / O, c = idx - r * O;
        float g = 0.f, sum = 0.f;
        for (int t = T - 1; t >= 0; --t) {
            float* gp = s_gy + (r * T + t) * kOMax + c;
            g = __fadd_rn(*gp, __fmul_rn(p.kappa, g));
            *gp = g;
            sum += g;
        }
        p.part_db[((size_t)blockIdx.x * R + r) * O + c] = sum;
    }
    __syncthreads();

    float gv[R], gu[R], racc[R];
    int crow[R];          // compact row of the run the sweep is in (run sums)
    uint32_t sbits[R];    // run-start bits of the current 32-step window
    bool valid[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        gv[r] = 0.f;
        gu[r] = 0.f;      // Izhikevich: adjoint of the recovery variable
        racc[r] = 0.f;
        valid[r] = b0 + r < B;
        crow[r] = (run_sums && valid[r]) ? __ldg(p.run_table + kRunHdrInts + (size_t)(b0 + r) * T + T - 1) : 0;
        sbits[r] = 0u;
    }

    for (int t = T - 1; t >= 0; --t) {
        {
            {
                const int ck = t / kChunk, tt = t - ck * kChunk;
                const int k = nchunks - 1 - ck, slot = k % kRing;
                if (t == T - 1 || tt == kChunk - 1) {
                    // all threads are past their last read of chunk k-1 (REC: the step barrier), refill its slot
                    if (!REC) __syncthreads();
                    if (i == 0 && k >= 1 && k - 1 + kRing < nchunks) issue_chunk(k - 1 + kRing);
                    tc::mbar_wait(s_bar + slot, (k / kRing) & 1);
                }
                float vt[R], at[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const int o = ((slot * R + r) * kChunk + tt) * H + i;
                    vt[r] = valid[r] ? s_v[o] : 0.f;
                    at[r] = (valid[r] && TWO) ? s_a[o] : 0.f;
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float4* gyv = reinterpret_cast<const float4*>(s_gy + (r * T + t) * kOMax);
                    float gy[kOMax];
#pragma unroll
                    for (int q = 0; q < kOMax / 4; ++q) {
                        const float4 g4 = gyv[q];
                        gy[4 * q + 0] = g4.x; gy[4 * q + 1] = g4.y; gy[4 * q + 2] = g4.z; gy[4 * q + 3] = g4.w;
                    }
                    const float zt = (float)((s_mask[(r * T + t) * W32 + warp] >> lane) & 1u);
                    float zprev;
                    if (t > 0) zprev = (float)((s_mask[(r * T + t - 1) * W32 + warp] >> lane) & 1u);
                    else zprev = (valid[r] && p.Z0) ? __ldg(p.Z0 + (size_t)(b0 + r) * H + i) : 0.f;
                    float s = 0.f;
#pragma unroll
                    for (int c = 0; c < kOMax; ++c) {
                        s = fmaf(gy[c], wo[c], s);               // gy_t W_out^T
                        dwo[c] = fmaf(zt, gy[c], dwo[c]);        // dW_out += Z_t^T gy_t
                    }
                    if constexpr (REC) {
                        const float4* gv4 =
                            reinterpret_cast<const float4*>(s_g + ((t + 1) & 1) * R * H + r * H);
                        s = __fadd_rn(s, dot_rec16_cb<REC ? H : 16>(w, gv4, i & 3));   // gI_{t+1} (W_rec . M)^T
                    }
                    const size_t o = ((size_t)(valid[r] ? b0 + r : 0) * T + t) * H + i;
                    if (p.g_Z && valid[r]) s = __fadd_rn(s, __ldg(p.g_Z + o));
                    float g, gi_scale = 1.0f;
                    if constexpr (IZH) {
                        // adjoint of spiking_layers.py:345-348 (operation order of oracle/snn_oracle.c):
                        //   dV'/dV = (1 + dt k ((V-vr) + (V-vth)) / C)(1-Z)   dV'/du = -(dt/C)(1-Z)   dV'/dI = (dt/C)(1-Z)
                        //   du'/dV = dt a b                                    du'/du = 1 - dt a
                        const float v = vt[r];
                        const float sg = surrogate_grad<SURR>(p.gamma, SURR == kSurrTrace ? at[r] : v, p.iz.vpeak);
                        const float dq = __fmul_rn(p.iz.k, __fadd_rn(__fsub_rn(v, p.iz.vr), __fsub_rn(v, p.iz.vth)));
                        const float A = __fmul_rn(__fadd_rn(1.0f, __fdiv_rn(__fmul_rn(p.iz.dt, dq), p.iz.C)), __fsub_rn(1.0f, zt));
                        const float dtC = __fdiv_rn(p.iz.dt, p.iz.C);
                        g = __fadd_rn(__fadd_rn(__fmul_rn(s, sg), __fmul_rn(gv[r], A)),
                                      __fmul_rn(gu[r], __fmul_rn(__fmul_rn(p.iz.dt, p.iz.a), p.iz.b)));
                        if (p.g_V && valid[r]) g = __fadd_rn(g, __ldg(p.g_V + o));
                        gu[r] = __fadd_rn(__fmul_rn(__fmul_rn(gv[r], -dtC), __fsub_rn(1.0f, zt)),
                                          __fmul_rn(gu[r], __fsub_rn(1.0f, __fmul_rn(p.iz.dt, p.iz.a))));
                        gi_scale = dtC;
                    } else {
                        float thr = p.theta;
                        if (ALIF) thr = __fadd_rn(p.theta, __fmul_rn(beta, at[r]));
                        const float sg = surrogate_grad<SURR>(p.gamma, vt[r], thr);
                        const float carry = __fmul_rn(__fmul_rn(p.alpha, gv[r]), __fsub_rn(1.0f, zt));
                        g = __fadd_rn(__fmul_rn(s, sg), carry);
                        if (p.g_V && valid[r]) g = __fadd_rn(g, __ldg(p.g_V + o));
                    }
                    gv[r] = g;
                    const float gi = IZH ? __fmul_rn(__fmul_rn(g, gi_scale), __fsub_rn(1.0f, zprev))
                                             : __fmul_rn(g, __fsub_rn(1.0f, zprev));
                    if (valid[r]) {
                        if (p.gI_lo) {   // tensor-core mode: exact two-plane tf32 split for the weight-gradient GEMM
                            const float hi = __uint_as_float(__float_as_uint(gi) & 0xFFFFE000u);
                            p.gI[o] = hi;
                            p.gI_lo[o] = __fsub_rn(gi, hi);
                        } else {
                            p.gI[o] = gi;
                        }
                    }
                    if (REC) s_g[(t & 1) * R * H + r * H + i] = gi;
                    if (run_sums) {   // sum of gI over the run of equal input frames this step belongs to
                        racc[r] = __fadd_rn(racc[r], gi);
                        if (t == T - 1 || (t & 31) == 31) sbits[r] = s_start[r * TW + (t >> 5)];
                        if ((sbits[r] >> (t & 31)) & 1u) {
                            if (valid[r]) {
                                const float hi = __uint_as_float(__float_as_uint(racc[r]) & 0xFFFFE000u);
                                p.Gu_hi[(size_t)crow[r] * H + i] = hi;
                                p.Gu_lo[(size_t)crow[r] * H + i] = __fsub_rn(racc[r], hi);
                            }
                            racc[r] = 0.f;
                            --crow[r];
                        }
                    }
                }
                if (REC) __syncthreads();
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kOMax; ++c)
        if (c < O) p.part_wout[((size_t)blockIdx.x * H + i) * O + c] = dwo[c];
}

// ---- gradient finalisation: every split-K / per-CTA partial buffer reduced in ONE launch ------------------------
// All sums run in a fixed order (ascending partial index per lane, then a fixed shuffle tree), so the gradients
// are run-to-run deterministic.  Loads are issued in independent batches so the kernel is bandwidth- rather than
// latency-bound.
struct FinalizeParams {
    // (a) thread per element, few partials:  dW_in (n_in elements) then dW_rec (n_rec elements, masked)
    const float* pw; int S; size_t w_stride; int n_in; int n_rec; const float* rec_mask;
    float* dW_in; float* dW_rec;
    // frame-dedup variant (runs.cuh): when run_table says ok, dW_rec comes from its own partial buffer instead
    const int* run_table; const float* pw_rec; int S_rec; size_t rec_stride;
    int S_cmp;   // number of dW_in partials the compact GEMM wrote (same buffer and stride as the dense ones)
    // The tcgen05 GEMMs read Z_{-1} as zeros (TMA fills t < 0), so the Z0 term of dW_rec is added here:
    // dW_rec[j][n] += sum_b Z0[b][j] (gI + gI_lo)[b, 0, n].  Z0 is null when the partials already hold it (SIMT K4);
    // a raised inexact flag means k_wgrad_simt redid them, Z0 included.
    const float* Z0; const float* gI; const float* gI_lo; const unsigned int* inexact_flag; int B, H; size_t row_stride;
    // (b) warp per element, many partials:   dW_out (n_out elements, P_out partials) then db (n_b, P_b partials)
    const float* pwout; int P_out; int n_out; float* dW_out;
    const float* pdb; int P_b; int n_b; float* db;
    int blocks_a;   // blocks [0, blocks_a) do (a), the rest do (b)
};

__device__ __forceinline__ float sum_partials_seq(const float* __restrict__ base, int nparts, size_t stride)
{
    // ascending order, loads issued 32 (then 8) at a time: the dW_rec-only GEMM of the dedup variant leaves 128 partials
    // and a chain of 8-load batches was the critical path of this kernel
    float s = 0.f;
    int q = 0;
    // (one batch of 128 spills under this kernel's 256-thread launch bound: 16.4 us against 11.4 us)
    for (; q + 64 <= nparts; q += 64) {      // two round trips instead of four for the 128 partials of dW_rec
        float v[64];
#pragma unroll
        for (int j = 0; j < 64; ++j) v[j] = __ldg(base + (size_t)(q + j) * stride);
#pragma unroll
        for (int j = 0; j < 64; ++j) s += v[j];
    }
    for (; q + 32 <= nparts; q += 32) {
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __ldg(base + (size_t)(q + j) * stride);
#pragma unroll
        for (int j = 0; j < 32; ++j) s += v[j];
    }
    for (; q + 8 <= nparts; q += 8) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldg(base + (size_t)(q + j) * stride);
#pragma unroll
        for (int j = 0; j < 8; ++j) s += v[j];
    }
    for (; q < nparts; ++q) s += __ldg(base + (size_t)q * stride);
    return s;
}

__global__ void __launch_bounds__(256) k_finalize_grads(const FinalizeParams p)
{
    if ((int)blockIdx.x < p.blocks_a) {
        const int e = blockIdx.x * blockDim.x + threadIdx.x;
        const bool compact = p.run_table && p.run_table[1] == 1;
        if (e < p.n_in) {
            p.dW_in[e] = sum_partials_seq(p.pw + e, compact ? p.S_cmp : p.S, p.w_stride);
        } else if (e - p.n_in < p.n_rec) {
            const int r = e - p.n_in;
            float s = (compact && p.pw_rec) ? sum_partials_seq(p.pw_rec + r, p.S_rec, p.rec_stride)
                              : sum_partials_seq(p.pw + p.n_in + r, p.S, p.w_stride);
            if (p.Z0 && !(p.inexact_flag && *p.inexact_flag != 0)) {
                const int j = r / p.H, n = r - j * p.H;
                float c = 0.f;
                for (int b = 0; b < p.B; ++b) {
                    const size_t g = (size_t)b * p.row_stride + n;
                    c = fmaf(__ldg(p.Z0 + (size_t)b * p.H + j), __ldg(p.gI + g) + __ldg(p.gI_lo + g), c);
                }
                s += c;
            }
            p.dW_rec[r] = p.rec_mask ? s * __ldg(p.rec_mask + r) : s;
        }
        return;
    }
    const int warp = (blockIdx.x - p.blocks_a) * (blockDim.x / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const float* base; int nparts, n; float* out; int e;
    if (warp < p.n_out) { base = p.pwout; nparts = p.P_out; n = p.n_out; out = p.dW_out; e = warp; }
    else if (warp - p.n_out < p.n_b) { base = p.pdb; nparts = p.P_b; n = p.n_b; out = p.db; e = warp - p.n_out; }
    else return;
    float s = 0.f;
    for (int q = lane; q < nparts; q += 32) s += __ldg(base + (size_t)q * n + e);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[e] = s;
}

}  // namespace snnk
