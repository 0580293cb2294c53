// recur_nr.cuh -- K2 / K3 for NON-recurrent layers (use_recurrent_connection = False: BASELINE configs[0] and [2]).
//
// Without the recurrent matmul (spiking_layers.py:164-165 / :234-235 are skipped) a neuron's trajectory depends on its
// own input current only:  V_t = (alpha V_{t-1} + I_t)(1 - Z_{t-1}),  so the time loop is B x H independent scans and
// needs no shared-memory ring, no per-step barrier and no matvec.  The generic kernels (recur_fwd.cuh / recur_bwd.cuh)
// carry all of that machinery through this case too: ncu showed ~250 instructions per warp and step for a 15-operation
// update (31 us + 45 us at B = 256, H = 128).  Here a thread owns one (row, neuron), streams its inputs straight from
// global memory eight steps at a time (the addresses do not depend on the recurrence, so the loads of a block are all
// in flight, one block ahead of their use) and keeps its state in registers.  The leaky readout + max over time (nr_tail) use
// short dependency chains; dW_out / db come from k_gy_scan + k_wout_grad (recur_tc.cuh / recur_gen.cuh) beside the sweep.
//
// Same per-element arithmetic and operation order as the generic kernels (spiking_layers.py:156-171, :229-243;
// spike_funcs.py:59-62 / :75-79): the forward traces are bit-identical to theirs.  LIF and ALIF; tensor-core mode.
#pragma once
#include "common.cuh"
#include "recur_fwd.cuh"

namespace snnk {

constexpr int kNrBlock = 16;     // time steps whose loads are issued together (one block ahead: ~an L2 round trip of compute)

template <int H>
constexpr size_t nonrec_fwd_smem_bytes(int T, int O)
{
    return sizeof(uint32_t) * (size_t)((T * (H / 32) + 3) & ~3) + sizeof(float) * (size_t)((H * O + T * O + 3) & ~3) +
           sizeof(int) * (size_t)((T + 3) & ~3);
}

// Leaky readout + max over time from the T spike words of one row (the job of fwd_tail, recur_fwd.cuh) with short
// dependency chains: one partial sum per 32-neuron word instead of one 128-deep chain (tensor-core mode does not
// promise the oracle's summation order), and a scan whose only loop-carried work is y = (kappa y + s) + b.
template <int H>
__device__ __forceinline__ void nr_tail(const FwdParams& p, const uint32_t* s_mask, const float* s_wout, float* s_s, int b, int tid)
{
    constexpr int W32 = H / 32;
    const int T = p.T, O = p.O;
    for (int idx = tid; idx < T * W32; idx += H) p.zbits[(size_t)b * T * W32 + idx] = s_mask[idx];
    {
        const int tpc = H / O, c = tid / tpc, u = tid - c * tpc;
        if (c < O) {
            float wc[H];
#pragma unroll
            for (int j = 0; j < H; ++j) wc[j] = s_wout[j * O + c];
            for (int t = u; t < T; t += tpc) {
                float part[W32];
#pragma unroll
                for (int wd = 0; wd < W32; ++wd) {
                    const uint32_t m = s_mask[t * W32 + wd];
                    float sum = 0.f;
#pragma unroll
                    for (int l = 0; l < 32; ++l)
                        if (m & (1u << l)) sum = __fadd_rn(sum, wc[wd * 32 + l]);
                    part[wd] = sum;
                }
                float sum = part[0];
#pragma unroll
                for (int wd = 1; wd < W32; ++wd) sum = __fadd_rn(sum, part[wd]);
                s_s[t * O + c] = sum;
            }
        }
    }
    __syncthreads();
    if (tid < O) {
        const int c = tid;
        const float bc = __ldg(p.b_out + c);
        float yv = 0.f, mx = 0.f;
        int mt = 0;
#pragma unroll 4
        for (int t = 0; t < T; ++t) {
            yv = __fadd_rn(__fadd_rn(__fmul_rn(p.kappa, yv), s_s[t * O + c]), bc);      // spiking_layers.py:407
            s_s[t * O + c] = yv;
            if (t == 0 || yv > mx) { mx = yv; mt = t; }                                   // first max wins (snn.py:228)
        }
        p.logits[(size_t)b * O + c] = mx;
        p.tstar[(size_t)b * O + c] = mt;
    }
    __syncthreads();
    for (int idx = tid; idx < T * O; idx += H) p.y[(size_t)b * T * O + idx] = s_s[idx];
}

// grid = B, block = H
template <int H, bool ALIF>
__global__ void __launch_bounds__(H) k_nonrec_fwd(const FwdParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int W32 = H / 32;
    const int T = p.T, O = p.O;
    const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
    const int b = blockIdx.x;
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(smem_raw);                       // [T][W32]
    float* s_wout = reinterpret_cast<float*>(s_mask + ((T * W32 + 3) & ~3));        // [H][O]
    float* s_s = s_wout + H * O;                                                    // [T][O]
    int* s_r2c = reinterpret_cast<int*>(s_wout + ((H * O + T * O + 3) & ~3));       // [T] compact row of every step

    const bool compact = p.run_table != nullptr && p.run_table[1] == 1;
    if (compact) {
        for (int t = i; t < T; t += H) s_r2c[t] = __ldg(p.run_table + kRunHdrInts + (size_t)b * T + t);
        __syncthreads();
    }
    const float* dense = p.I_in + (size_t)b * T * H + i;
    const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
    const size_t s0 = (size_t)b * H + i;
    float v = p.V0 ? p.V0[s0] : 0.f, a = p.a0 ? p.a0[s0] : 0.f, zp = p.Z0 ? p.Z0[s0] : 0.f;
    for (int idx = i; idx < H * O; idx += H) s_wout[idx] = __ldg(p.W_out + idx);
    float* outV = p.V + (size_t)b * T * H + i;
    float* outZ = p.Z + (size_t)b * T * H + i;
    float* outA = p.a + (size_t)b * T * H + i;

    // the loads of block k + 1 are in flight while block k is computed
    auto load_block = [&](int t0, float (&dst)[kNrBlock]) {
#pragma unroll
        for (int u = 0; u < kNrBlock; ++u) {
            const int t = t0 + u;
            dst[u] = 0.f;
            if (t < T) dst[u] = __ldg(compact ? p.I_u + (size_t)s_r2c[t] * H + i : dense + (size_t)t * H);
        }
    };
    float cur[kNrBlock], nxt[kNrBlock];
    load_block(0, cur);
    for (int t0 = 0; t0 < T; t0 += kNrBlock) {
        load_block(t0 + kNrBlock, nxt);
#pragma unroll
        for (int u = 0; u < kNrBlock; ++u) {
            const int t = t0 + u;
            if (t < T) {
                // V' = (alpha V + I_in [+ 0])(1 - Z.detach())     spiking_layers.py:169/239
                const float t1 = __fmul_rn(p.alpha, v);
                const float t2 = __fadd_rn(t1, cur[u]);
                const float t3 = __fadd_rn(t2, 0.0f);
                const float vn = __fmul_rn(t3, __fsub_rn(1.0f, zp));
                float thr = p.theta;
                if constexpr (ALIF) {
                    a = __fadd_rn(__fmul_rn(p.rho, a), zp);             // :240
                    thr = __fadd_rn(p.theta, __fmul_rn(beta, a));       // :241
                }
                const float zn = vn >= thr ? 1.0f : 0.0f;               // spike_funcs.py:27-28
                if (p.traces) {
                    outV[(size_t)t * H] = vn;
                    outZ[(size_t)t * H] = zn;
                    if constexpr (ALIF) outA[(size_t)t * H] = a;
                }
                const unsigned m = __ballot_sync(0xffffffffu, zn != 0.f);
                if (lane == 0) s_mask[t * W32 + warp] = m;
                v = vn;
                zp = zn;
            }
        }
#pragma unroll
        for (int u = 0; u < kNrBlock; ++u) cur[u] = nxt[u];
    }
    __syncthreads();
    nr_tail<H>(p, s_mask, s_wout, s_s, b, i);
}

template <int H>
constexpr size_t nonrec_bwd_smem_bytes(int T)
{
    return sizeof(float) * (size_t)T * kOMax + sizeof(uint32_t) * (size_t)(((T + 1) * (H / 32) + 3) & ~3) +
           sizeof(uint32_t) * (size_t)((T + 31) / 32 + 1);
}

// grid = B, block = H.  gy_scan: (B, T, kOMax) from k_gy_scan.  Writes gI (one or two tf32 planes) and, with a frame-run
// table, the run sums of gI for the compact dW_in contraction.
template <int H, bool ALIF, int SURR>
__global__ void __launch_bounds__(H) k_nonrec_bwd(const BwdParams p, const float* __restrict__ gy_scan)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int W32 = H / 32;
    const int T = p.T, O = p.O;
    const int i = threadIdx.x, lane = i & 31, warp = i >> 5;
    const int b = blockIdx.x;
    float* s_gy = reinterpret_cast<float*>(smem_raw);                                   // [T][kOMax]
    uint32_t* s_zw = reinterpret_cast<uint32_t*>(s_gy + (size_t)T * kOMax);             // [T + 1][W32]: slot 0 = Z_{-1}
    uint32_t* s_start = s_zw + (((T + 1) * W32 + 3) & ~3);                              // run-start bits
    const bool run_sums = p.run_table != nullptr && p.run_table[1] == 1;
    const int TW = (T + 31) / 32 + 1;

    for (int idx = i; idx < T * kOMax / 4; idx += H)
        reinterpret_cast<float4*>(s_gy)[idx] = __ldg(reinterpret_cast<const float4*>(gy_scan + (size_t)b * T * kOMax) + idx);
    for (int idx = i; idx < (T + 1) * W32; idx += H) {
        const int ts = idx / W32, wd = idx - ts * W32;
        uint32_t w = 0u;
        if (ts > 0) w = __ldg(p.zbits + ((size_t)b * T + ts - 1) * W32 + wd);
        else if (p.Z0)
            for (int l = 0; l < 32; ++l)
                if (__ldg(p.Z0 + (size_t)b * H + wd * 32 + l) != 0.f) w |= 1u << l;
        s_zw[idx] = w;
    }
    if (run_sums) {
        for (int idx = i; idx < TW; idx += H) s_start[idx] = 0u;
        __syncthreads();
        const int* rc = p.run_table + kRunHdrInts + (size_t)b * T;
        for (int t = i; t < T; t += H)
            if (t == 0 || __ldg(rc + t) != __ldg(rc + t - 1)) atomicOr(s_start + (t >> 5), 1u << (t & 31));
        if (b == 0) {   // the weight-gradient GEMM contracts whole 32-row blocks: zero the tail of the last one
            const int n_rows = p.run_table[0], n_pad = (n_rows + 31) & ~31;
            for (int idx = i; idx < (n_pad - n_rows) * H; idx += H) {
                p.Gu_hi[(size_t)n_rows * H + idx] = 0.f;
                p.Gu_lo[(size_t)n_rows * H + idx] = 0.f;
            }
        }
    }
    float wo[kOMax];
#pragma unroll
    for (int c = 0; c < kOMax; ++c) wo[c] = c < O ? __ldg(p.W_out + (size_t)i * O + c) : 0.f;
    const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
    __syncthreads();

    const size_t base = (size_t)b * T * H + i;
    float gv = 0.f, racc = 0.f;
    int crow = run_sums ? __ldg(p.run_table + kRunHdrInts + (size_t)b * T + T - 1) : 0;
    auto load_block = [&](int t1, float (&dv)[kNrBlock], float (&da)[kNrBlock]) {
#pragma unroll
        for (int u = 0; u < kNrBlock; ++u) {
            const int t = t1 - u;
            dv[u] = 0.f; da[u] = 0.f;
            if (t >= 0) {
                dv[u] = __ldg(p.V + base + (size_t)t * H);
                if constexpr (ALIF) da[u] = __ldg(p.a + base + (size_t)t * H);
            }
        }
    };
    float vt[kNrBlock], at[kNrBlock], vn[kNrBlock], an[kNrBlock];
    load_block(T - 1, vt, at);
    for (int t1 = T - 1; t1 >= 0; t1 -= kNrBlock) {
        load_block(t1 - kNrBlock, vn, an);      // in flight while this block is computed
#pragma unroll
        for (int u = 0; u < kNrBlock; ++u) {
            const int t = t1 - u;
            if (t >= 0) {
                const float4* gyv = reinterpret_cast<const float4*>(s_gy + t * kOMax);
                float sq[kOMax / 4];
#pragma unroll
                for (int q = 0; q < kOMax / 4; ++q) {      // gy_t W_out^T as four independent chains
                    const float4 g4 = gyv[q];
                    sq[q] = fmaf(g4.w, wo[4 * q + 3], fmaf(g4.z, wo[4 * q + 2], fmaf(g4.y, wo[4 * q + 1], __fmul_rn(g4.x, wo[4 * q]))));
                }
                float s = __fadd_rn(__fadd_rn(sq[0], sq[1]), __fadd_rn(sq[2], sq[3]));
                const size_t o = base + (size_t)t * H;
                if (p.g_Z) s = __fadd_rn(s, __ldg(p.g_Z + o));
                const float zt = (float)((s_zw[(t + 1) * W32 + warp] >> lane) & 1u);
                const float zprev = (float)((s_zw[t * W32 + warp] >> lane) & 1u);
                float thr = p.theta;
                if constexpr (ALIF) thr = __fadd_rn(p.theta, __fmul_rn(beta, at[u]));
                const float sg = surrogate_grad<SURR>(p.gamma, vt[u], thr);
                const float carry = __fmul_rn(__fmul_rn(p.alpha, gv), __fsub_rn(1.0f, zt));
                float g = __fadd_rn(__fmul_rn(s, sg), carry);
                if (p.g_V) g = __fadd_rn(g, __ldg(p.g_V + o));
                gv = g;
                const float gi = __fmul_rn(g, __fsub_rn(1.0f, zprev));
                if (p.gI_lo) {      // exact two-plane tf32 split for the weight-gradient GEMM
                    const float hi = __uint_as_float(__float_as_uint(gi) & 0xFFFFE000u);
                    p.gI[o] = hi;
                    p.gI_lo[o] = __fsub_rn(gi, hi);
                } else {
                    p.gI[o] = gi;
                }
                if (run_sums) {      // sum of gI over the run of equal input frames this step belongs to
                    racc = __fadd_rn(racc, gi);
                    if ((s_start[t >> 5] >> (t & 31)) & 1u) {
                        const float hi = __uint_as_float(__float_as_uint(racc) & 0xFFFFE000u);
                        p.Gu_hi[(size_t)crow * H + i] = hi;
                        p.Gu_lo[(size_t)crow * H + i] = __fsub_rn(racc, hi);
                        racc = 0.f;
                        --crow;
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < kNrBlock; ++u) { vt[u] = vn[u]; at[u] = an[u]; }
    }
}

}  // namespace snnk
