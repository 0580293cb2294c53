// recur_gen.cuh -- the recurrence kernels for wide hidden layers (128 < H <= 2048, H a multiple of 128).
//
// Same algorithm, same summation orders and therefore the same bits as recur_fwd.cuh / recur_bwd.cuh; what
// changes is residency: an H x H fp32 recurrent matrix (4 MB at H = 1024) no longer fits in registers or
// shared memory, so it is streamed from L2 once per step and per CTA and amortised over the R batch rows a
// CTA owns (thread = neuron, R rows, sixteen accumulation chains evaluated one after the other, previous spike / gradient vector
// broadcast from shared memory as one LDS per k for all R rows).  The leaky readout and dW_out, which in the
// narrow kernels ride along in registers / shared memory, become two small separate kernels here
// (k_readout_scan, k_wout_grad).
//
// This is the functional wide path (BASELINE configs[3] and [4]); its recurrent matvec runs on the fp32 pipes and
// re-reads W from L2 every step.  The weight-stationary tensor-core version is SURVEY.md section 7 item 8.
#pragma once
#include "common.cuh"

namespace snnk {

constexpr int kGenMaxThreads = 1024;

__host__ __device__ constexpr int gen_npt(int H) { return (H + kGenMaxThreads - 1) / kGenMaxThreads; }
__host__ __device__ constexpr int gen_rows(int H) { return gen_npt(H) == 1 ? 4 : 2; }

// acc[j][r] = sum over k = c, c+16, ... of Wm[k][i_j] * vec[k][r]   for one accumulation chain c
template <int NPT, int R>
__device__ __forceinline__ void chain_dot(const float* __restrict__ Wm, const float* __restrict__ s_vec, int H, int BD,
                                          int tid, int c, float (&acc)[NPT][R])
{
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) acc[j][r] = 0.f;
#pragma unroll 4
    for (int k = c; k < H; k += 16) {
        float z[R];
        if constexpr (R == 4) {
            const float4 z4 = *reinterpret_cast<const float4*>(s_vec + k * 4);
            z[0] = z4.x; z[1] = z4.y; z[2] = z4.z; z[3] = z4.w;
        } else {
            const float2 z2 = *reinterpret_cast<const float2*>(s_vec + k * 2);
            z[0] = z2.x; z[1] = z2.y;
        }
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const float w = __ldg(Wm + (size_t)k * H + tid + j * BD);
#pragma unroll
            for (int r = 0; r < R; ++r) acc[j][r] = fmaf(w, z[r], acc[j][r]);
        }
    }
}

// Sum of the eight chains c0 .. c0+7 as the balanced tree ((s0+s1)+(s2+s3))+((s4+s5)+(s6+s7)).
template <int NPT, int R>
__device__ __forceinline__ void tree8(const float* __restrict__ Wm, const float* __restrict__ s_vec, int H, int BD, int tid,
                                      int c0, float (&out)[NPT][R])
{
    float a[NPT][R], b[NPT][R], u[NPT][R];
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 0, a);
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 1, b);
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) u[j][r] = __fadd_rn(a[j][r], b[j][r]);
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 2, a);
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 3, b);
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) u[j][r] = __fadd_rn(u[j][r], __fadd_rn(a[j][r], b[j][r]));
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 4, a);
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 5, b);
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) out[j][r] = __fadd_rn(a[j][r], b[j][r]);
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 6, a);
    chain_dot<NPT, R>(Wm, s_vec, H, BD, tid, c0 + 7, b);
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r)
            out[j][r] = __fadd_rn(u[j][r], __fadd_rn(out[j][r], __fadd_rn(a[j][r], b[j][r])));
}

// Full dot product in the oracle's order: sixteen chains over k mod 16, balanced tree over adjacent chains.
template <int NPT, int R>
__device__ __forceinline__ void dot_rec16_gen(const float* __restrict__ Wm, const float* __restrict__ s_vec, int H, int BD,
                                              int tid, float (&out)[NPT][R])
{
    float lo[NPT][R];
    tree8<NPT, R>(Wm, s_vec, H, BD, tid, 0, lo);
    tree8<NPT, R>(Wm, s_vec, H, BD, tid, 8, out);
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) out[j][r] = __fadd_rn(lo[j][r], out[j][r]);
}

// ---- forward --------------------------------------------------------------------------------------------------------
// grid = ceil(B / R), block = H / NPT threads, dynamic smem = 2 * H * R floats
template <int NPT, int R, bool REC>
__global__ void __launch_bounds__(kGenMaxThreads) k_recur_fwd_gen(const FwdParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* s_z = reinterpret_cast<float*>(smem_raw);          // [2][H][R]: spike vectors of the R rows, row-interleaved
    const int T = p.T, B = p.B, H = p.H, BD = blockDim.x;
    const int tid = threadIdx.x, lane = tid & 31;
    const int b0 = blockIdx.x * R;
    const float beta = (p.alif && p.beta) ? __ldg(p.beta) : 0.f;

    float v[NPT][R], a[NPT][R], zp[NPT][R];
    bool valid[R];
#pragma unroll
    for (int r = 0; r < R; ++r) valid[r] = b0 + r < B;
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int i = tid + j * BD;
            const size_t s = (size_t)(valid[r] ? b0 + r : 0) * H + i;
            v[j][r] = (valid[r] && p.V0) ? p.V0[s] : (p.iz.on ? p.iz.vr : 0.f);   // Izhikevich starts at v_rest (:309)
            a[j][r] = (valid[r] && p.a0) ? p.a0[s] : 0.f;
            zp[j][r] = (valid[r] && p.Z0) ? p.Z0[s] : 0.f;
            if (REC) s_z[(1 * H + i) * R + r] = zp[j][r];
        }
    __syncthreads();

    for (int t = 0; t < T; ++t) {
        float cur[NPT][R];
#pragma unroll
        for (int j = 0; j < NPT; ++j)
#pragma unroll
            for (int r = 0; r < R; ++r)
                cur[j][r] = valid[r] ? __ldg(p.I_in + ((size_t)(b0 + r) * T + t) * H + tid + j * BD) : 0.f;
        float rec[NPT][R];
        if constexpr (REC) {
            dot_rec16_gen<NPT, R>(p.W_eff, s_z + ((t + 1) & 1) * H * R, H, BD, tid, rec);
        } else {
#pragma unroll
            for (int j = 0; j < NPT; ++j)
#pragma unroll
                for (int r = 0; r < R; ++r) rec[j][r] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const int i = tid + j * BD;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                // identical arithmetic to k_recur_fwd (spiking_layers.py:169/239-242; Izhikevich :344-349)
                float vn, thr = p.theta;
                if (p.iz.on) {
                    const float I = __fadd_rn(cur[j][r], rec[j][r]);
                    const float d1 = __fsub_rn(v[j][r], p.iz.vr), d2 = __fsub_rn(v[j][r], p.iz.vth);
                    const float q = __fsub_rn(__fmul_rn(__fmul_rn(p.iz.k, d1), d2), a[j][r]);
                    const float inc = __fdiv_rn(__fmul_rn(p.iz.dt, __fadd_rn(q, I)), p.iz.C);
                    vn = __fadd_rn(__fmul_rn(__fadd_rn(v[j][r], inc), __fsub_rn(1.0f, zp[j][r])), __fmul_rn(p.iz.c, zp[j][r]));
                    const float du = __fmul_rn(p.iz.a, __fsub_rn(__fmul_rn(p.iz.b, d1), a[j][r]));
                    a[j][r] = __fadd_rn(__fadd_rn(a[j][r], __fmul_rn(p.iz.dt, du)), __fmul_rn(p.iz.d, zp[j][r]));
                    thr = p.iz.vpeak;
                } else {
                    const float t1 = __fmul_rn(p.alpha, v[j][r]);
                    const float t2 = __fadd_rn(t1, cur[j][r]);
                    const float t3 = __fadd_rn(t2, rec[j][r]);
                    vn = __fmul_rn(t3, __fsub_rn(1.0f, zp[j][r]));
                    if (p.alif) {
                        a[j][r] = __fadd_rn(__fmul_rn(p.rho, a[j][r]), zp[j][r]);
                        thr = __fadd_rn(p.theta, __fmul_rn(beta, a[j][r]));
                    }
                }
                const float zn = vn >= thr ? 1.0f : 0.0f;
                const unsigned m = __ballot_sync(0xffffffffu, zn != 0.f);
                if (valid[r]) {
                    const size_t o = ((size_t)(b0 + r) * T + t) * H + i;
                    if (p.traces) {
                        p.V[o] = vn;
                        p.Z[o] = zn;
                        if (p.alif || p.iz.on) p.a[o] = a[j][r];
                    }
                    if (lane == 0) p.zbits[((size_t)(b0 + r) * T + t) * (H / 32) + (i >> 5)] = m;
                }
                if (REC) s_z[((t & 1) * H + i) * R + r] = zn;
                v[j][r] = vn;
                zp[j][r] = zn;
            }
        }
        if (REC) __syncthreads();
    }
}

// Leaky readout + max over time from the bit-packed raster (same arithmetic and order as the tail of k_recur_fwd).
// grid = B, block = 128, dynamic smem = T*H/32 words + H*O + T*O floats
__global__ void __launch_bounds__(128) k_readout_scan(int T, int H, int O, float kappa, const uint32_t* __restrict__ zbits,
                                                     const float* __restrict__ W_out, const float* __restrict__ b_out,
                                                     float* __restrict__ y, float* __restrict__ logits,
                                                     int32_t* __restrict__ tstar)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int W32 = H / 32, i = threadIdx.x, b = blockIdx.x;
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(smem_raw);       // [T][W32]
    float* s_wout = reinterpret_cast<float*>(s_mask + T * W32);     // [H][O]
    float* s_s = s_wout + H * O;                                    // [T][O]
    for (int idx = i; idx < T * W32; idx += blockDim.x) s_mask[idx] = __ldg(zbits + (size_t)b * T * W32 + idx);
    for (int idx = i; idx < H * O; idx += blockDim.x) s_wout[idx] = __ldg(W_out + idx);
    __syncthreads();
    for (int idx = i; idx < T * O; idx += blockDim.x) {
        const int t = idx / O, c = idx - t * O;
        const uint32_t* mw = s_mask + t * W32;
        float s = 0.f;
        for (int wd = 0; wd < W32; ++wd) {
            const uint32_t m = mw[wd];
#pragma unroll 8
            for (int l = 0; l < 32; ++l) {
                const float wv = s_wout[(wd * 32 + l) * O + c];
                s = __fadd_rn(s, ((m >> l) & 1u) ? wv : 0.f);
            }
        }
        s_s[idx] = s;
    }
    __syncthreads();
    for (int c = i; c < O; c += blockDim.x) {
        const float bc = __ldg(b_out + c);
        float yv = 0.f, mx = 0.f;
        int mt = 0;
        for (int t = 0; t < T; ++t) {
            yv = __fadd_rn(__fadd_rn(__fmul_rn(kappa, yv), s_s[t * O + c]), bc);
            s_s[t * O + c] = yv;
            if (t == 0 || yv > mx) { mx = yv; mt = t; }
        }
        logits[(size_t)b * O + c] = mx;
        tstar[(size_t)b * O + c] = mt;
    }
    __syncthreads();
    for (int idx = i; idx < T * O; idx += blockDim.x) y[(size_t)b * T * O + idx] = s_s[idx];
}

// ---- backward -------------------------------------------------------------------------------------------------------
// grid = ceil(B / R), block = H / NPT, dynamic smem = 2*H*R floats + R*T*kOMax floats.
// Writes gI (one or two tf32 planes) and the scanned readout adjoint gy (B,T,kOMax) for k_wout_grad.
// TRACE: surrogate SNNK_SURROGATE_TRACE -- sigma' is read from the V slot (LIF / ALIF, run as LIF) or from `a` (Izhikevich).
template <int NPT, int R, bool REC, bool TRACE = false>
__global__ void __launch_bounds__(kGenMaxThreads) k_recur_bwd_gen(const BwdParams p, float* __restrict__ gy_scan)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int T = p.T, B = p.B, H = p.H, O = p.O, BD = blockDim.x, W32 = H / 32;
    const int tid = threadIdx.x, lane = tid & 31;
    const int b0 = blockIdx.x * R;
    float* s_g = reinterpret_cast<float*>(smem_raw);      // [2][H][R]
    float* s_gy = s_g + 2 * H * R;                         // [R][T][kOMax]
    const float beta = (p.alif && p.beta) ? __ldg(p.beta) : 0.f;

    for (int idx = tid; idx < 2 * H * R; idx += BD) s_g[idx] = 0.f;
    for (int idx = tid; idx < R * T * kOMax; idx += BD) s_gy[idx] = 0.f;
    __syncthreads();
    if (p.g_y) {
        for (int idx = tid; idx < R * T * O; idx += BD) {
            const int r = idx / (T * O), rem = idx - r * (T * O);
            const int t = rem / O, c = rem - t * O;
            if (b0 + r < B) s_gy[(r * T + t) * kOMax + c] = __ldg(p.g_y + (size_t)(b0 + r) * T * O + rem);
        }
    } else {
        const float scale = p.g_scale ? __ldg(p.g_scale) : 1.0f;
        for (int idx = tid; idx < R * O; idx += BD) {
            const int r = idx / O, c = idx - r * O;
            if (b0 + r < B) {
                const int ts = __ldg(p.tstar + (size_t)(b0 + r) * O + c);
                s_gy[(r * T + ts) * kOMax + c] = __fmul_rn(__ldg(p.g_logits + (size_t)(b0 + r) * O + c), scale);
            }
        }
    }
    __syncthreads();
    for (int idx = tid; idx < R * O; idx += BD) {
        const int r = idx / O, c = idx - r * O;
        float g = 0.f;
        for (int t = T - 1; t >= 0; --t) {
            float* gp = s_gy + (r * T + t) * kOMax + c;
            g = __fadd_rn(*gp, __fmul_rn(p.kappa, g));
            *gp = g;
        }
    }
    __syncthreads();
    for (int idx = tid; idx < R * T * kOMax; idx += BD) {
        const int r = idx / (T * kOMax), rem = idx - r * (T * kOMax);
        if (b0 + r < B) gy_scan[(size_t)(b0 + r) * T * kOMax + rem] = s_gy[idx];
    }

    float gv[NPT][R], gu[NPT][R];      // gu: adjoint of the Izhikevich recovery variable
    bool valid[R];
#pragma unroll
    for (int r = 0; r < R; ++r) valid[r] = b0 + r < B;
#pragma unroll
    for (int j = 0; j < NPT; ++j)
#pragma unroll
        for (int r = 0; r < R; ++r) gv[j][r] = gu[j][r] = 0.f;

    for (int t = T - 1; t >= 0; --t) {
        float rec[NPT][R];
        if constexpr (REC) {
            dot_rec16_gen<NPT, R>(p.W_effT, s_g + ((t + 1) & 1) * H * R, H, BD, tid, rec);
        } else {
#pragma unroll
            for (int j = 0; j < NPT; ++j)
#pragma unroll
                for (int r = 0; r < R; ++r) rec[j][r] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < NPT; ++j) {
            const int i = tid + j * BD;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const size_t row = (size_t)(valid[r] ? b0 + r : 0) * T + t;
                const size_t o = row * H + i;
                const uint32_t mt = valid[r] ? __ldg(p.zbits + row * W32 + (i >> 5)) : 0u;
                const float zt = (float)((mt >> lane) & 1u);
                float zprev;
                if (t > 0) zprev = valid[r] ? (float)((__ldg(p.zbits + (row - 1) * W32 + (i >> 5)) >> lane) & 1u) : 0.f;
                else zprev = (valid[r] && p.Z0) ? __ldg(p.Z0 + (size_t)(b0 + r) * H + i) : 0.f;
                const float* gy = s_gy + (r * T + t) * kOMax;
                float s = 0.f;
                for (int c = 0; c < O; ++c) s = fmaf(gy[c], __ldg(p.W_out + (size_t)i * O + c), s);
                if (REC) s = __fadd_rn(s, rec[j][r]);
                if (p.g_Z && valid[r]) s = __fadd_rn(s, __ldg(p.g_Z + o));
                const float vt = valid[r] ? __ldg(p.V + o) : 0.f;
                float g, gi;
                if (p.iz.on) {
                    // the coupled (gV, gu) adjoint of spiking_layers.py:345-348, operation order of k_recur_bwd
                    const float sg = TRACE ? (valid[r] ? __ldg(p.a + o) : 0.f)
                                           : surrogate_grad(p.surrogate, p.gamma, vt, p.iz.vpeak);
                    const float dq = __fmul_rn(p.iz.k, __fadd_rn(__fsub_rn(vt, p.iz.vr), __fsub_rn(vt, p.iz.vth)));
                    const float A = __fmul_rn(__fadd_rn(1.0f, __fdiv_rn(__fmul_rn(p.iz.dt, dq), p.iz.C)), __fsub_rn(1.0f, zt));
                    const float dtC = __fdiv_rn(p.iz.dt, p.iz.C);
                    g = __fadd_rn(__fadd_rn(__fmul_rn(s, sg), __fmul_rn(gv[j][r], A)),
                                  __fmul_rn(gu[j][r], __fmul_rn(__fmul_rn(p.iz.dt, p.iz.a), p.iz.b)));
                    if (p.g_V && valid[r]) g = __fadd_rn(g, __ldg(p.g_V + o));
                    gu[j][r] = __fadd_rn(__fmul_rn(__fmul_rn(gv[j][r], -dtC), __fsub_rn(1.0f, zt)),
                                         __fmul_rn(gu[j][r], __fsub_rn(1.0f, __fmul_rn(p.iz.dt, p.iz.a))));
                    gi = __fmul_rn(__fmul_rn(g, dtC), __fsub_rn(1.0f, zprev));
                } else {
                    float thr = p.theta;
                    if (p.alif) thr = __fadd_rn(p.theta, __fmul_rn(beta, valid[r] ? __ldg(p.a + o) : 0.f));
                    const float sg = TRACE ? vt : surrogate_grad(p.surrogate, p.gamma, vt, thr);
                    const float carry = __fmul_rn(__fmul_rn(p.alpha, gv[j][r]), __fsub_rn(1.0f, zt));
                    g = __fadd_rn(__fmul_rn(s, sg), carry);
                    if (p.g_V && valid[r]) g = __fadd_rn(g, __ldg(p.g_V + o));
                    gi = __fmul_rn(g, __fsub_rn(1.0f, zprev));
                }
                gv[j][r] = g;
                if (valid[r]) {
                    if (p.gI_lo) {
                        const float hi = __uint_as_float(__float_as_uint(gi) & 0xFFFFE000u);
                        p.gI[o] = hi;
                        p.gI_lo[o] = __fsub_rn(gi, hi);
                    } else {
                        p.gI[o] = gi;
                    }
                }
                if (REC) s_g[((t & 1) * H + i) * R + r] = gi;
            }
        }
        if (REC) __syncthreads();
    }
}

// dW_out[i][c] = sum_{b,t} Z[b,t,i] gy[b,t,c];  db[c] = sum_{b,t} gy[b,t,c]   as per-CTA partials for k_finalize_grads.
// grid = (nparts, ceil(H / 128)), block = 128: thread = neuron; CTA column q owns the CONTIGUOUS rows [q per, (q+1) per) of the
// (B T) axis, stages their adjoint rows (64 B each) and spike words through shared memory with coalesced loads, then
// accumulates from shared memory (a load-use chain per row from global memory made this kernel latency-bound: 59 us
// at B T = 25 600; it runs beside the BPTT sweep and must not outlast it).
constexpr int kWoutStage = 128;      // rows staged per pass
__global__ void __launch_bounds__(128) k_wout_grad(int BT, int H, int O, const uint32_t* __restrict__ zbits,
                                                  const float* __restrict__ gy_scan, float* __restrict__ part_wout,
                                                  float* __restrict__ part_db)
{
    __shared__ __align__(16) float s_gy[kWoutStage * kOMax];
    __shared__ uint32_t s_zw[kWoutStage * 4];
    const int tid = threadIdx.x, lane = tid & 31, W32 = H / 32;
    const int i = blockIdx.y * 128 + tid;
    const int per = (BT + gridDim.x - 1) / gridDim.x;
    const int r0 = blockIdx.x * per, r1 = min(BT, r0 + per);
    float acc[kOMax], dbacc[kOMax];
#pragma unroll
    for (int c = 0; c < kOMax; ++c) { acc[c] = 0.f; dbacc[c] = 0.f; }
    for (int base = r0; base < r1; base += kWoutStage) {
        const int n = min(kWoutStage, r1 - base);
        __syncthreads();
        for (int idx = tid; idx < n * (kOMax / 4); idx += 128)
            reinterpret_cast<float4*>(s_gy)[idx] = __ldg(reinterpret_cast<const float4*>(gy_scan + (size_t)base * kOMax) + idx);
        const int wpc = W32 < 4 ? W32 : 4;                // spike words of this CTA's (up to) 128 neurons
        for (int idx = tid; idx < n * wpc; idx += 128) {
            const int r = idx / wpc, w = idx - r * wpc;
            s_zw[r * 4 + w] = __ldg(zbits + (size_t)(base + r) * W32 + blockIdx.y * 4 + w);
        }
        __syncthreads();
        for (int r = 0; r < n; ++r) {
            const float z = i < H ? (float)((s_zw[r * 4 + (tid >> 5)] >> lane) & 1u) : 0.f;
            const float4* g4 = reinterpret_cast<const float4*>(s_gy + r * kOMax);
#pragma unroll
            for (int q = 0; q < kOMax / 4; ++q) {
                const float4 g = g4[q];
                acc[4 * q] = fmaf(z, g.x, acc[4 * q]); acc[4 * q + 1] = fmaf(z, g.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(z, g.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(z, g.w, acc[4 * q + 3]);
                dbacc[4 * q] += g.x; dbacc[4 * q + 1] += g.y; dbacc[4 * q + 2] += g.z; dbacc[4 * q + 3] += g.w;
            }
        }
    }
#pragma unroll
    for (int c = 0; c < kOMax; ++c)
        if (c < O && i < H) part_wout[((size_t)blockIdx.x * H + i) * O + c] = acc[c];
    if (blockIdx.y == 0 && tid == 0) {
#pragma unroll
        for (int c = 0; c < kOMax; ++c)
            if (c < O) part_db[(size_t)blockIdx.x * O + c] = dbacc[c];
    }
}

}  // namespace snnk
