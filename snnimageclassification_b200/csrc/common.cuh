// common.cuh -- shared device helpers and kernel parameter blocks for libsnnk.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace snnk {

constexpr int kOMax = 16;   // readout units are padded to 16 lanes in shared memory / registers

constexpr int kRunHdrInts = 4;   // header words of the frame-run table (runs.cuh)

// IzhikevichLayer constants (spiking_layers.py:275-296); on == 0 for LIF / ALIF
struct IzhConsts {
    int on;
    float dt, C, vr, vth, k, a, b, c, d, vpeak;
};

struct FwdParams {
    int B, T, H, O;
    int alif, traces;
    float alpha, rho, theta, kappa;
    const float* I_in;      // (B,T,H) input current from the projection GEMM
    const float* W_eff;     // (H,H) W_rec (.) rec_mask, prepared by k_prep_rec: column i belongs to thread i
    const float* beta;      // device scalar or null
    const float* W_out;     // (H,O)
    const float* b_out;     // (O)
    const float* V0; const float* a0; const float* Z0;   // (B,H) or null
    float* V; float* a; float* Z;                        // (B,T,H) traces (traces != 0)
    uint32_t* zbits;        // (B,T,H/32)
    float* y;               // (B,T,O)
    float* logits;          // (B,O)
    int32_t* tstar;         // (B,O)
    // frame-dedup variant (runs.cuh): when the table says ok, the input current of step (b,t) is row
    // table[4 + b*T + t] of the compact projection I_u instead of row b*T+t of I_in
    const int* run_table; const float* I_u;
    IzhConsts iz;           // Izhikevich layer: the `a` trace / a0 state hold the recovery variable u
    // Fused head (k_recur_fwd, snnk_forward_nll): the CTA that owns a row also evaluates its log_softmax, NLL term and
    // dL/dlogits in the kernel's tail; the last CTA to finish reduces the loss.  labels == nullptr: no head.
    const long long* labels; float* logp; float* g_logits; float* loss;
    float* part_nll;        // (B) per-row NLL terms
    unsigned int* ticket;   // zero before the launch; the last CTA leaves it zero again
    unsigned long long* mailbox; unsigned int* mail_counter;
    // 1: launched as a programmatic dependent of the projection kernel (k_recur_fwd_lean): the kernel may start while the
    // projection still runs and must execute griddepcontrol.wait before it touches I_in / I_u
    int pdl;
};

struct BwdParams {
    int B, T, H, O;
    int alif, surrogate;
    float alpha, theta, gamma, kappa;
    const float* W_effT;    // (H,H) transpose of W_rec (.) rec_mask: column i = row i of the masked matrix
    const float* beta; const float* W_out;
    const float* Z0;
    const float* V; const float* a; const uint32_t* zbits;
    const float* g_y;                               // (B,T,O) dense seeds, or null
    const float* g_logits; const int32_t* tstar;    // (B,O) sparse seeds, or null
    const float* g_scale;                           // device scalar multiplying the sparse seeds (dL/dloss), or null
    const float* g_V; const float* g_Z;             // optional (B,T,H) seeds
    float* gI;          // (B,T,H)
    float* gI_lo;       // (B,T,H) or null: when set, gI receives trunc_tf32(gI) and gI_lo the exact remainder
    float* part_wout;   // [grid][H][O]
    float* part_db;     // [grid*R][O]
    // frame-dedup variant (runs.cuh): when the table says ok, the sweep also leaves the sum of gI over every run of
    // equal input frames in Gu_hi / Gu_lo (two tf32 planes, compact rows) for the dW_in contraction
    const int* run_table; float* Gu_hi; float* Gu_lo;
    IzhConsts iz;
};

// W_rec (.) rec_mask (spiking_layers.py:165/235 re-multiplies the mask at every step) and its transpose, once per call.
__global__ void __launch_bounds__(256) k_prep_rec(const float* __restrict__ W_rec, const float* __restrict__ mask,
                                                 int H, float* __restrict__ W_eff, float* __restrict__ W_effT)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= H * H) return;
    const int r = idx / H, c = idx - r * H;
    const float v = mask ? __fmul_rn(W_rec[idx], mask[idx]) : W_rec[idx];
    if (W_eff) W_eff[idx] = v;
    if (W_effT) W_effT[c * H + r] = v;
}

// Surrogate derivatives, spike_funcs.py:59-62 (FastSigmoid) and :75-79 (Phi, epsilon = 1e-5).
__device__ __forceinline__ float surrogate_grad(int kind, float gamma, float v, float thr)
{
    if (kind == 0) {
        float d = __fadd_rn(__fmul_rn(gamma, fabsf(__fsub_rn(v, thr))), 1.0f);
        return __frcp_rn(__fmul_rn(d, d));     // correctly rounded reciprocal == 1.0f / (d * d), fewer instructions
    }
    float te = __fadd_rn(thr, 1e-5f);
    float r = __fsub_rn(1.0f, fabsf(__fdiv_rn(__fsub_rn(v, thr), te)));
    r = r < 0.f ? 0.f : r;
    return __fmul_rn(__fdiv_rn(gamma, te), r);
}

// SNNK_SURROGATE_TRACE: the caller evaluated sigma' of a user-defined surrogate itself and snnk_backward streams it in
// place of the V trace (include/snnk.h).
constexpr int kSurrTrace = 2;

// The same with the kind fixed at compile time, as the BPTT sweeps instantiate it; for kSurrTrace v already is sigma'.
template <int SURR>
__device__ __forceinline__ float surrogate_grad(float gamma, float v, float thr)
{
    if constexpr (SURR == kSurrTrace) return v;
    else return surrogate_grad(SURR, gamma, v, thr);
}

// sum_k w[k] * z[k] with sixteen accumulators over k mod 16 (the order oracle/snn_oracle.c fixes), held as eight
// float2 and advanced with the packed FFMA2 of sm_100: H/2 FMA instructions instead of H, and eight independent
// dependency chains per warp so the FMA latency is covered without help from other warps.  Each lane of an FFMA2
// is an independent IEEE fma, so the result is bit-identical to sixteen scalar fmaf chains.
template <int H>
__device__ __forceinline__ float dot_rec16(const float (&w)[H], const float4* __restrict__ zv)
{
    float2 acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < H / 4; ++j) {
        const float4 z = zv[j];
        const int k = 4 * j, q = 2 * (j & 3);
        acc[q] = __ffma2_rn(make_float2(w[k], w[k + 1]), make_float2(z.x, z.y), acc[q]);
        acc[q + 1] = __ffma2_rn(make_float2(w[k + 2], w[k + 3]), make_float2(z.z, z.w), acc[q + 1]);
    }
    const float lo = __fadd_rn(__fadd_rn(__fadd_rn(acc[0].x, acc[0].y), __fadd_rn(acc[1].x, acc[1].y)),
                               __fadd_rn(__fadd_rn(acc[2].x, acc[2].y), __fadd_rn(acc[3].x, acc[3].y)));
    const float hi = __fadd_rn(__fadd_rn(__fadd_rn(acc[4].x, acc[4].y), __fadd_rn(acc[5].x, acc[5].y)),
                               __fadd_rn(__fadd_rn(acc[6].x, acc[6].y), __fadd_rn(acc[7].x, acc[7].y)));
    return __fadd_rn(lo, hi);
}

// ---- column-blocked form of the same sum ----------------------------------------------------------------------------
// dot_rec16 makes every thread read the whole broadcast vector (H/4 LDS.128 per row and step); at 128 threads per row
// that is 64 KB of shared-memory return traffic per row-step, and the recurrence kernels were measured to be bound by
// exactly that path, not by the FMAs.  Here the four lanes of a quad share the quad's four columns: lane g holds, for
// EACH of the four columns, the weights of accumulation chains 4g..4g+3 (k mod 16 in [4g, 4g+4)), so it needs only
// every fourth float4 of the vector (H/16 LDS.128 per row-step, a quarter of the traffic) for the same H FMAs.  The
// partial q_g = (c_4g + c_4g+1) + (c_4g+2 + c_4g+3) of a column is a subtree of dot_rec16's summation tree
// (lo = q0 + q1, hi = q2 + q3, sum = lo + hi), so three quad shuffles finish the tree and the result is bit-identical;
// lane g ends up with the finished sum of column 4*(i/4)+g = i, its own neuron.
template <int H>
__device__ __forceinline__ void load_w_cb(float (&w)[H], const float* __restrict__ s_w, int i)
{
    const int g = i & 3, c0 = i & ~3;
#pragma unroll
    for (int ci = 0; ci < 4; ++ci)
#pragma unroll
        for (int j = 0; j < H / 16; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) w[(ci * (H / 16) + j) * 4 + e] = s_w[(16 * j + 4 * g + e) * H + c0 + ci];
}

template <int H>
__device__ __forceinline__ float dot_rec16_cb(const float (&w)[H], const float4* __restrict__ zv, int g)
{
    float2 acc[4][2];
#pragma unroll
    for (int ci = 0; ci < 4; ++ci) acc[ci][0] = acc[ci][1] = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j < H / 16; ++j) {
        const float4 z = zv[4 * j + g];
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
            const int o = (ci * (H / 16) + j) * 4;
            acc[ci][0] = __ffma2_rn(make_float2(w[o], w[o + 1]), make_float2(z.x, z.y), acc[ci][0]);
            acc[ci][1] = __ffma2_rn(make_float2(w[o + 2], w[o + 3]), make_float2(z.z, z.w), acc[ci][1]);
        }
    }
    float q[4];
#pragma unroll
    for (int ci = 0; ci < 4; ++ci)
        q[ci] = __fadd_rn(__fadd_rn(acc[ci][0].x, acc[ci][0].y), __fadd_rn(acc[ci][1].x, acc[ci][1].y));
    // quad butterfly: (xor 1) lo = q0 + q1 on lanes 0,1 and hi = q2 + q3 on lanes 2,3; (xor 2) lo + hi
    const bool odd = g & 1, upper = g & 2;
    const float rA = __shfl_xor_sync(0xffffffffu, odd ? q[0] : q[1], 1);
    const float rB = __shfl_xor_sync(0xffffffffu, odd ? q[2] : q[3], 1);
    const float sA = odd ? __fadd_rn(rA, q[1]) : __fadd_rn(q[0], rA);     // columns 0 (even lanes) / 1 (odd lanes)
    const float sB = odd ? __fadd_rn(rB, q[3]) : __fadd_rn(q[2], rB);     // columns 2 / 3
    const float rC = __shfl_xor_sync(0xffffffffu, upper ? sA : sB, 2);
    return upper ? __fadd_rn(rC, sB) : __fadd_rn(sA, rC);
}

}  // namespace snnk
