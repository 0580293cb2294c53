// recur_wide.cuh -- the recurrence of WIDE hidden layers (128 < H <= 2048, BASELINE configs[3] and [4]) as a
// weight-stationary, grid-synchronous tensor-core kernel.
//
// The masked recurrent matrix of a wide layer (4 MB fp32 at H = 1024, 16 MB at 2048) fits neither the registers nor
// the shared memory of one SM -- nor of a 16-CTA cluster at fp32-grade precision -- so it is partitioned over the
// WHOLE chip: CTA (m, n) owns the rows [m MT, (m+1) MT) of the batch and the NS = 16 NSM output neurons
// [n NS, (n+1) NS); its slice W[:, n NS ..] stays in shared memory for the entire sequence as two fp16 planes
// (w s = hi + lo / 2048, 22 significant bits, see recur_tc.cuh), 128 KB.  A time step is
//     S^T (NS x MT) = W_slice^T (NS x H) . Z_{t-1}^T (H x MT)
// on mma.sync.m16n8k16 with the NEURONS on M: A fragments come from the resident slice by ldmatrix, each one reused
// for the four 8-row n-tiles a warp owns; B fragments are expanded in registers straight from the BIT-PACKED spike
// tile of the previous step (H MT / 8 bytes: 16 KB at H = 1024, MT = 128), which is all the CTAs of an m-tile have to
// exchange: every CTA publishes the NS bits per row it produced into a double-buffered tile in global memory (L2),
// bumps the m-tile's arrival counter (release), and the next step starts when the counter shows all H / NS slices
// (acquire; ~1 us, tools/ubench.cu).  The kernel is launched cooperatively (all CTAs co-resident; batches larger than
// n_mt MT rows are processed in passes) and never waits on anything but that counter.
//
// Replaces recur_gen.cuh's forward, which re-read the whole matrix from L2 for every 4 rows and step (c4: 8.1 ms;
// here the matrix is read once per launch).  Same arithmetic as recur_tc.cuh / recur_fwd.cuh per element
// (spiking_layers.py:156-171, :229-243); tensor-core mode only.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "recur_tc.cuh"

namespace snnk {

constexpr int kWideThreads = 256;       // 8 compute warps
constexpr int kWideFlagStride = 32;     // uint32 words between the arrival counters of two m-tiles (128 B)

struct WideParams {
    int B, T, H, O;
    int alif, traces, surrogate;
    float alpha, rho, theta, gamma;
    const float* I_in;          // (B,T,H)
    const float* W;             // forward: W_eff [k][i]; backward: W_effT [k][i] = W_eff[i][k]
    const float* beta;
    const float* V0; const float* a0; const float* Z0;
    float* V; float* a; float* Z;      // traces (forward: written when traces != 0; backward: read)
    uint32_t* zbits;            // (B,T,H/32)
    // exchange through L2
    uint32_t* zx;               // forward: [2][n_mt][H/32][MT] spike words of the previous step
    unsigned int* flags;        // [n_mt] arrival counters, kWideFlagStride words apart, zero at launch
    int n_mt, n_nt;             // grid = n_mt * n_nt CTAs: blockIdx.x = m * n_nt + n
};

// NSM = 16-neuron m-tiles per CTA (1, 2, 4); rows per m-tile of the batch MT = 256 / NSM (8 warps x 32 rows / NSM)
__host__ __device__ constexpr int wide_nsm(int H) { return H <= 512 ? 4 : (H <= 1024 ? 2 : 1); }
__host__ __device__ constexpr int wide_mt(int nsm) { return 256 / nsm; }
__host__ __device__ constexpr int wide_wstride(int H) { return H + 8; }      // halves per neuron row of a plane (conflict-free ldmatrix)

__host__ __device__ constexpr size_t wide_fwd_smem_bytes(int H)
{
    return sizeof(__half) * 2 * (size_t)(16 * wide_nsm(H)) * wide_wstride(H)        // weight slice, two planes
           + sizeof(uint32_t) * (size_t)(H / 32) * wide_mt(wide_nsm(H))              // spike words of the previous step
           + sizeof(uint16_t) * (size_t)wide_mt(wide_nsm(H)) * wide_nsm(H)            // this step's bits [row][m-tile]
           + 64;
}

// Spin until the m-tile's arrival counter reaches `target` (thread 0; bounded: a missing peer traps instead of hanging).
__device__ __forceinline__ void wide_wait_flag(const unsigned int* flag, unsigned int target)
{
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
    if ((int)(v - target) >= 0) return;
    const long long t0 = clock64();
    do {
        __nanosleep(64);
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (clock64() - t0 > 8000000000ll) __trap();
    } while ((int)(v - target) < 0);
}

// Slice of Wm[k][i] (row-major, ld = H) for neurons i0 .. i0 + NS into shared memory as two fp16 planes [plane][NS][H + 8],
// scaled by the power of two that puts the slice's largest magnitude at 2^13..2^14.  Returns 1 / scale.
template <int NSM>
__device__ __forceinline__ float wide_load_slice(const float* __restrict__ Wm, int H, int i0, __half* s_w, float* s_red)
{
    constexpr int NS = 16 * NSM;
    const int tid = threadIdx.x, ws = wide_wstride(H);
    float mx = 0.f;
    for (int idx = tid; idx < H * NS; idx += kWideThreads) {
        const int k = idx / NS, m = idx - k * NS;
        mx = fmaxf(mx, fabsf(__ldg(Wm + (size_t)k * H + i0 + m)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((tid & 31) == 0) s_red[tid >> 5] = mx;
    __syncthreads();
    mx = s_red[0];
#pragma unroll
    for (int q = 1; q < kWideThreads / 32; ++q) mx = fmaxf(mx, s_red[q]);
    const float s = pow2_scale_for(mx);
    for (int idx = tid; idx < H * NS; idx += kWideThreads) {
        const int k = idx / NS, m = idx - k * NS;
        __half hi, lo;
        split_h2(__fmul_rn(__ldg(Wm + (size_t)k * H + i0 + m), s), hi, lo);
        s_w[(size_t)m * ws + k] = hi;
        s_w[(size_t)(NS + m) * ws + k] = lo;
    }
    __syncthreads();
    return __fdiv_rn(1.0f, s);
}

// B fragment (k16 x n8) from 16 spike bits of one row: b0 = (k = 2 tig, 2 tig + 1), b1 = (k + 8, k + 9).  A spike is
// encoded as fp16 2.0 = 0x4000 -- a SINGLE bit -- so a fragment register is one multiply (two shifted copies of the
// four relevant bits) and one mask; the factor 2 is folded into the weight scale.  (1.0 = 0x3C00 cost ~9 ALU
// instructions per fragment and made the kernel issue-bound: 4400 instructions per warp and step for 512 MMAs.)
__device__ __forceinline__ void bits_to_bfrag(uint32_t bits16_shifted /* >> 2 tig */, uint32_t (&b)[2])
{
    const uint32_t y = bits16_shifted & 0x0303u;                     // bits 0, 1 (k, k + 1) and 8, 9 (k + 8, k + 9)
    b[0] = (y * ((1u << 14) | (1u << 29))) & 0x40004000u;            // bit 0 -> 14, bit 1 -> 30
    b[1] = (y * ((1u << 6) | (1u << 21))) & 0x40004000u;             // bit 8 -> 14, bit 9 -> 30
}

// every 4th bit of x (bits 0, 4, ..., 28) gathered into the low byte
__device__ __forceinline__ uint32_t gather4(uint32_t x)
{
    x &= 0x11111111u;
    x = (x | (x >> 3)) & 0x03030303u;
    x = (x | (x >> 6)) & 0x000F000Fu;
    x = (x | (x >> 12)) & 0xFFu;
    return x;
}

// ---- forward --------------------------------------------------------------------------------------------------------
// cooperative launch, grid = n_mt * n_nt, block = 256, dynamic smem = wide_fwd_smem_bytes(H)
template <int NSM, bool ALIF>
__global__ void __launch_bounds__(kWideThreads, 1) k_wide_fwd(const WideParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NS = 16 * NSM, MT = 256 / NSM, NT = 4;      // a warp owns one m-tile and 32 rows = 4 n-tiles
    const int T = p.T, H = p.H, B = p.B, KW = H / 32, ws = wide_wstride(H);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const int m = blockIdx.x / p.n_nt, n = blockIdx.x - m * p.n_nt;
    const int i0 = n * NS;
    const int mt = warp % NSM, rg = warp / NSM;

    __half* s_w = reinterpret_cast<__half*>(smem_raw);                              // [2][NS][H + 8]
    uint32_t* s_zx = reinterpret_cast<uint32_t*>(s_w + 2 * (size_t)NS * ws);        // [H/32][MT]
    uint16_t* s_out = reinterpret_cast<uint16_t*>(s_zx + (size_t)KW * MT);          // [MT][NSM]
    float* s_red = reinterpret_cast<float*>(s_out + MT * NSM);                      // [8]

    const float inv_s = 0.5f * wide_load_slice<NSM>(p.W, H, i0, s_w, s_red);      // spikes enter the MMA as 2.0
    const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
    unsigned int* flag = p.flags + (size_t)m * kWideFlagStride;

    // ldmatrix source of this lane for the A tile (m16 x k16) of m-tile mt: matrices (rows 0-7, k 0-7), (rows 8-15, k 0-7),
    // (rows 0-7, k 8-15), (rows 8-15, k 8-15) = a0..a3
    const uint32_t a_base = tc::smem_u32(s_w) + (uint32_t)((mt * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * ws + 8 * (lane >> 4)) * 2;
    const uint32_t a_plane = (uint32_t)(NS * ws) * 2;
    const int rows_per_pass = p.n_mt * MT;
    const int n_pass = (B + rows_per_pass - 1) / rows_per_pass;
    const int wrow = rg * 32;      // first row (within the m-tile) of this warp

    for (int pass = 0; pass < n_pass; ++pass) {
        const int row0 = pass * rows_per_pass + m * MT;      // first batch row of this CTA's m-tile
        // element (nt, e): neuron i0 + 16 mt + g + 8 (e >> 1), row row0 + wrow + 8 nt + 2 tig + (e & 1)
        float v[NT][4], a[NT][4], zp[NT][4];
        bool ok[NT][2];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
            for (int rh = 0; rh < 2; ++rh) ok[nt][rh] = row0 + wrow + 8 * nt + 2 * tig + rh < B;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int row = row0 + wrow + 8 * nt + 2 * tig + (e & 1), col = i0 + 16 * mt + g + 8 * (e >> 1);
                const bool o = ok[nt][e & 1];
                const size_t s = (size_t)(o ? row : 0) * H + col;
                v[nt][e] = (o && p.V0) ? p.V0[s] : 0.f;
                a[nt][e] = (o && p.a0) ? p.a0[s] : 0.f;
                zp[nt][e] = (o && p.Z0) ? p.Z0[s] : 0.f;
            }
        }
        // Everybody has finished the previous pass (its last tile was read before its last publish) before the exchange
        // buffers are written again.
        if (pass > 0) {
            if (tid == 0) wide_wait_flag(flag, (unsigned int)p.n_nt * (unsigned int)(pass * T));
            __syncthreads();
        }
        // spike words of "step -1": the initial state (zeros unless Z0 is given)
        for (int idx = tid; idx < KW * MT; idx += kWideThreads) {
            uint32_t w = 0u;
            if (p.Z0) {
                const int kw = idx / MT, r = idx - kw * MT;
                if (row0 + r < B)
                    for (int l = 0; l < 32; ++l)
                        if (__ldg(p.Z0 + (size_t)(row0 + r) * H + kw * 32 + l) != 0.f) w |= 1u << l;
            }
            s_zx[idx] = w;
        }
        __syncthreads();

        for (int t = 0; t < T; ++t) {
            const unsigned int gstep = (unsigned int)(pass * T + t);
            if (t > 0) {
                // all n_nt slices of step t-1 published?  then fetch the m-tile's spike words (L2 only: they change every step)
                if (tid == 0) wide_wait_flag(flag, (unsigned int)p.n_nt * gstep);
                __syncthreads();
                const uint4* src = reinterpret_cast<const uint4*>(p.zx + ((size_t)((gstep - 1) & 1) * p.n_mt + m) * KW * MT);
                for (int idx = tid; idx < KW * MT / 4; idx += kWideThreads) reinterpret_cast<uint4*>(s_zx)[idx] = __ldcg(src + idx);
                __syncthreads();
            }
            // input current of this step: issued now, consumed after the MMA phase
            float cur[NT][4];
            {
                const float* pin = p.I_in + ((size_t)(row0 + wrow + 2 * tig) * T + t) * H + i0 + 16 * mt + g;
                const uint32_t TH = (uint32_t)T * (uint32_t)H;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        cur[nt][e] = ok[nt][e & 1] ? __ldg(pin + (uint32_t)(8 * nt + (e & 1)) * TH + 8u * (e >> 1)) : 0.f;
            }
            // ---- S^T = W_slice^T Z_{t-1}^T ----
            float ch[NT][4], cl[NT][4];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) { ch[nt][e] = 0.f; cl[nt][e] = 0.f; }
#pragma unroll 2
            for (int kw = 0; kw < KW; ++kw) {
                uint32_t ah0[4], al0[4], ah1[4], al1[4];
                ldsm_x4(ah0, a_base + (uint32_t)(kw * 32) * 2);
                ldsm_x4(al0, a_base + a_plane + (uint32_t)(kw * 32) * 2);
                ldsm_x4(ah1, a_base + (uint32_t)(kw * 32 + 16) * 2);
                ldsm_x4(al1, a_base + a_plane + (uint32_t)(kw * 32 + 16) * 2);
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const uint32_t w = s_zx[kw * MT + wrow + 8 * nt + g] >> (2 * tig);
                    uint32_t b0[2], b1[2];
                    bits_to_bfrag(w, b0);
                    bits_to_bfrag(w >> 16, b1);
                    mma_f16(ch[nt], ah0, b0);
                    mma_f16(cl[nt], al0, b0);
                    mma_f16(ch[nt], ah1, b1);
                    mma_f16(cl[nt], al1, b1);
                }
            }
            // ---- state update and spike bits; the traces are stored AFTER the step has been published ----
            uint32_t mine[2] = {0u, 0u};
        #pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int nh = e >> 1, rh = e & 1;
                    const float rec = __fmul_rn(fmaf(cl[nt][e], 1.0f / 2048.0f, ch[nt][e]), inv_s);
                    const float t1 = __fmul_rn(p.alpha, v[nt][e]);
                    const float t2 = __fadd_rn(t1, cur[nt][e]);
                    const float t3 = __fadd_rn(t2, rec);
                    const float vn = __fmul_rn(t3, __fsub_rn(1.0f, zp[nt][e]));      // spiking_layers.py:169/239
                    float thr = p.theta;
                    if constexpr (ALIF) {
                        a[nt][e] = __fadd_rn(__fmul_rn(p.rho, a[nt][e]), zp[nt][e]);      // :240
                        thr = __fadd_rn(p.theta, __fmul_rn(beta, a[nt][e]));              // :241
                    }
                    const bool spk = ok[nt][rh] && vn >= thr;                             // spike_funcs.py:27-28
                    v[nt][e] = vn;
                    zp[nt][e] = spk ? 1.0f : 0.0f;
                    // ballot bit 4 g' + tig' = spike of (neuron g' + 8 nh, row 8 nt + 2 tig' + rh); lane L keeps the
                    // ballots of ITS row L = 8 nt + 2 tig' + rh
                    const uint32_t bal = __ballot_sync(0xffffffffu, spk);
                    if ((lane >> 3) == nt && (lane & 1) == rh) mine[nh] = bal;
                }
            }
            {
                const int tl = (lane & 7) >> 1;
                const uint32_t half = gather4(mine[0] >> tl) | (gather4(mine[1] >> tl) << 8);      // 16 neurons of row `lane`
                s_out[(wrow + lane) * NSM + mt] = (uint16_t)half;
            }
            __syncthreads();
            // publish: warp 0 copies this CTA's NS bits per row into the exchange tile of step t and RELEASES the m-tile's
            // counter.  It does so before anybody issues the step's trace stores: a release (like a __threadfence) waits
            // for the issuing thread's earlier writes, and 48 scattered stores per thread in front of it made every
            // step wait for HBM.
            if (warp == 0) {
                uint16_t* zx16 = reinterpret_cast<uint16_t*>(p.zx + ((size_t)(gstep & 1) * p.n_mt + m) * KW * MT);
                for (int idx = lane; idx < NSM * MT; idx += 32) {
                    const int q = idx / MT, r = idx - q * MT;
                    const int hc = n * NSM + q;                    // 16-neuron group (half word) of the hidden axis
                    zx16[((size_t)(hc >> 1) * MT + r) * 2 + (hc & 1)] = s_out[r * NSM + q];
                }
                __syncwarp();
                if (lane == 0) asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(flag), "r"(1u) : "memory");
            }
            // the raster (B,T,H/32) and the traces of this step
            {
                uint16_t* zb16 = reinterpret_cast<uint16_t*>(p.zbits);
                for (int idx = tid; idx < NSM * MT; idx += kWideThreads) {
                    const int q = idx / MT, r = idx - q * MT;
                    const int hc = n * NSM + q;
                    if (row0 + r < B) zb16[(((size_t)(row0 + r) * T + t) * KW + (hc >> 1)) * 2 + (hc & 1)] = s_out[r * NSM + q];
                }
            }
            if (p.traces) {
                // one 64-bit base per thread and step, 32-bit offsets (8 nt + rh) T H + 8 nh per element
                const size_t ob = ((size_t)(row0 + wrow + 2 * tig) * T + t) * H + i0 + 16 * mt + g;
                float* pv = p.V + ob;
                float* pz = p.Z + ob;
                float* pa = ALIF ? p.a + ob : nullptr;
                const uint32_t TH = (uint32_t)T * (uint32_t)H;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if (!ok[nt][e & 1]) continue;
                        const uint32_t o = (uint32_t)(8 * nt + (e & 1)) * TH + 8u * (e >> 1);
                        pv[o] = v[nt][e];
                        pz[o] = zp[nt][e];
                        if constexpr (ALIF) pa[o] = a[nt][e];
                    }
            }
        }
    }
}


// ---- backward -------------------------------------------------------------------------------------------------------
// Reverse-time sweep of a wide layer (same recurrences as recur_bwd.cuh / recur_tc.cuh):
//     gZ_t = gy_t W_out^T + gI_{t+1} (W_rec . M)^T ;  gV_t = gZ_t sigma'_t + alpha gV_{t+1} (1 - Z_t) ;  gI_t = gV_t (1 - Z_{t-1})
// with the matvec as  gZ^T (NS x MT) = W_eff[slice rows] (NS x H) . gI_{t+1}^T (H x MT)  on the tensor cores.  The slice of
// W_eff is resident as in the forward kernel; what the CTAs of an m-tile exchange per step is the REAL-valued tile
// gI_t: every CTA writes its NS columns in fp32 into a chunked, padded tile in global memory (L2) together with the
// exponent classes it contains (atomicOr into a per-step mask word), releases the m-tile's counter, and the readers
// stream the tile through a two-buffer shared-memory ring with one bulk copy per 36 KB chunk and split every value
// into fp16 hi + lo / 2048 in registers, with the power-of-two scale the mask dictates (recur_tc.cuh explains the
// scale).  Products hi.hi, hi.lo, lo.hi: 24 MMAs per 16 x 16 x 16 block pair, i.e. 1.5x the forward kernel.
struct WideBwdParams {
    int B, T, H, O;
    int alif, surrogate;
    float alpha, theta, gamma;
    const float* W;             // W_effT [k][i] = W_eff[i][k]
    const float* beta; const float* W_out;      // (H,O)
    const float* V; const float* a; const uint32_t* zbits; const float* Z0;
    const float* gy_scan;       // (B,T,kOMax) from k_gy_scan
    const float* g_V; const float* g_Z;         // optional (B,T,H) seeds
    float* gI; float* gI_lo;    // (B,T,H): gI, or its two tf32 planes
    float* gx;                  // [2][n_mt][H / KC][MT][KC + 8] fp32 exchange tiles
    unsigned int* gmask;        // [n_mt][n_pass * T] exponent-class masks, zero at launch
    unsigned int* flags;        // [n_mt] arrival counters, zero at launch
    int n_mt, n_nt;
};

__host__ __device__ constexpr int wide_bwd_ntw(int nsm) { return nsm == 4 ? 1 : 2; }       // n-tiles (8 rows) per warp
__host__ __device__ constexpr int wide_bwd_mt(int nsm) { return 64 * wide_bwd_ntw(nsm); }   // rows per m-tile: 8 warps x 8 NTW
__host__ __device__ constexpr int wide_bwd_kc(int nsm) { return nsm == 4 ? 128 : 64; }      // k per exchange chunk
__host__ __device__ constexpr size_t wide_bwd_chunk_floats(int nsm) { return (size_t)wide_bwd_mt(nsm) * (wide_bwd_kc(nsm) + 8); }

__host__ __device__ constexpr size_t wide_bwd_smem_bytes(int H)
{
    return sizeof(__half) * 2 * (size_t)(16 * wide_nsm(H)) * wide_wstride(H)        // weight slice, two planes
           + sizeof(float) * 2 * wide_bwd_chunk_floats(wide_nsm(H))                   // two chunk buffers
           + sizeof(float) * (size_t)wide_bwd_mt(wide_nsm(H)) * kOMax                 // readout adjoint of the step
           + sizeof(float) * (size_t)(16 * wide_nsm(H)) * kOMax                       // W_out rows of the slice
           + 128;
}

template <int NSM, bool ALIF, int SURR>
__global__ void __launch_bounds__(kWideThreads, 1) k_wide_bwd(const WideBwdParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NS = 16 * NSM, NTW = wide_bwd_ntw(NSM), MT = wide_bwd_mt(NSM), KC = wide_bwd_kc(NSM), CS = KC + 8;
    constexpr uint32_t kChunkBytes = (uint32_t)(MT * CS * sizeof(float));
    const int T = p.T, H = p.H, B = p.B, O = p.O, KW = H / 32, ws = wide_wstride(H);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const int m = blockIdx.x / p.n_nt, n = blockIdx.x - m * p.n_nt;
    const int i0 = n * NS;
    const int wrow = warp * 8 * NTW;       // this warp: all NSM m-tiles of the slice x rows [wrow, wrow + 8 NTW)
    const int n_chunks = H / KC;

    __half* s_w = reinterpret_cast<__half*>(smem_raw);                              // [2][NS][H + 8]
    float* s_ch = reinterpret_cast<float*>(s_w + 2 * (size_t)NS * ws);              // [2][MT][CS]
    float* s_gy = s_ch + 2 * (size_t)MT * CS;                                       // [MT][kOMax]
    float* s_wo = s_gy + MT * kOMax;                                                // [NS][kOMax]
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_wo + NS * kOMax);               // [2]
    float* s_red = reinterpret_cast<float*>(s_bar + 2);                             // [8]
    uint32_t* s_misc = reinterpret_cast<uint32_t*>(s_red + 8);                      // [0] mask read, [1] classes written

    const float inv_sw = wide_load_slice<NSM>(p.W, H, i0, s_w, s_red);
    for (int idx = tid; idx < NS * kOMax; idx += kWideThreads) {
        const int r = idx / kOMax, c = idx - r * kOMax;
        s_wo[idx] = c < O ? __ldg(p.W_out + (size_t)(i0 + r) * O + c) : 0.f;
    }
    if (tid == 0) {
        tc::mbar_init(s_bar, 1);
        tc::mbar_init(s_bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_misc[0] = 0u; s_misc[1] = 0u;
    }
    const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
    unsigned int* flag = p.flags + (size_t)m * kWideFlagStride;
    uint32_t ph0 = 0u, ph1 = 0u;    // mbarrier phase of the two chunk buffers (every thread waits on every chunk)

    // ldmatrix source of this lane for the A tile of m-tile 0 (+ mt * 16 rows); see k_wide_fwd
    const uint32_t a_base = tc::smem_u32(s_w) + (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * ws + 8 * (lane >> 4)) * 2;
    const uint32_t a_plane = (uint32_t)(NS * ws) * 2, a_mt = (uint32_t)(16 * ws) * 2;
    const int rows_per_pass = p.n_mt * MT;
    const int n_pass = (B + rows_per_pass - 1) / rows_per_pass;
    const uint16_t* zb16 = reinterpret_cast<const uint16_t*>(p.zbits);
    __syncthreads();

    for (int pass = 0; pass < n_pass; ++pass) {
        const int row0 = pass * rows_per_pass + m * MT;
        // element (mt, nt, e): neuron i0 + 16 mt + g + 8 (e >> 1), row row0 + wrow + 8 nt + 2 tig + (e & 1)
        float gv[NSM][NTW][4];
        uint32_t zt[NSM][NTW][2];           // 16 spike bits of (row, m-tile) at the step being processed (carried to the next)
        bool ok[NTW][2];
#pragma unroll
        for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
            for (int rh = 0; rh < 2; ++rh) ok[nt][rh] = row0 + wrow + 8 * nt + 2 * tig + rh < B;
        auto load_bits = [&](int tl, uint32_t (&dst)[NSM][NTW][2]) {      // Z_tl of this thread's rows (tl = -1: initial state)
#pragma unroll
            for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                    for (int rh = 0; rh < 2; ++rh) {
                        const int row = row0 + wrow + 8 * nt + 2 * tig + rh, hc = n * NSM + mt;
                        uint32_t w = 0u;
                        if (ok[nt][rh]) {
                            if (tl >= 0) w = zb16[(((size_t)row * T + tl) * KW + (hc >> 1)) * 2 + (hc & 1)];
                            else if (p.Z0) {
                                for (int l = 0; l < 16; ++l)
                                    if (__ldg(p.Z0 + (size_t)row * H + i0 + 16 * mt + l) != 0.f) w |= 1u << l;
                            }
                        }
                        dst[mt][nt][rh] = w;
                    }
        };
#pragma unroll
        for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                for (int e = 0; e < 4; ++e) gv[mt][nt][e] = 0.f;
        load_bits(T - 1, zt);
        if (pass > 0) {      // everybody is done with the previous pass before its exchange tiles are overwritten
            if (tid == 0) wide_wait_flag(flag, (unsigned int)p.n_nt * (unsigned int)(pass * T));
            __syncthreads();
        }

        for (int s = 0; s < T; ++s) {
            const int t = T - 1 - s;
            const unsigned int gstep = (unsigned int)(pass * T + s);
            const float* tile = p.gx + ((size_t)((gstep + 1) & 1) * p.n_mt + m) * n_chunks * (size_t)(MT * CS);     // written at step s - 1
            if (s > 0 && tid == 0) {
                wide_wait_flag(flag, (unsigned int)p.n_nt * gstep);
                s_misc[0] = __ldcg(p.gmask + (size_t)m * n_pass * T + gstep - 1);
                asm volatile("fence.proxy.async;" ::: "memory");      // the bulk copies below read what the peers just wrote
                for (int c = 0; c < 2 && c < n_chunks; ++c) {
                    tc::mbar_expect_tx(s_bar + c, kChunkBytes);
                    tc::bulk_g2s(s_ch + (size_t)c * MT * CS, tile + (size_t)c * MT * CS, kChunkBytes, s_bar + c);
                }
            }
            // readout adjoint rows of this step, saved traces and previous spikes: issued before the MMA phase
            for (int idx = tid; idx < MT * (kOMax / 4); idx += kWideThreads) {
                const int r = idx / (kOMax / 4);
                float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
                if (row0 + r < B) q = __ldg(reinterpret_cast<const float4*>(p.gy_scan + ((size_t)(row0 + r) * T + t) * kOMax) + (idx - r * (kOMax / 4)));
                reinterpret_cast<float4*>(s_gy)[idx] = q;
            }
            float vt[NSM][NTW][4], at[NSM][NTW][4];
            uint32_t zp[NSM][NTW][2];
            {
                const size_t ob = ((size_t)(row0 + wrow + 2 * tig) * T + t) * H + i0 + g;
                const uint32_t TH = (uint32_t)T * (uint32_t)H;
#pragma unroll
                for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const uint32_t o = (uint32_t)(8 * nt + (e & 1)) * TH + 16u * mt + 8u * (e >> 1);
                            vt[mt][nt][e] = ok[nt][e & 1] ? __ldg(p.V + ob + o) : 0.f;
                            at[mt][nt][e] = (ALIF && ok[nt][e & 1]) ? __ldg(p.a + ob + o) : 0.f;
                        }
            }
            load_bits(t - 1, zp);
            __syncthreads();      // s_misc[0], s_gy visible
            float chh[NSM][NTW][4], cx[NSM][NTW][4];
#pragma unroll
            for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                    for (int e = 0; e < 4; ++e) { chh[mt][nt][e] = 0.f; cx[mt][nt][e] = 0.f; }
            float inv_sg = 1.0f;
            if (s > 0) {
                const uint32_t mask = s_misc[0];
                float sg = 1.0f;
                if (mask) {
                    int kexp = 133 - 8 * (31 - __clz(mask));      // classes of 8 binades: scaled maximum < 2^14
                    kexp = kexp > 126 ? 126 : kexp;
                    sg = __uint_as_float((uint32_t)(kexp + 127) << 23);
                }
                inv_sg = __fdiv_rn(1.0f, sg);
                for (int c = 0; c < n_chunks; ++c) {
                    const int b = c & 1;
                    tc::mbar_wait(s_bar + b, b ? ph1 : ph0);
                    if (b) ph1 ^= 1u; else ph0 ^= 1u;
                    const float* ch = s_ch + (size_t)b * MT * CS;
#pragma unroll 2
                    for (int kt = 0; kt < KC / 16; ++kt) {
                        const uint32_t koff = (uint32_t)(c * KC + kt * 16) * 2;
                        uint32_t bh[NTW][2], bl[NTW][2];
#pragma unroll
                        for (int nt = 0; nt < NTW; ++nt) {
                            const float* src = ch + (wrow + 8 * nt + g) * CS + kt * 16 + 2 * tig;
                            const float2 x0 = *reinterpret_cast<const float2*>(src), x1 = *reinterpret_cast<const float2*>(src + 8);
                            const float2 y0 = make_float2(__fmul_rn(x0.x, sg), __fmul_rn(x0.y, sg));
                            const float2 y1 = make_float2(__fmul_rn(x1.x, sg), __fmul_rn(x1.y, sg));
                            const __half2 h0 = __float22half2_rn(y0), h1 = __float22half2_rn(y1);
                            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
                            const __half2 l0 = __floats2half2_rn(__fmul_rn(__fsub_rn(y0.x, f0.x), 2048.0f), __fmul_rn(__fsub_rn(y0.y, f0.y), 2048.0f));
                            const __half2 l1 = __floats2half2_rn(__fmul_rn(__fsub_rn(y1.x, f1.x), 2048.0f), __fmul_rn(__fsub_rn(y1.y, f1.y), 2048.0f));
                            bh[nt][0] = *reinterpret_cast<const uint32_t*>(&h0); bh[nt][1] = *reinterpret_cast<const uint32_t*>(&h1);
                            bl[nt][0] = *reinterpret_cast<const uint32_t*>(&l0); bl[nt][1] = *reinterpret_cast<const uint32_t*>(&l1);
                        }
#pragma unroll
                        for (int mt = 0; mt < NSM; ++mt) {
                            uint32_t ah[4], al[4];
                            ldsm_x4(ah, a_base + mt * a_mt + koff);
                            ldsm_x4(al, a_base + a_plane + mt * a_mt + koff);
#pragma unroll
                            for (int nt = 0; nt < NTW; ++nt) {
                                mma_f16(chh[mt][nt], ah, bh[nt]);
                                mma_f16(cx[mt][nt], ah, bl[nt]);
                                mma_f16(cx[mt][nt], al, bh[nt]);
                            }
                        }
                    }
                    __syncthreads();      // everybody is done with buffer b: refill it with chunk c + 2
                    if (tid == 0 && c + 2 < n_chunks) {
                        tc::mbar_expect_tx(s_bar + b, kChunkBytes);
                        tc::bulk_g2s(s_ch + (size_t)b * MT * CS, tile + (size_t)(c + 2) * MT * CS, kChunkBytes, s_bar + b);
                    }
                }
            }
            // ---- elementwise part of the step ----
            const float sc = __fmul_rn(inv_sw, inv_sg);
            float gi[NSM][NTW][4];
            uint32_t cls = 0u;
#pragma unroll
            for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                for (int rh = 0; rh < 2; ++rh) {
                    const int rl = wrow + 8 * nt + 2 * tig + rh;      // row within the m-tile
                    float gy[kOMax];
#pragma unroll
                    for (int q = 0; q < kOMax / 4; ++q) {
                        const float4 v4 = reinterpret_cast<const float4*>(s_gy + rl * kOMax)[q];
                        gy[4 * q] = v4.x; gy[4 * q + 1] = v4.y; gy[4 * q + 2] = v4.z; gy[4 * q + 3] = v4.w;
                    }
#pragma unroll
                    for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                        for (int nh = 0; nh < 2; ++nh) {
                            const int e = 2 * nh + rh, il = 16 * mt + g + 8 * nh;      // neuron within the slice
                            float rdo = 0.f;
#pragma unroll
                            for (int q = 0; q < kOMax / 4; ++q) {
                                const float4 w4 = reinterpret_cast<const float4*>(s_wo + il * kOMax)[q];
                                rdo = fmaf(gy[4 * q], w4.x, rdo); rdo = fmaf(gy[4 * q + 1], w4.y, rdo);
                                rdo = fmaf(gy[4 * q + 2], w4.z, rdo); rdo = fmaf(gy[4 * q + 3], w4.w, rdo);
                            }
                            const float rec = __fmul_rn(fmaf(cx[mt][nt][e], 1.0f / 2048.0f, chh[mt][nt][e]), sc);
                            float sum = __fadd_rn(rdo, rec);
                            const bool o_ = ok[nt][rh];
                            const size_t o = ((size_t)(row0 + rl) * T + t) * H + i0 + il;
                            if (p.g_Z && o_) sum = __fadd_rn(sum, __ldg(p.g_Z + o));
                            float thr = p.theta;
                            if constexpr (ALIF) thr = __fadd_rn(p.theta, __fmul_rn(beta, at[mt][nt][e]));
                            const float zcur = (float)((zt[mt][nt][rh] >> (g + 8 * nh)) & 1u);
                            const float zprev = (float)((zp[mt][nt][rh] >> (g + 8 * nh)) & 1u);
                            const float sgr = surrogate_grad<SURR>(p.gamma, vt[mt][nt][e], thr);
                            const float carry = __fmul_rn(__fmul_rn(p.alpha, gv[mt][nt][e]), __fsub_rn(1.0f, zcur));
                            float gq = __fadd_rn(__fmul_rn(sum, sgr), carry);
                            if (p.g_V && o_) gq = __fadd_rn(gq, __ldg(p.g_V + o));
                            gv[mt][nt][e] = gq;
                            const float gix = o_ ? __fmul_rn(gq, __fsub_rn(1.0f, zprev)) : 0.f;
                            gi[mt][nt][e] = gix;
                            cls |= gix != 0.f ? 1u << (((__float_as_uint(gix) >> 23) & 0xFFu) >> 3) : 0u;
                        }
                }
            // ---- publish gI_t: this CTA's NS columns of the exchange tile of step s, its exponent classes, the counter ----
            {
                float* out = p.gx + ((size_t)(gstep & 1) * p.n_mt + m) * n_chunks * (size_t)(MT * CS) + (size_t)(i0 / KC) * (MT * CS) + (i0 % KC);
#pragma unroll
                for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            out[(wrow + 8 * nt + 2 * tig + (e & 1)) * CS + 16 * mt + g + 8 * (e >> 1)] = gi[mt][nt][e];
                const uint32_t wor = __reduce_or_sync(0xffffffffu, cls);
                if (lane == 0 && wor) atomicOr(s_misc + 1, wor);
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) {
                const uint32_t mine = s_misc[1];
                s_misc[1] = 0u;
                if (mine) atomicOr(p.gmask + (size_t)m * n_pass * T + gstep, mine);
                asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(flag), "r"(1u) : "memory");
            }
            // ---- gI of this step for the weight-gradient GEMM (after the publish: see k_wide_fwd) ----
            {
                const size_t ob = ((size_t)(row0 + wrow + 2 * tig) * T + t) * H + i0 + g;
                const uint32_t TH = (uint32_t)T * (uint32_t)H;
#pragma unroll
                for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            if (!ok[nt][e & 1]) continue;
                            const uint32_t o = (uint32_t)(8 * nt + (e & 1)) * TH + 16u * mt + 8u * (e >> 1);
                            const float x = gi[mt][nt][e];
                            if (p.gI_lo) {      // exact two-plane tf32 split
                                const float hi = __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
                                p.gI[ob + o] = hi;
                                p.gI_lo[ob + o] = __fsub_rn(x, hi);
                            } else {
                                p.gI[ob + o] = x;
                            }
                        }
            }
#pragma unroll
            for (int mt = 0; mt < NSM; ++mt)
#pragma unroll
                for (int nt = 0; nt < NTW; ++nt)
#pragma unroll
                    for (int rh = 0; rh < 2; ++rh) zt[mt][nt][rh] = zp[mt][nt][rh];
        }
    }
}

}  // namespace snnk
