// recur_tc.cuh -- K2 / K3 on the tensor cores for H = 128: the recurrent matvec of every time step as warp MMAs with the
// NEURONS on M and the batch rows on N.
//
// Why this shape.  Measured on B200 (tools/ubench.cu, profiles/r02_ubench.txt): mma.sync.m16n8k16 issues every 8.1
// cycles per SM sub-partition (1012 MAC/cycle/SM, 8x the fp32 FMA rate) with 21 cycles of latency, a 288-thread
// bar.sync costs 31 cycles.  The fp32 SIMT kernels (recur_fwd.cuh / recur_bwd.cuh) spend >= 128 FMA-pipe cycles per
// row and step and ran at ~1000 / ~1300 cycles per step with two rows per SM: latency-bound, 4x off even that floor.
// Here one CTA owns EIGHT batch rows (the n8 of the MMA) for all T steps; warp w owns neurons 16w..16w+15 (the m16),
// the masked recurrent matrix lives in its A fragments for the whole sequence, and a step is
//     S^T (128 x 8) = W^T (128 x 128) . Z_{t-1}^T (128 x 8)
// i.e. 16 (forward) / 24 (backward) MMAs per warp against B fragments fetched with 4 / 8 ldmatrix from a 2 KB tile in
// shared memory, 4 state elements per thread, one stmatrix that publishes the new spikes / gradients, one barrier.
// A batch of 256 rows then occupies 32 SMs for ~450-600 cycles per step instead of 148 SMs for 1000-1300.
// (tcgen05 does not fit this step: its M = 128 tile would be the neurons as well, but the round trip
// mma -> commit -> mbarrier -> tcgen05.ld -> registers -> st.shared -> fence.proxy.async per step costs more than the
// 130-190 cycles of MMA time it saves; the tile per step is 128 x 8 x 128.)
//
// Numerics (tensor-core mode only; the fp32 SIMT kernels stay the bit-exact mode).  Spikes are exact in fp16.  A
// weight is split as  w s = hi + lo / 2048  with hi, lo in fp16 and s a power of two that puts max|W| at 2^13..2^14:
// 22 significant bits, the same class as the tf32-plane tcgen05 GEMMs (gemm_tc.cuh).  Products are exact, sums are
// fp32 in the tensor pipe, so results differ from the fp32 kernels by summation order only (~1e-6 relative).  The
// backward operand gI is real-valued: it is split the same way with a scale chosen per CTA and per step from the
// largest exponent in the tile (an OR of exponent-class bits across the CTA before the tile is published), and the three products
// hi.hi, hi.lo, lo.hi are accumulated (the dropped lo.lo term is 2^-22 relative).
//
// Replaces, like recur_fwd.cuh / recur_bwd.cuh: the time loop of SNN.forward (src/modules/snn.py:209-214) around
// LIFLayer/ALIFLayer.forward (src/modules/spiking_layers.py:156-171, :229-243) and ReadoutLayer.forward (:402-408),
// and autograd's reverse sweep for batch_loss.backward() (snn.py:413) with the surrogates of spike_funcs.py:59-62/75-79.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "gemm_tc.cuh"

namespace snnk {

constexpr int kTcH = 128;          // hidden width of these kernels
constexpr int kTcRows = 8;         // batch rows per CTA = N of the MMA
constexpr int kTcThreads = 288;    // 8 neuron warps + 1 service warp
constexpr int kTcTileStride = 136; // halves per row of a spike / gradient tile (272 B: conflict-free ldmatrix)

__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2])
{
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t saddr)
{
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(saddr));
}

__device__ __forceinline__ void stsm_x2_trans(uint32_t saddr, uint32_t r0, uint32_t r1)
{
    asm volatile("stmatrix.sync.aligned.m8n8.x2.trans.shared.b16 [%0], {%1, %2};" ::"r"(saddr), "r"(r0), "r"(r1) : "memory");
}

__device__ __forceinline__ void stsm_x4_trans(uint32_t saddr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3)
{
    asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(r0), "r"(r1),
                 "r"(r2), "r"(r3)
                 : "memory");
}

__device__ __forceinline__ uint32_t pack_h2(__half lo, __half hi)
{
    return (uint32_t)__half_as_ushort(lo) | ((uint32_t)__half_as_ushort(hi) << 16);
}

// x s = hi + lo / 2048 (hi, lo fp16): 22 significant bits when x s is in fp16's normal range
__device__ __forceinline__ void split_h2(float xs, __half& hi, __half& lo)
{
    hi = __float2half_rn(xs);
    lo = __float2half_rn(__fmul_rn(__fsub_rn(xs, __half2float(hi)), 2048.0f));
}

// power of two s with  max * s  in [2^13, 2^14)  (1 for max == 0); exact to multiply and divide by
__device__ __forceinline__ float pow2_scale_for(float mx)
{
    if (!(mx > 0.f)) return 1.0f;
    int e = (int)((__float_as_uint(mx) >> 23) & 0xFFu) - 127;     // floor(log2(mx)) for normal numbers
    int k = 13 - e;
    k = k > 120 ? 120 : (k < -120 ? -120 : k);
    return __uint_as_float((uint32_t)(k + 127) << 23);
}

// Block-wide maximum of a non-negative value (all NT threads of the block call it; s_red: NT / 32 floats of shared memory).
template <int NT = kTcThreads>
__device__ __forceinline__ float block_max_tc(float v, float* s_red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    float m = s_red[0];
#pragma unroll
    for (int q = 1; q < NT / 32; ++q) m = fmaxf(m, s_red[q]);
    __syncthreads();
    return m;
}

// A fragments (m16 x k16, "row") of the two fp16 planes of Wm[k][i] (row-major, leading dimension ld) for the 16
// output neurons i0..i0+15 and K = 16 * KT: thread (g = lane >> 2, tig = lane & 3) holds rows m = g, g + 8 and
// k = 16 kt + 2 tig + {0, 1} (+ 8).  raw[] receives the fp32 values (so the caller can find the scale first).
template <int KT>
__device__ __forceinline__ void load_a_raw(const float* __restrict__ Wm, int ld, int i0, int kmax, int g, int tig,
                                           float (&raw)[KT][8])
{
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            // register order a0 a1 a2 a3, two halves each: a0 = (g, k..k+1), a1 = (g+8, k..), a2 = (g, k+8..), a3 = (g+8, k+8..)
            const int k = 16 * kt + 2 * tig + (q & 1) + 8 * (q >> 2);
            const int m = g + 8 * ((q >> 1) & 1);
            raw[kt][q] = k < kmax ? __ldg(Wm + (size_t)k * ld + i0 + m) : 0.f;
        }
}

template <int KT>
__device__ __forceinline__ void split_a(const float (&raw)[KT][8], float s, uint32_t (&ah)[KT][4], uint32_t (&al)[KT][4])
{
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            __half h0, l0, h1, l1;
            split_h2(__fmul_rn(raw[kt][2 * r], s), h0, l0);
            split_h2(__fmul_rn(raw[kt][2 * r + 1], s), h1, l1);
            ah[kt][r] = pack_h2(h0, h1);
            al[kt][r] = pack_h2(l0, l1);
        }
}

template <int KT>
__device__ __forceinline__ float absmax_raw(const float (&raw)[KT][8])
{
    float m = 0.f;
#pragma unroll
    for (int kt = 0; kt < KT; ++kt)
#pragma unroll
        for (int q = 0; q < 8; ++q) m = fmaxf(m, fabsf(raw[kt][q]));
    return m;
}

// ---- forward --------------------------------------------------------------------------------------------------------
// What bounds this kernel is the SM's load/store pipe, not the tensor pipe and not issue slots (ncu, profiles/r02_*: a
// step of the first versions moved ~730 shared/global "wavefronts" of 128 B through the LSU and took ~1300 cycles
// for 290 cycles of MMA; every shared-memory load of the dependency chain queued behind trace stores that touch four
// cache lines per instruction).  So the design minimises LSU wavefronts per step and keeps everything that merely
// FOLLOWS the dependency chain off the warps that carry it:
//
//   8 NEURON warps (warp w: neurons 16 w ..+15; element e = 2 nh + rh: neuron 16 w + g + 8 nh, row 2 tig + rh), step t:
//       4 ldmatrix (Z_{t-1}) -> 16 MMAs -> update of the 4 elements (input current: 4 LDS from the ring) -> V_t, a_t,
//       Z_t as 12 conflict-free STS into a 128B-swizzled staging box -> Z_t by stmatrix into the fp16 spike tile -> the
//       step's ONE barrier.  No global memory instruction at all.
//   the traces leave by TMA: every kTcK steps ONE cp.async.bulk.tensor store per array writes the box
//       {32 neurons, 8 rows, 4 neuron groups, kTcK steps} of the (B, T, H) tensor (a 4-D view: H = 4 x 32) straight
//       from the staging buffer -- no LSU traffic, full-line writes; rows past the batch are clipped by the map.
//   4 HELPER warps (helper h: neurons 32 h ..+31), one step behind: cp.async of the input current of step t + kTcDist
//       into the ring (same swizzled layout); 4 MMAs: readout partial of Z_{t-1} over its 32 neurons, whose spare row
//       15 (A[15][k] = 2^k) returns the 16 spike bits of each k-tile per row, exact in fp32 -> bit-packed raster.
//   1 SCAN warp: sums the four readout partials, leaky scan, max over time (two steps behind); its lane 0 issues the
//       TMA stores.
constexpr int kTcFwdThreads = 13 * 32;
constexpr int kTcSlots = 8;        // ring slots (steps of input current resident in shared memory)
constexpr int kTcDist = 6;         // steps between a copy and its use
constexpr int kTcK = 4;            // steps per trace box (one TMA store per array)
constexpr int kTcSlab = 4096;      // bytes of one step of one array in the swizzled layout: [4 hq][8 rows][32 hr] floats

__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t saddr, const void* g)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Byte offset of element (row b, neuron n) inside a 4 KB slab: line = (n / 32) * 8 + b, the 16-byte chunk index
// (n % 32) / 4 XOR-ed with line % 8 = b  (TMA SWIZZLE_128B over 128-byte lines; the slab is 1024-byte aligned).
__host__ __device__ constexpr uint32_t tc_slab_off(int b, int n)
{
    return (uint32_t)((((n >> 5) * 8 + b) << 7) | (((((n & 31) >> 2) ^ b) & 7) << 4) | ((n & 3) << 2));
}

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t saddr, int c0, int c1, int c2, int c3)
{
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
                 ::"l"(map), "r"(saddr), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

constexpr size_t fwd_tc_smem_bytes(int T)
{
    return 1024                                                                           // alignment slack (swizzle atoms)
           + (size_t)2 * 3 * kTcK * kTcSlab                                               // staging [2][V, a, Z][kTcK] slabs
           + (size_t)kTcSlots * kTcSlab                                                   // input-current ring
           + sizeof(__half) * 2 * kTcRows * kTcTileStride                                 // spike tiles [2][8][136]
           + sizeof(float) * 2 * 4 * 32 * 4                                               // readout partials [2][helper][lane][4]
           + sizeof(int) * (size_t)((kTcRows * T + 3) & ~3)                               // compact row of every (row, step)
           + sizeof(float) * 16;
}

// grid = ceil(B / 8), block = 416.  Recurrent layers only (without the matvec the scan kernels have nothing to lose).
// mV / mA / mZ: 4-D maps {32, B, 4, T} (strides T H, 32, H floats) of the trace tensors, box {32, 8, 4, kTcK}, SWIZZLE_128B.
template <bool ALIF>
__global__ void __launch_bounds__(kTcFwdThreads, 1) k_recur_fwd_tc(const FwdParams p, const __grid_constant__ CUtensorMap mV,
                                                                  const __grid_constant__ CUtensorMap mA,
                                                                  const __grid_constant__ CUtensorMap mZ)
{
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    constexpr int H = kTcH;
    const int T = p.T, O = p.O, B = p.B;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const int b0 = blockIdx.x * kTcRows;
    const int nvalid = min(kTcRows, B - b0);

    unsigned char* smem_raw = smem_dyn + ((1024u - (tc::smem_u32(smem_dyn) & 1023u)) & 1023u);
    unsigned char* s_stage = smem_raw;                                                           // [2][3][kTcK][4096]
    unsigned char* s_ring = s_stage + 2 * 3 * kTcK * kTcSlab;                                    // [kTcSlots][4096]
    __half* s_z = reinterpret_cast<__half*>(s_ring + kTcSlots * kTcSlab);                        // [2][8][136]
    float* s_yp = reinterpret_cast<float*>(s_z + 2 * kTcRows * kTcTileStride);                   // [2][4][32][4]
    int* s_r2c = reinterpret_cast<int*>(s_yp + 2 * 4 * 32 * 4);                                  // [8][T]
    float* s_red = reinterpret_cast<float*>(s_r2c + ((kTcRows * T + 3) & ~3));                   // [16]

    // frame-dedup variant: row table[b*T + t] of the compact projection I_u instead of row b*T + t of I_in.
    const bool compact = p.run_table != nullptr && p.run_table[1] == 1;
    if (compact)
        for (int idx = tid; idx < nvalid * T; idx += kTcFwdThreads)
            s_r2c[idx] = __ldg(p.run_table + kRunHdrInts + (size_t)b0 * T + idx);      // rows b0.. are consecutive
    // spike tiles: buffer 1 holds Z_{-1} (the initial state), read by step 0
    for (int idx = tid; idx < 2 * kTcRows * kTcTileStride; idx += kTcFwdThreads) s_z[idx] = __float2half_rn(0.f);
    __syncthreads();
    if (p.Z0)
        for (int idx = tid; idx < kTcRows * H; idx += kTcFwdThreads) {
            const int r = idx / H, c = idx - r * H;
            if (b0 + r < B) s_z[(kTcRows + r) * kTcTileStride + c] = __float2half_rn(p.Z0[(size_t)(b0 + r) * H + c]);
        }
    constexpr uint32_t kTileBytes = kTcRows * kTcTileStride * 2;
    const uint32_t z_u32 = tc::smem_u32(s_z);
    const bool traces = p.traces != 0;
    // barrier count of every role: 1 (above) + 4 (two block maxima) + 1 (ready) + T + 1

    if (warp < 8) {
        // ---------------- neuron warps: neurons 16 warp .. 16 warp + 15 ----------------
        const int i0 = 16 * warp;
        uint32_t ah[8][4], al[8][4];          // W_eff^T fragments, two fp16 planes: 64 registers for the whole sequence
        float inv_s;
        {
            float raw[8][8];
            load_a_raw<8>(p.W_eff, H, i0, H, g, tig, raw);
            const float mx = block_max_tc<kTcFwdThreads>(absmax_raw<8>(raw), s_red);
            const float s = pow2_scale_for(mx);
            inv_s = __fdiv_rn(1.0f, s);
            split_a<8>(raw, s, ah, al);
            block_max_tc<kTcFwdThreads>(0.f, s_red);      // the helpers' reduction (readout scale)
        }
        const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
        const float alpha = p.alpha, rho = p.rho, theta = p.theta;
        // Rows past the batch compute on a copy of the last valid row (their columns of the MMA are independent); the
        // trace boxes are clipped at the batch by the tensor maps.
        float v[4], a[4], zp[4], nz[4];       // zp = Z_{t-1}, nz = 1 - Z_{t-1}
        uint32_t eo[4];                       // slab offsets of the 4 elements
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int rowc = min(2 * tig + (e & 1), nvalid - 1);
            const size_t s = (size_t)(b0 + rowc) * H + i0 + g + 8 * (e >> 1);
            v[e] = p.V0 ? p.V0[s] : 0.f;
            a[e] = p.a0 ? p.a0[s] : 0.f;
            zp[e] = p.Z0 ? p.Z0[s] : 0.f;
            nz[e] = __fsub_rn(1.0f, zp[e]);
            eo[e] = tc_slab_off(2 * tig + (e & 1), i0 + g + 8 * (e >> 1));
        }
        // ldmatrix source of this lane inside a tile: matrix j = lane >> 3 covers k = 8 j .. 8 j + 7 of a 32-wide k group
        const uint32_t tile_base = z_u32 + (uint32_t)((lane & 7) * kTcTileStride + 8 * (lane >> 3)) * 2;
        const uint32_t st_off = (uint32_t)((lane & 7) * kTcTileStride + i0 + 8 * ((lane >> 3) & 1)) * 2;
        const uint32_t ring_u32 = tc::smem_u32(s_ring), stage_u32 = tc::smem_u32(s_stage);
        __syncthreads();      // ready: tiles, table and the first ring slot

        for (int t = 0; t < T; ++t) {
            const uint32_t rd = ((t + 1) & 1) * kTileBytes;
            // B fragments of Z_{t-1}: bfr[kt] = (k = 16 kt + 2 tig + {0,1}, n = g), (k + 8 ..)
            uint32_t bfr[8][2];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t r[4];
                ldsm_x4(r, tile_base + rd + q * 64);
                bfr[2 * q][0] = r[0]; bfr[2 * q][1] = r[1]; bfr[2 * q + 1][0] = r[2]; bfr[2 * q + 1][1] = r[3];
            }
            float cur[4];
            {
                const uint32_t cs = ring_u32 + (uint32_t)(t & (kTcSlots - 1)) * kTcSlab;
#pragma unroll
                for (int e = 0; e < 4; ++e) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(cur[e]) : "r"(cs + eo[e]));
            }
            float ch[4] = {0.f, 0.f, 0.f, 0.f}, cl[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int kt = 0; kt < 8; ++kt) {
                mma_f16(ch, ah[kt], bfr[kt]);
                mma_f16(cl, al[kt], bfr[kt]);
            }
            bool spk[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float rec = __fmul_rn(fmaf(cl[e], 1.0f / 2048.0f, ch[e]), inv_s);
                // V' = (alpha V + I_in + I_rec)(1 - Z.detach())          spiking_layers.py:169/239
                const float t1 = __fmul_rn(alpha, v[e]);
                const float t2 = __fadd_rn(t1, cur[e]);
                const float t3 = __fadd_rn(t2, rec);
                const float vn = __fmul_rn(t3, nz[e]);
                float thr = theta;
                if constexpr (ALIF) {
                    a[e] = __fadd_rn(__fmul_rn(rho, a[e]), zp[e]);                   // :240
                    thr = __fadd_rn(theta, __fmul_rn(beta, a[e]));                   // :241
                }
                spk[e] = vn >= thr;                                                  // spike_funcs.py:27-28
                zp[e] = spk[e] ? 1.0f : 0.0f;
                nz[e] = spk[e] ? 0.0f : 1.0f;
                v[e] = vn;
            }
            if (traces) {      // V_t, a_t, Z_t into the staging box of steps kTcK * (t / kTcK) ..
                const uint32_t sb = stage_u32 + (uint32_t)(((t / kTcK) & 1) * 3 * kTcK + (t % kTcK)) * kTcSlab;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    asm volatile("st.shared.f32 [%0], %1;" ::"r"(sb + eo[e]), "f"(v[e]) : "memory");
                    if constexpr (ALIF) asm volatile("st.shared.f32 [%0], %1;" ::"r"(sb + eo[e] + kTcK * kTcSlab), "f"(a[e]) : "memory");
                    asm volatile("st.shared.f32 [%0], %1;" ::"r"(sb + eo[e] + 2 * kTcK * kTcSlab), "f"(zp[e]) : "memory");
                }
                if ((t % kTcK) == kTcK - 1 || t == T - 1) fence_proxy_async();      // box complete: visible to the TMA store
            }
            // publish Z_t: tile[t & 1][row n][i0 + 8 j + m]  (matrix j: lanes 8 j .. 8 j + 7 give the row addresses);
            // fp16 1.0 = 0x3C00
            const uint32_t zp0 = (spk[0] ? 0x3C00u : 0u) | (spk[1] ? 0x3C000000u : 0u);
            const uint32_t zp1 = (spk[2] ? 0x3C00u : 0u) | (spk[3] ? 0x3C000000u : 0u);
            stsm_x2_trans(z_u32 + (t & 1) * kTileBytes + st_off, zp0, zp1);
            __syncthreads();
        }
        __syncthreads();      // the helpers' / scan warp's flush step
    } else if (warp < 12) {
        // ---------------- helper warps: neurons 32 h .. 32 h + 31 ----------------
        const int h = warp - 8;
        block_max_tc<kTcFwdThreads>(0.f, s_red);      // the neuron warps' reduction (recurrent scale)
        // readout: A[m = class][k = neuron 32 h + 16 j + k] = W_out[.][m] for the two k-tiles j = 0, 1 of this helper
        uint32_t oh[2][4], ol[2][4];
        float inv_so;
        {
            float ro[2][8];
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const int k = 2 * tig + (q & 1) + 8 * (q >> 2), m = g + 8 * ((q >> 1) & 1);
                    ro[j][q] = m < O ? __ldg(p.W_out + (size_t)(32 * h + 16 * j + k) * O + m) : 0.f;
                }
            const float mo = block_max_tc<kTcFwdThreads>(absmax_raw<2>(ro), s_red);
            const float so = pow2_scale_for(mo);
            inv_so = __fdiv_rn(1.0f, so);
            split_a<2>(ro, so, oh, ol);
            if (g == 7) {
                // row m = 15 (no class lives there: O <= 15 on this path) of the hi planes: A[15][k] = 2^k, so that
                // D[15][n] = sum_k 2^k Z[n][k-tile neuron k] = the 16 spike bits of row n, exact in fp32.  This thread
                // holds a1 = (m 15, k 2 tig, 2 tig + 1) and a3 = (m 15, k 2 tig + 8, 2 tig + 9).
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    oh[j][1] = pack_h2(__float2half_rn((float)(1u << (2 * tig))), __float2half_rn((float)(2u << (2 * tig))));
                    oh[j][3] = pack_h2(__float2half_rn((float)(256u << (2 * tig))), __float2half_rn((float)(512u << (2 * tig))));
                    ol[j][1] = 0u;
                    ol[j][3] = 0u;
                }
            }
        }
        // input current of step ts: this helper fills the 8 lines (rows) of neuron group h of the slot, 64 chunks of
        // 16 bytes, two per lane: chunk (row = lane >> 3 (+ 4), c = lane & 7) -> swizzled position c ^ row
        const int c = lane & 7;
        const int rwA = lane >> 3, rwB = rwA + 4;
        const int rcA = min(rwA, nvalid - 1), rcB = min(rwB, nvalid - 1);
        const float* srcA = p.I_in + ((size_t)(b0 + rcA) * T) * H + 32 * h + 4 * c;
        const float* srcB = p.I_in + ((size_t)(b0 + rcB) * T) * H + 32 * h + 4 * c;
        const float* src_u = p.I_u + 32 * h + 4 * c;
        const int* r2cA = s_r2c + rcA * T;
        const int* r2cB = s_r2c + rcB * T;
        const uint32_t dA = tc::smem_u32(s_ring) + (uint32_t)(((h * 8 + rwA) << 7) | ((c ^ rwA) << 4));
        const uint32_t dB = tc::smem_u32(s_ring) + (uint32_t)(((h * 8 + rwB) << 7) | ((c ^ rwB) << 4));
        auto prefetch = [&](int ts) {
            if (ts < T) {
                const uint32_t so = (uint32_t)(ts & (kTcSlots - 1)) * kTcSlab;
                cp_async16(dA + so, compact ? src_u + (size_t)r2cA[ts] * H : srcA + (size_t)ts * H);
                cp_async16(dB + so, compact ? src_u + (size_t)r2cB[ts] * H : srcB + (size_t)ts * H);
            }
            cp_async_commit();
        };
#pragma unroll
        for (int d = 0; d < kTcDist; ++d) prefetch(d);
        cp_async_wait<kTcDist - 1>();      // step 0 has landed
        const uint32_t own_off = (uint32_t)(g * kTcTileStride + 32 * h + 2 * tig) * 2;      // B fragment (n = g) of k-tile 2 h
        const int rA = 2 * tig, rB = 2 * tig + 1;                                            // rows of this lane's D fragment
        const bool zstA = g == 7 && rA < nvalid, zstB = g == 7 && rB < nvalid;
        size_t zoffA = ((size_t)(b0 + min(rA, nvalid - 1)) * T) * (H / 32) + h;
        size_t zoffB = ((size_t)(b0 + min(rB, nvalid - 1)) * T) * (H / 32) + h;
        __syncthreads();      // ready

        for (int t = 0; t <= T; ++t) {
            prefetch(t + kTcDist);
            if (t >= 1) {
                const int pb = (t + 1) & 1;      // tile written during step t - 1
                // ---- readout partial of step t-1 over this helper's 32 neurons + the spike bits ----
                float yh0[4] = {0.f, 0.f, 0.f, 0.f}, yh1[4] = {0.f, 0.f, 0.f, 0.f}, yl[4] = {0.f, 0.f, 0.f, 0.f};
                uint32_t bA[2], bB[2];
                const uint32_t ta = z_u32 + pb * kTileBytes + own_off;
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(bA[0]) : "r"(ta));
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(bA[1]) : "r"(ta + 16));
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(bB[0]) : "r"(ta + 32));
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(bB[1]) : "r"(ta + 48));
                mma_f16(yh0, oh[0], bA);
                mma_f16(yh1, oh[1], bB);
                mma_f16(yl, ol[0], bA);
                mma_f16(yl, ol[1], bB);
                if (zstA) p.zbits[zoffA] = __float2uint_rn(yh0[2]) | (__float2uint_rn(yh1[2]) << 16);
                if (zstB) p.zbits[zoffB] = __float2uint_rn(yh0[3]) | (__float2uint_rn(yh1[3]) << 16);
                zoffA += H / 32;
                zoffB += H / 32;
                float4 part;
                part.x = __fmul_rn(fmaf(yl[0], 1.0f / 2048.0f, __fadd_rn(yh0[0], yh1[0])), inv_so);
                part.y = __fmul_rn(fmaf(yl[1], 1.0f / 2048.0f, __fadd_rn(yh0[1], yh1[1])), inv_so);
                part.z = __fmul_rn(fmaf(yl[2], 1.0f / 2048.0f, __fadd_rn(yh0[2], yh1[2])), inv_so);
                part.w = __fmul_rn(fmaf(yl[3], 1.0f / 2048.0f, __fadd_rn(yh0[3], yh1[3])), inv_so);
                reinterpret_cast<float4*>(s_yp)[((t & 1) * 4 + h) * 32 + lane] = part;
            }
            cp_async_wait<kTcDist - 1>();      // the input current of step t + 1 has landed
            __syncthreads();
        }
        cp_async_wait<0>();
    } else {
        // ---------------- scan warp: TMA trace stores; readout scan + max over time, two steps behind ----------------
        block_max_tc<kTcFwdThreads>(0.f, s_red);
        block_max_tc<kTcFwdThreads>(0.f, s_red);
        float yv[4], mx[4], bias[4];
        int mt[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int cls = g + 8 * (e >> 1);
            yv[e] = 0.f; mx[e] = 0.f; mt[e] = 0;
            bias[e] = cls < O ? __ldg(p.b_out + cls) : 0.f;
        }
        const float kappa = p.kappa;
        auto finish_y = [&](int ty, int buf) {      // y_ty = kappa y_{ty-1} + sum of the 4 helpers' partials + b
            float4 q[4];
#pragma unroll
            for (int w = 0; w < 4; ++w) q[w] = reinterpret_cast<const float4*>(s_yp)[(buf * 4 + w) * 32 + lane];
            float s4[4] = {q[0].x, q[0].y, q[0].z, q[0].w};
            // ascending neuron blocks (the order of the fp32 kernels' neuron sum, coarsened to 32-neuron blocks)
#pragma unroll
            for (int w = 1; w < 4; ++w) {
                s4[0] = __fadd_rn(s4[0], q[w].x); s4[1] = __fadd_rn(s4[1], q[w].y);
                s4[2] = __fadd_rn(s4[2], q[w].z); s4[3] = __fadd_rn(s4[3], q[w].w);
            }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int cls = g + 8 * (e >> 1), row = 2 * tig + (e & 1);
                const float y = __fadd_rn(__fadd_rn(__fmul_rn(kappa, yv[e]), s4[e]), bias[e]);     // spiking_layers.py:407
                yv[e] = y;
                if (ty == 0 || y > mx[e]) { mx[e] = y; mt[e] = ty; }                                 // first max wins (snn.py:228)
                if (cls < O && b0 + row < B) p.y[((size_t)(b0 + row) * T + ty) * O + cls] = y;
            }
        };
        const uint32_t stage_u32 = tc::smem_u32(s_stage);
        if (lane == 0 && traces) {
            tc::prefetch_tmap(&mV);
            tc::prefetch_tmap(&mZ);
            if (ALIF) tc::prefetch_tmap(&mA);
        }
        __syncthreads();      // ready
        for (int t = 0; t <= T; ++t) {
            // the box of steps kTcK q .. was completed by step t - 1 (t a multiple of kTcK, or the last, partial box)
            if (traces && lane == 0 && t >= 1 && ((t % kTcK) == 0 || t == T)) {
                const int q = (t - 1) / kTcK;
                const uint32_t sb = stage_u32 + (uint32_t)((q & 1) * 3 * kTcK) * kTcSlab;
                tma_store_4d(&mV, sb, 0, b0, 0, q * kTcK);
                if (ALIF) tma_store_4d(&mA, sb + kTcK * kTcSlab, 0, b0, 0, q * kTcK);
                tma_store_4d(&mZ, sb + 2 * kTcK * kTcSlab, 0, b0, 0, q * kTcK);
                tma_store_commit();
            }
            if (t >= 2) finish_y(t - 2, (t - 1) & 1);
            // the other staging buffer is written again from step t + 1 on: its store must have read it by then
            if (traces && lane == 0 && (t % kTcK) == kTcK - 1) tma_store_wait_read();
            __syncthreads();
        }
        finish_y(T - 1, T & 1);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int cls = g + 8 * (e >> 1), row = 2 * tig + (e & 1);
            if (cls < O && b0 + row < B) {
                p.logits[(size_t)(b0 + row) * O + cls] = mx[e];
                p.tstar[(size_t)(b0 + row) * O + cls] = mt[e];
            }
        }
        if (lane == 0) tma_store_wait_all();
    }
}

// ---- readout adjoint scan (pre-pass of the tensor-core sweep) ----------------------------------------------------------
// gy_t = seed_t + kappa gy_{t+1}  (spiking_layers.py:407 backwards) for every (row, class) -> gy_scan (B, T, kOMax), zero
// in the padded classes.  It does not depend on the recurrence, so it runs before the sweep; dW_out and db are
// contractions of it with the spike raster (k_wout_grad, recur_gen.cuh) and run BESIDE the sweep on the idle SMs.
__global__ void __launch_bounds__(256) k_gy_scan(int B, int T, int O, float kappa, const float* __restrict__ g_y,
                                                const float* __restrict__ g_logits, const int32_t* __restrict__ tstar,
                                                const float* __restrict__ g_scale, float* __restrict__ gy_scan)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = idx / kOMax, c = idx - b * kOMax;
    if (b >= B) return;
    float* out = gy_scan + (size_t)b * T * kOMax + c;
    if (c >= O) {
        for (int t = 0; t < T; ++t) out[(size_t)t * kOMax] = 0.f;
        return;
    }
    float g = 0.f;
    if (g_y) {
        const float* src = g_y + (size_t)b * T * O + c;
        for (int t = T - 1; t >= 0; --t) {
            g = __fadd_rn(__ldg(src + (size_t)t * O), __fmul_rn(kappa, g));
            out[(size_t)t * kOMax] = g;
        }
    } else {
        const float scale = g_scale ? __ldg(g_scale) : 1.0f;
        const int ts = __ldg(tstar + (size_t)b * O + c);
        const float seed = __fmul_rn(__ldg(g_logits + (size_t)b * O + c), scale);
        for (int t = T - 1; t >= 0; --t) {
            g = __fadd_rn(t == ts ? seed : 0.f, __fmul_rn(kappa, g));
            out[(size_t)t * kOMax] = g;
        }
    }
}

// ---- backward -------------------------------------------------------------------------------------------------------
__host__ __device__ constexpr int tc_zstride(int T) { return ((T + 1) * (kTcH / 32) + 3) & ~3; }      // words per row of the spike-word table

constexpr int kTcKb = 2;           // steps per gI box (one TMA store per plane); the saved traces arrive in boxes of kTcK steps

constexpr size_t bwd_tc_smem_bytes(int T)
{
    return 1024                                                                             // alignment slack (swizzle atoms)
           + (size_t)2 * 2 * kTcK * kTcSlab                                                 // trace boxes [2][V, a][kTcK] slabs
           + (size_t)3 * 2 * kTcKb * kTcSlab                                                // gI staging [3][hi, lo][kTcKb] slabs
           + sizeof(__half) * 2 * 2 * kTcRows * kTcTileStride                               // gI tiles [buf][plane][8][136]
           + sizeof(__half) * 2 * (size_t)T * kTcRows * 16                                  // gy planes [plane][T][8][16]
           + sizeof(uint32_t) * (size_t)kTcRows * tc_zstride(T)                             // spike words [8][T+1][4] (slot 0: Z_{-1})
           + sizeof(uint32_t) * (size_t)kTcRows * ((T + 31) / 32 + 1)                        // run-start bits
           + sizeof(float) * 16 + sizeof(uint64_t) * 2 + 8;
}

// Surrogate derivatives with the hardware reciprocal (1 ulp): the tensor-core sweep does not promise the fp32 kernels'
// bit pattern anyway (22-bit operands), and __frcp_rn / __fdiv_rn are 8-15 instructions each on this issue-bound path.
__device__ __forceinline__ float rcp_fast(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
template <int SURR>
__device__ __forceinline__ float surrogate_grad_fast(float gamma, float v, float thr)
{
    if constexpr (SURR == kSurrTrace) {
        return v;                   // the streamed value is sigma' (common.cuh)
    } else if constexpr (SURR == 0) {      // spike_funcs.py:59-62
        const float d = fmaf(gamma, fabsf(__fsub_rn(v, thr)), 1.0f);
        return rcp_fast(__fmul_rn(d, d));
    } else {                        // spike_funcs.py:75-79
        const float inv = rcp_fast(__fadd_rn(thr, 1e-5f));
        const float r = fmaxf(__fsub_rn(1.0f, fabsf(__fmul_rn(__fsub_rn(v, thr), inv))), 0.f);
        return __fmul_rn(__fmul_rn(gamma, inv), r);
    }
}

// The gradient tile of a step is published as two fp16 planes under a power-of-two scale 2^kexp that is STICKY: it
// changes only when the largest exponent class of a tile (classes of 8 binades, OR-ed into a shared word before the
// step's barrier) leaves the window in which fp16 still carries 22 bits relative to the tile's maximum
// (scaled maximum in [2^-14, 2^10): one class up, two classes down).  A tile found outside the window when it is
// about to be read is re-published under the new scale (one extra barrier; happens a handful of times per sequence),
// so the common step has ONE barrier.  All threads derive the decision from the same shared word: it is uniform.
struct TcScale {
    int top;          // exponent class the current scale was chosen for
    float s, inv;     // 2^kexp and its reciprocal
    __device__ __forceinline__ void set(int t)
    {
        top = t;
        int kexp = 129 - 8 * t;                          // scaled maximum in [2^2, 2^10)
        kexp = kexp > 126 ? 126 : (kexp < -126 ? -126 : kexp);
        s = __uint_as_float((uint32_t)(kexp + 127) << 23);
        inv = __uint_as_float((uint32_t)(127 - kexp) << 23);
    }
    // mask: exponent classes present in the tile about to be read; true -> the tile must be re-published
    __device__ __forceinline__ bool update(uint32_t mask)
    {
        if (!mask) return false;
        const int t = 31 - __clz(mask);
        if (t <= top && t >= top - 2) return false;
        set(t);
        return true;
    }
};

// grid = ceil(B / 8), block = 288.  gy_scan: output of k_gy_scan.  Writes gI (one or two tf32 planes) and, with a
// frame-run table, the run sums; dW_out / db are NOT produced here (k_wout_grad).
// Memory paths (same reasoning as the forward kernel: the LSU is the bound, so nothing avoidable goes through it): the
// saved traces V_t (a_t) arrive as TMA tensor loads of {32, 8, 4, kTcK} boxes into 128B-swizzled slabs (two boxes, one
// in use, one in flight; mbarrier completion), gI leaves through swizzled staging slabs by TMA tensor stores every
// kTcKb steps; both are issued by lane 0 of the ninth warp.  mV / mA: box kTcK steps; mG / mGlo: box kTcKb steps.
template <bool ALIF, int SURR>
__global__ void __launch_bounds__(kTcThreads, 1) k_recur_bwd_tc(const BwdParams p, const float* __restrict__ gy_scan,
                                                               const __grid_constant__ CUtensorMap mV,
                                                               const __grid_constant__ CUtensorMap mA,
                                                               const __grid_constant__ CUtensorMap mG,
                                                               const __grid_constant__ CUtensorMap mGlo)
{
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    constexpr int H = kTcH, W32 = kTcH / 32;
    const int T = p.T, B = p.B, O = p.O;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const int b0 = blockIdx.x * kTcRows;
    const int nvalid = min(kTcRows, B - b0);
    const int zstride = tc_zstride(T);
    const int TW = (T + 31) / 32 + 1;

    unsigned char* smem_raw = smem_dyn + ((1024u - (tc::smem_u32(smem_dyn) & 1023u)) & 1023u);
    unsigned char* s_in = smem_raw;                                                          // [2][2][kTcK][4096]
    unsigned char* s_out = s_in + 2 * 2 * kTcK * kTcSlab;                                    // [3][2][kTcKb][4096]
    __half* s_g = reinterpret_cast<__half*>(s_out + 3 * 2 * kTcKb * kTcSlab);                // [2][2][8][136]
    __half* s_gy = s_g + 2 * 2 * kTcRows * kTcTileStride;                                    // [2][T][8][16]
    uint32_t* s_zw = reinterpret_cast<uint32_t*>(s_gy + 2 * (size_t)T * kTcRows * 16);       // [8][zstride]
    uint32_t* s_start = s_zw + (size_t)kTcRows * zstride;                                    // [8][TW]
    float* s_red = reinterpret_cast<float*>(s_start + kTcRows * TW);                         // [12] + exponent-class words [3]
    uint32_t* s_cls = reinterpret_cast<uint32_t*>(s_red + 12);
    uint64_t* s_full = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s_cls + 4) + 7) & ~uintptr_t(7));   // [2]

    // trace boxes in processing order j = 0, 1, ...: steps kTcK (nbox - 1 - j) .., buffer j & 1, parity (j >> 1) & 1
    const int nbox = (T + kTcK - 1) / kTcK;
    constexpr uint32_t kInBox = 2 * kTcK * kTcSlab;                                          // one buffer: V slabs then a slabs
    auto issue_box = [&](int j) {      // lane 0 of the ninth warp
        const int q = nbox - 1 - j;
        uint64_t* bar = s_full + (j & 1);
        unsigned char* dst = s_in + (size_t)(j & 1) * kInBox;
        tc::mbar_expect_tx(bar, (uint32_t)(kTcK * kTcSlab) * (ALIF ? 2u : 1u));
        tc::tma_load_4d(dst, &mV, bar, 0, b0, 0, q * kTcK);
        if (ALIF) tc::tma_load_4d(dst + kTcK * kTcSlab, &mA, bar, 0, b0, 0, q * kTcK);
    };
    if (tid == 256) {
        tc::mbar_init(s_full, 1);
        tc::mbar_init(s_full + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        tc::prefetch_tmap(&mV);
        tc::prefetch_tmap(&mG);
        issue_box(0);
        if (nbox > 1) issue_box(1);
    }

    const bool run_sums = p.run_table != nullptr && p.run_table[1] == 1;
    if (tid == 256) s_cls[0] = s_cls[1] = s_cls[2] = 0u;
    // gradient tiles start at zero (gI_T = 0)
    for (int idx = tid; idx < 2 * 2 * kTcRows * kTcTileStride; idx += kTcThreads) s_g[idx] = __float2half_rn(0.f);
    // spike words: slot 0 of a row is Z_{-1} (initial state), slot t + 1 is Z_t
    for (int idx = tid; idx < kTcRows * (T + 1) * W32; idx += kTcThreads) {
        const int r = idx / ((T + 1) * W32), rem = idx - r * ((T + 1) * W32);
        const int ts = rem / W32, wd = rem - ts * W32;
        uint32_t w = 0u;
        if (b0 + r < B) {
            if (ts > 0) w = __ldg(p.zbits + ((size_t)(b0 + r) * T + ts - 1) * W32 + wd);
            else if (p.Z0) {
                for (int l = 0; l < 32; ++l)
                    if (__ldg(p.Z0 + (size_t)(b0 + r) * H + wd * 32 + l) != 0.f) w |= 1u << l;
            }
        }
        s_zw[r * zstride + rem] = w;
    }
    if (run_sums) {
        for (int idx = tid; idx < kTcRows * TW; idx += kTcThreads) s_start[idx] = 0u;
    }
    __syncthreads();
    if (run_sums) {
        // bit t of a row's word: step t is the first of its run of equal input frames
        for (int idx = tid; idx < nvalid * T; idx += kTcThreads) {
            const int r = idx / T, t = idx - r * T;
            const int* rc = p.run_table + kRunHdrInts + (size_t)(b0 + r) * T;
            if (t == 0 || __ldg(rc + t) != __ldg(rc + t - 1)) atomicOr(s_start + r * TW + (t >> 5), 1u << (t & 31));
        }
        if (blockIdx.x == 0) {   // the weight-gradient GEMM contracts whole 32-row blocks: zero the tail of the last one
            const int n_rows = p.run_table[0], n_pad = (n_rows + 31) & ~31;
            for (int idx = tid; idx < (n_pad - n_rows) * H; idx += kTcThreads) {
                p.Gu_hi[(size_t)n_rows * H + idx] = 0.f;
                p.Gu_lo[(size_t)n_rows * H + idx] = 0.f;
            }
        }
    }
    // readout adjoint of the tile as two fp16 planes: B operand (k = class, n = row) of every step
    float gymax = 0.f;
    for (int idx = tid; idx < nvalid * T * kOMax; idx += kTcThreads) gymax = fmaxf(gymax, fabsf(__ldg(gy_scan + (size_t)b0 * T * kOMax + idx)));
    gymax = block_max_tc(gymax, s_red);
    const float s_gyscale = pow2_scale_for(gymax);
    for (int idx = tid; idx < kTcRows * T * kOMax; idx += kTcThreads) {
        const int r = idx / (T * kOMax), rem = idx - r * (T * kOMax);
        const int t = rem / kOMax, c = rem - t * kOMax;
        __half hi = __float2half_rn(0.f), lo = hi;
        if (r < nvalid) split_h2(__fmul_rn(__ldg(gy_scan + (size_t)(b0 + r) * T * kOMax + rem), s_gyscale), hi, lo);
        s_gy[(t * kTcRows + r) * 16 + c] = hi;
        s_gy[((size_t)T * kTcRows + t * kTcRows + r) * 16 + c] = lo;
    }

    constexpr uint32_t kTileBytes = kTcRows * kTcTileStride * 2;       // one plane of one buffer
    const uint32_t g_u32 = tc::smem_u32(s_g);
    const uint32_t tile_base = g_u32 + (uint32_t)((lane & 7) * kTcTileStride + 8 * (lane >> 3)) * 2;
    // ldmatrix.x4 source inside the gy planes: matrices (hi k 0-7, hi k 8-15, lo k 0-7, lo k 8-15)
    const uint32_t gy_base = tc::smem_u32(s_gy) + (uint32_t)(((lane >> 4) * T * kTcRows + (lane & 7)) * 16 + 8 * ((lane >> 3) & 1)) * 2;

    TcScale sc;
    sc.set(16);
    int c_rd = 0, c_wr = 1, c_zr = 2;      // exponent-class words: of the tile being read, being written, to clear

    if (warp < 8) {
        const int i0 = 16 * warp;
        uint32_t ah[8][4], al[8][4];          // rows i0.. of W_eff as A fragments: A[m][k] = W_eff[i0 + m][k] = W_effT[k][i0 + m]
        uint32_t oh[4], ol[4];                // A[m][k = class] = W_out[i0 + m][k]
        float inv_sw, inv_so;
        {
            float raw[8][8];
            load_a_raw<8>(p.W_effT, H, i0, H, g, tig, raw);
            const float s = pow2_scale_for(block_max_tc(absmax_raw<8>(raw), s_red));
            inv_sw = __fdiv_rn(1.0f, s);
            split_a<8>(raw, s, ah, al);
            float ro[1][8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int k = 2 * tig + (q & 1) + 8 * (q >> 2), m = g + 8 * ((q >> 1) & 1);
                ro[0][q] = k < O ? __ldg(p.W_out + (size_t)(i0 + m) * O + k) : 0.f;
            }
            const float so = pow2_scale_for(block_max_tc(absmax_raw<1>(ro), s_red));
            inv_so = __fdiv_rn(__fdiv_rn(1.0f, so), s_gyscale);       // both scales of the readout-adjoint product
            uint32_t th[1][4], tl[1][4];
            split_a<1>(ro, so, th, tl);
#pragma unroll
            for (int r = 0; r < 4; ++r) { oh[r] = th[0][r]; ol[r] = tl[0][r]; }
        }
        const float beta = (ALIF && p.beta) ? __ldg(p.beta) : 0.f;
        const float alpha = p.alpha, theta = p.theta, gamma = p.gamma;
        // element e = 2 nh + rh: neuron i0 + g + 8 nh, row 2 tig + rh.  Rows past the batch sweep a copy of the last
        // valid row (their columns of the MMA are independent) and store nothing.
        float gv[4], racc[4], gi[4];
        int crow[2], rowc[2];
        uint32_t sbits[2], wt[2];
        bool okr[2];
#pragma unroll
        for (int e = 0; e < 4; ++e) { gv[e] = 0.f; racc[e] = 0.f; gi[e] = 0.f; }
#pragma unroll
        for (int rh = 0; rh < 2; ++rh) {
            okr[rh] = b0 + 2 * tig + rh < B;
            rowc[rh] = min(2 * tig + rh, nvalid - 1);
            crow[rh] = run_sums ? __ldg(p.run_table + kRunHdrInts + (size_t)(b0 + rowc[rh]) * T + T - 1) : 0;
            sbits[rh] = 0u;
        }
        const bool sums0 = run_sums && okr[0], sums1 = run_sums && okr[1];
        uint32_t eo[4];      // slab offsets of the 4 elements (trace boxes and gI staging share the layout)
#pragma unroll
        for (int e = 0; e < 4; ++e) eo[e] = tc_slab_off(2 * tig + (e & 1), i0 + g + 8 * (e >> 1));
        // element offset of (row 2 tig + rh, step T - 1, neuron i0 + g) in the (B, T, H) tensors (optional seeds)
        size_t off0 = ((size_t)(b0 + rowc[0]) * T + (T - 1)) * H + i0 + g, off1 = ((size_t)(b0 + rowc[1]) * T + (T - 1)) * H + i0 + g;
        const int zword = warp >> 1, zsh = 16 * (warp & 1) + g;      // this thread's neurons in a spike word: bits zsh, zsh + 8
        const uint32_t* zw0 = s_zw + rowc[0] * zstride + zword;
        const uint32_t* zw1 = s_zw + rowc[1] * zstride + zword;
        const uint32_t* st0p = s_start + rowc[0] * TW;
        const uint32_t* st1p = s_start + rowc[1] * TW;
        const uint32_t in_u32 = tc::smem_u32(s_in), out_u32 = tc::smem_u32(s_out);
        const bool two_planes = p.gI_lo != nullptr;
        auto publish = [&](int buf) {      // gi (registers) -> tile `buf` as two fp16 planes under the current scale
            uint32_t pk[4];
#pragma unroll
            for (int nh = 0; nh < 2; ++nh) {
                __half h0, l0, h1, l1;
                split_h2(__fmul_rn(gi[2 * nh], sc.s), h0, l0);
                split_h2(__fmul_rn(gi[2 * nh + 1], sc.s), h1, l1);
                pk[nh] = pack_h2(h0, h1);
                pk[2 + nh] = pack_h2(l0, l1);
            }
            // matrices: (hi, neurons i0..+7), (hi, i0+8..), (lo, i0..), (lo, i0+8..); lane 8 j + n gives row n of matrix j
            const uint32_t sa = g_u32 + (uint32_t)(((buf * 2 + (lane >> 4)) * kTcRows + (lane & 7)) * kTcTileStride + i0 +
                                                   8 * ((lane >> 3) & 1)) * 2;
            stsm_x4_trans(sa, pk[0], pk[1], pk[2], pk[3]);
        };
        __syncthreads();          // planes and tables visible
        wt[0] = zw0[T * W32];     // Z_{T-1}
        wt[1] = zw1[T * W32];
        const bool has_gZ = p.g_Z != nullptr, has_gV = p.g_V != nullptr;

        int ob = 0;      // gI staging buffer of the current box (rotates over 3)
        for (int t = T - 1; t >= 0; --t) {
            if (sc.update(s_cls[c_rd])) {      // rare: the tile about to be read needs another scale
                publish((t + 1) & 1);
                __syncthreads();
            }
            // ---- gZ^T = W_eff gI_{t+1}^T  +  W_out gy_t^T ----
            float chh[4] = {0.f, 0.f, 0.f, 0.f}, chl[4] = {0.f, 0.f, 0.f, 0.f}, clh[4] = {0.f, 0.f, 0.f, 0.f};
            float ohh[4] = {0.f, 0.f, 0.f, 0.f}, ox[4] = {0.f, 0.f, 0.f, 0.f};
            {
                uint32_t r4[4];
                ldsm_x4(r4, gy_base + (uint32_t)(t * kTcRows * 16) * 2);
                const uint32_t byh[2] = {r4[0], r4[1]}, byl[2] = {r4[2], r4[3]};
                mma_f16(ohh, oh, byh);
                mma_f16(ox, oh, byl);
                mma_f16(ox, ol, byh);
            }
            const uint32_t tb = tile_base + ((t + 1) & 1) * 2 * kTileBytes;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t rh4[4], rl4[4];
                ldsm_x4(rh4, tb + q * 64);
                ldsm_x4(rl4, tb + kTileBytes + q * 64);
                const uint32_t bh0[2] = {rh4[0], rh4[1]}, bh1[2] = {rh4[2], rh4[3]};
                const uint32_t bl0[2] = {rl4[0], rl4[1]}, bl1[2] = {rl4[2], rl4[3]};
                mma_f16(chh, ah[2 * q], bh0);
                mma_f16(chl, ah[2 * q], bl0);
                mma_f16(clh, al[2 * q], bh0);
                mma_f16(chh, ah[2 * q + 1], bh1);
                mma_f16(chl, ah[2 * q + 1], bl1);
                mma_f16(clh, al[2 * q + 1], bh1);
            }
            // saved traces of step t: box j (processing order), buffer j & 1; the first step of a box waits for its load
            float vt[4], at[4];
            {
                const int j = nbox - 1 - t / kTcK;
                if (t == T - 1 || (t % kTcK) == kTcK - 1) tc::mbar_wait(s_full + (j & 1), (uint32_t)((j >> 1) & 1));
                const uint32_t vb = in_u32 + (uint32_t)(j & 1) * kInBox + (uint32_t)(t % kTcK) * kTcSlab;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(vt[e]) : "r"(vb + eo[e]));
                    if constexpr (ALIF) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(at[e]) : "r"(vb + eo[e] + kTcK * kTcSlab));
                    else at[e] = 0.f;
                }
            }
            const uint32_t wp[2] = {zw0[t * W32], zw1[t * W32]};      // Z_{t-1}
            const float sc_rec = __fmul_rn(inv_sw, sc.inv);
            float amax = 0.f;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int nh = e >> 1, rh = e & 1;
                const float rec = __fmul_rn(fmaf(__fadd_rn(chl[e], clh[e]), 1.0f / 2048.0f, chh[e]), sc_rec);
                const float rdo = __fmul_rn(fmaf(ox[e], 1.0f / 2048.0f, ohh[e]), inv_so);
                float s = __fadd_rn(rdo, rec);
                const size_t o = (rh ? off1 : off0) + 8 * nh;
                if (has_gZ) s = __fadd_rn(s, __ldg(p.g_Z + o));
                float thr = theta;
                if constexpr (ALIF) thr = __fadd_rn(theta, __fmul_rn(beta, at[e]));
                const bool zt = (wt[rh] >> (zsh + 8 * nh)) & 1u, zprev = (wp[rh] >> (zsh + 8 * nh)) & 1u;
                const float sg = surrogate_grad_fast<SURR>(gamma, vt[e], thr);
                const float carry = zt ? 0.f : __fmul_rn(alpha, gv[e]);             // alpha gV_{t+1} (1 - Z_t)
                float gq = __fadd_rn(__fmul_rn(s, sg), carry);
                if (has_gV) gq = __fadd_rn(gq, __ldg(p.g_V + o));
                gv[e] = gq;
                gi[e] = zprev ? 0.f : gq;                                           // gI_t = gV_t (1 - Z_{t-1})
                amax = fmaxf(amax, fabsf(gi[e]));
            }
            // gI for the weight-gradient GEMM: staging slab of step t (box t / kTcKb), exact two-plane tf32 split
            {
                const uint32_t sb = out_u32 + (uint32_t)(ob * 2 * kTcKb + (t % kTcKb)) * kTcSlab;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (two_planes) {
                        const float hi = __uint_as_float(__float_as_uint(gi[e]) & 0xFFFFE000u);
                        asm volatile("st.shared.f32 [%0], %1;" ::"r"(sb + eo[e]), "f"(hi) : "memory");
                        asm volatile("st.shared.f32 [%0], %1;" ::"r"(sb + eo[e] + kTcKb * kTcSlab), "f"(__fsub_rn(gi[e], hi)) : "memory");
                    } else {
                        asm volatile("st.shared.f32 [%0], %1;" ::"r"(sb + eo[e]), "f"(gi[e]) : "memory");
                    }
                }
                if ((t % kTcKb) == 0) {      // box complete: visible to the TMA store; next box, next buffer
                    fence_proxy_async();
                    ob = ob == 2 ? 0 : ob + 1;
                }
            }
            off0 -= H;
            off1 -= H;
            if (run_sums) {      // sum of gI over the run of equal input frames this step belongs to
#pragma unroll
                for (int e = 0; e < 4; ++e) racc[e] = __fadd_rn(racc[e], gi[e]);
                if (t == T - 1 || (t & 31) == 31) { sbits[0] = st0p[t >> 5]; sbits[1] = st1p[t >> 5]; }
#pragma unroll
                for (int rh = 0; rh < 2; ++rh) {
                    if ((sbits[rh] >> (t & 31)) & 1u) {
                        if (rh ? sums1 : sums0) {
#pragma unroll
                            for (int nh = 0; nh < 2; ++nh) {
                                const float r = racc[2 * nh + rh];
                                const float hi = __uint_as_float(__float_as_uint(r) & 0xFFFFE000u);
                                const size_t ro = (size_t)crow[rh] * H + i0 + g + 8 * nh;
                                p.Gu_hi[ro] = hi;
                                p.Gu_lo[ro] = __fsub_rn(r, hi);
                            }
                        }
                        racc[rh] = 0.f;
                        racc[2 + rh] = 0.f;
                        --crow[rh];
                    }
                }
            }
            // exponent class of the tile's largest element: warp maximum (positive floats order like their bit
            // patterns), one shared-memory atomicOr per warp
            const uint32_t wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(amax));
            if (lane == 0 && (wmax >> 23) != 0u) atomicOr(s_cls + c_wr, 1u << (wmax >> 26));
            if (tid == 0) s_cls[c_zr] = 0u;
            publish(t & 1);
            wt[0] = wp[0];
            wt[1] = wp[1];
            { const int r = c_rd; c_rd = c_wr; c_wr = c_zr; c_zr = r; }
            __syncthreads();
        }
    } else {
        // ninth warp: takes part in the barriers (the block-wide reductions of the prologue count 288 threads), follows
        // the scale decisions, which may add a barrier, and its lane 0 issues the TMA loads and stores
        block_max_tc(0.f, s_red);
        block_max_tc(0.f, s_red);
        __syncthreads();
        const uint32_t out_u32 = tc::smem_u32(s_out);
        const bool two_planes = p.gI_lo != nullptr;
        int ob = 0;      // staging buffer of the next box to store
        auto after_step = [&](int td) {      // td: the step whose barrier has just completed
            if (lane != 0) return;
            if ((td % kTcK) == 0) {          // last step of trace box j: its buffer is free for box j + 2
                const int j = nbox - 1 - td / kTcK;
                if (j + 2 < nbox) issue_box(j + 2);
            }
            if ((td % kTcKb) == 0) {         // gI box td / kTcKb is complete
                const uint32_t sb = out_u32 + (uint32_t)(ob * 2 * kTcKb) * kTcSlab;
                tma_store_4d(&mG, sb, 0, b0, 0, td);
                if (two_planes) tma_store_4d(&mGlo, sb + kTcKb * kTcSlab, 0, b0, 0, td);
                tma_store_commit();
                ob = ob == 2 ? 0 : ob + 1;
            }
        };
        for (int t = T - 1; t >= 0; --t) {
            if (t < T - 1) after_step(t + 1);
            if (sc.update(s_cls[c_rd])) __syncthreads();
            { const int r = c_rd; c_rd = c_wr; c_wr = c_zr; c_zr = r; }
            // staging buffers rotate over three: the store issued two boxes ago must have read its buffer before the
            // box after this one is written (at most the latest store may still be reading)
            if (lane == 0 && (t % kTcKb) == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            __syncthreads();
        }
        after_step(0);
        if (lane == 0) tma_store_wait_all();
    }
}

}  // namespace snnk
