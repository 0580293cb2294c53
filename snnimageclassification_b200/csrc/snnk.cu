// snnk.cu -- C-ABI entry points of libsnnk.so (see include/snnk.h for the contract).
//
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -shared
#include "../../include/snnk.h"

#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <type_traits>

#include "common.cuh"
#include "encode_head.cuh"
#include "gemm_simt.cuh"
#include "gemm_tc.cuh"
#include "gemm_bits.cuh"
#include "recur_bwd.cuh"
#include "recur_fwd.cuh"
#include "recur_gen.cuh"
#include "recur_lean.cuh"
#include "recur_nr.cuh"
#include "recur_tc.cuh"
#include "recur_wide.cuh"
#include "runs.cuh"

using namespace snnk;

namespace {

thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e, const char* where)
{
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", where, cudaGetErrorString(e));
    return SNNK_ERR_CUDA;
}

#define SNNK_CUDA(call)                                        \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call);  \
    } while (0)

// ---- optional per-kernel CUDA-event profiler (bench.py's roofline numbers; off by default) ----------------
// When enabled, every launch is bracketed by two cudaEventRecord calls on the launching stream.  Debug
// facility: process-global, not thread-safe, never touched on the normal path.
constexpr int kMaxProfiledLaunches = 1 << 14;
struct ProfiledLaunch { int id; cudaEvent_t a, b; };
bool g_prof_on = false;
int g_prof_n = 0;
ProfiledLaunch g_prof[kMaxProfiledLaunches];

struct ProfScope {
    cudaStream_t st; int slot;
    ProfScope(int id, cudaStream_t s) : st(s), slot(-1)
    {
        if (!g_prof_on || g_prof_n >= kMaxProfiledLaunches) return;
        ProfiledLaunch& L = g_prof[g_prof_n];
        if (cudaEventCreate(&L.a) != cudaSuccess || cudaEventCreate(&L.b) != cudaSuccess) return;
        L.id = id;
        slot = g_prof_n++;
        cudaEventRecord(L.a, st);
    }
    ~ProfScope() { if (slot >= 0) cudaEventRecord(g_prof[slot].b, st); }
};

// Set the kernel's dynamic shared-memory limit (when it uses any), launch it inside the profiler bracket `id` and
// check the launch.
template <class... P, class... A>
int launch(int id, void (*kern)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const A&... args)
{
    if (smem) SNNK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    { ProfScope ps(id, st); kern<<<grid, block, smem, st>>>(args...); }
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

// Fork / join onto a helper stream (one per device, created on first use) so that two independent kernels of one call
// overlap.  Event record / wait are legal during stream capture: the helper stream joins the capture and the graph
// gets two parallel branches.  The call still returns with everything ordered behind the caller's stream.  A call
// with parallel work has no serial form: it fails if the helper stream cannot be had.
struct Fork {
    cudaStream_t side = nullptr;
    cudaEvent_t forked = nullptr, joined = nullptr, mid = nullptr, forked2 = nullptr, forked3 = nullptr, joined3 = nullptr;
    bool ok = false;
};
int fork_for_device(Fork** out)
{
    static Fork forks[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess && (dev < 0 || dev >= 64)) e = cudaErrorInvalidDevice;
    if (e != cudaSuccess) return cuda_fail(e, "helper stream for the parallel branches of the call");
    Fork& f = forks[dev];
    if (!f.ok) {
        e = cudaStreamCreateWithFlags(&f.side, cudaStreamNonBlocking);
        for (cudaEvent_t* ev : {&f.forked, &f.joined, &f.mid, &f.forked2, &f.forked3, &f.joined3})
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
        if (e != cudaSuccess) return cuda_fail(e, "creating the helper stream for the parallel branches of the call");
        f.ok = true;
    }
    *out = &f;
    return SNNK_OK;
}

// Measuring switches ("0" turns a default off, anything else on), read on every call so that one process can compare
// kernel families: SNNK_LEAN (lean recurrence kernels) and SNNK_MMA_RECUR (tensor-core recurrence at any batch).
bool env_switch(const char* name, bool dflt)
{
    const char* env = getenv(name);
    return env ? env[0] != '0' : dflt;
}

// Run-time values -> template arguments.  Each selector lists every instantiation its callers are built with.
template <int V> using Int = std::integral_constant<int, V>;
template <bool V> using Bool = std::integral_constant<bool, V>;

template <class F> int by_width(int w, F&& f)   // tile width of the tensor-core GEMMs, hidden width of narrow layers
{
    switch (w) {
    case 32: return f(Int<32>{});
    case 64: return f(Int<64>{});
    default: return f(Int<128>{});
    }
}

// (layer, surrogate): mode 0 LIF, 1 ALIF, 2 Izhikevich (only the SIMT kernels have an Izhikevich body: the other
// families are passed mode 0 / 1 and read ALIF as mode == 1).  A sigma' trace (SNNK_SURROGATE_TRACE) replaces the only
// read of the ALIF threshold, so snnk_backward hands it over as mode 0 with sigma' in the V slot.
template <class F> int by_cell(int mode, int surrogate, F&& f)
{
    if (surrogate == SNNK_SURROGATE_TRACE) return mode == 2 ? f(Int<2>{}, Int<kSurrTrace>{}) : f(Int<0>{}, Int<kSurrTrace>{});
    switch (mode * 2 + (surrogate ? 1 : 0)) {
    case 0: return f(Int<0>{}, Int<0>{});
    case 1: return f(Int<0>{}, Int<1>{});
    case 2: return f(Int<1>{}, Int<0>{});
    case 3: return f(Int<1>{}, Int<1>{});
    case 4: return f(Int<2>{}, Int<0>{});
    default: return f(Int<2>{}, Int<1>{});
    }
}

template <class F> int by_rows_rec(int R, bool rec, F&& f)   // rows per CTA and recurrence of the SIMT kernels
{
    if (R == 1) return rec ? f(Int<1>{}, Bool<true>{}) : f(Int<1>{}, Bool<false>{});
    return rec ? f(Int<2>{}, Bool<true>{}) : f(Int<2>{}, Bool<false>{});
}

template <class F> int by_nsm(int nsm, F&& f)   // SMs per n-slice of the wide weight-stationary kernels
{
    switch (nsm) {
    case 4: return f(Int<4>{});
    case 2: return f(Int<2>{});
    default: return f(Int<1>{});
    }
}

int device_ok()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
    return major == 10;
}

int sm_count()
{
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 1;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) return 1;
    return n;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr int kBitsMT = 2;   // row / feature tiles per CTA of the bit-fed GEMMs (both accumulators fit TMEM)

// The kernel family of the recurrence (forward sweep and BPTT sweep), chosen from the descriptor by make_plan.
enum class Family {
    Simt,     // register-resident SIMT kernels (recur_fwd.cuh / recur_bwd.cuh; lean variants in recur_lean.cuh)
    TcRec,    // tensor-core recurrence (recur_tc.cuh)
    NonRec,   // non-recurrent layer on the lean scan kernels (recur_nr.cuh)
    WideTc,   // H > 128 on the weight-stationary tensor-core kernels (recur_wide.cuh)
    WideGen,  // H > 128 on the fp32 kernels (recur_gen.cuh)
};

// How the batch is cut into CTAs and how the weight-gradient GEMM is split; shared by the workspace
// query and the launches so they can never disagree.
struct Plan {
    Family family;
    bool lean_fwd;    // Simt: the lean forward kernel (recur_lean.cuh)
    int R;            // batch rows per recurrence CTA
    int grid_rows;    // recurrence CTAs
    int m_total;      // rows of the stacked weight gradient [dW_in ; dW_rec]
    int mtiles_x, mtiles_z, ntiles, BN;
    int S;            // split-K factor of the weight-gradient GEMM (splits are whole samples)
    int samples_per_split;
    bool tc;          // tcgen05 GEMMs eligible for this geometry (the flag asks for them and TMA can address x)
    bool check;       // tensor-core path must verify on the device that x is tf32-exact (caller did not vouch)
    bool bits;        // x is the bit-packed raster (SNNK_F_INPUT_BITS): k_proj_bits / k_wgrad_bits
    int kpad;         // K of the projection padded to the k-block
    bool wide;        // H > 128: N-tiled tensor-core GEMMs
    int w_nmt, w_nnt; // WideTc grid: m-tiles of the batch x n-slices of the hidden axis
    int w_nmt_b, w_npass_b;   // backward: m-tiles (its row tile differs) and passes over the batch
    size_t off_zx, off_wflags, off_gx, off_gmask, off_wflags_b;
    int tileN;        // N extent of one tensor-core tile
    int ntiles_tc;
    int n_pwout, n_pdb;   // number of dW_out / db partial buffers
    size_t off_gI, off_gIlo, off_pwout, off_pdb, off_pw, off_flag, bwd_bytes;
    size_t off_wplanes, off_fflag, off_weff, fwd_bytes;
    size_t off_weffT, off_gyscan;
    // frame-dedup variant (runs.cuh); eligible = tensor-core GEMMs on a non-wide layer
    bool runs;            // workspace for the compact kernels is reserved
    bool dedup;           // and the call takes a run table (x is vouched {0,1}: no tf32 check)
    int run_rows;         // rows of the compact buffers: run_cap(B*T) rounded up to whole 128-row tiles
    int S_rec, sps_rec;   // split of the dW_rec-only GEMM of the variant
    int S_cmp;            // split of the dW_in GEMM over compact rows (few 32-row blocks: a handful of splits)
    size_t off_xu_f, off_iu, off_xu_b, off_gu, gu_plane, off_pwrec;

    // The SIMT sweeps evaluate the readout and its adjoint themselves (fused head, dW_out / db partials per CTA); the
    // other families run the stand-alone head, the readout-adjoint scan (k_gy_scan) and k_wout_grad beside them.
    bool readout_in_sweep() const { return family == Family::Simt; }
};

int check_desc(const SnnkDesc* d)
{
    if (!d) return SNNK_ERR_ARG;
    if (d->B <= 0 || d->T <= 0 || d->N <= 0 || d->H <= 0 || d->O <= 0) return SNNK_ERR_SHAPE;
    if (d->layer_type != SNNK_LIF && d->layer_type != SNNK_ALIF && d->layer_type != SNNK_IZHIKEVICH) return SNNK_ERR_ARG;
    if (d->layer_type == SNNK_IZHIKEVICH && !(d->iz_C != 0.0f)) return SNNK_ERR_ARG;
    if (d->surrogate != SNNK_FAST_SIGMOID && d->surrogate != SNNK_PHI && d->surrogate != SNNK_SURROGATE_TRACE)
        return SNNK_ERR_ARG;
    if (d->O > kOMax) return SNNK_ERR_SHAPE;
    if (d->H != 32 && d->H != 64 && d->H != 128 && !(d->H % 128 == 0 && d->H <= 2048)) return SNNK_ERR_UNSUPPORTED;
    if ((long long)d->B * d->T >= (1ll << 31) / 4) return SNNK_ERR_SHAPE;
    return SNNK_OK;
}

IzhConsts izh_consts(const SnnkDesc* d)
{
    IzhConsts z{};
    z.on = d->layer_type == SNNK_IZHIKEVICH;
    z.dt = d->dt; z.C = d->iz_C; z.vr = d->iz_v_rest; z.vth = d->iz_v_th; z.k = d->iz_k; z.a = d->iz_a; z.b = d->iz_b;
    z.c = d->iz_c; z.d = d->iz_d; z.vpeak = d->iz_v_peak;
    return z;
}

// The recurrence family of a checked descriptor (H is 32, 64, 128 or a multiple of 128 up to 2048).  In tensor-core
// mode, LIF / ALIF layers take:
// - H > 128, recurrent: the weight-stationary kernels when their shared memory fits and their grid fits the chip;
// - H <= 128, not recurrent: the lean scan kernels;
// - H = 128, recurrent, O <= 15 (row 15 of the readout MMA packs the spike bits): the tensor-core recurrence from
//   B >= 1024 on.  Measured on B200 (profiles/r02_*): a step of an 8-row tile takes ~1400 (forward) / ~3000
//   (backward) cycles on one SM whatever the batch -- bound by the dependent-issue latency of its ~200 / ~580
//   instructions per warp, not by the 36 / 54 MMAs -- so these kernels win once the tiles fill the chip (B = 4096: K3
//   0.58 ms vs 0.73 ms) and lose to the one-row-per-CTA SIMT kernels, which spread a small batch over all SMs (B = 256:
//   82 / 168 us vs 55 / 72 us).  SNNK_MMA_RECUR = 0 / 1 forces the choice.
// Everything else runs the fp32 wide kernels (H > 128) or the SIMT kernels.
Family pick_family(const SnnkDesc* d, Plan& p)
{
    const bool tc_cell = d->layer_type != SNNK_IZHIKEVICH && (d->flags & SNNK_F_TENSOR_CORE) != 0;
    if (d->H > 128) {
        if (!tc_cell || !d->recurrent) return Family::WideGen;
        if (wide_fwd_smem_bytes(d->H) > 225 * 1024 || wide_bwd_smem_bytes(d->H) > 225 * 1024) return Family::WideGen;
        const int nsm = wide_nsm(d->H), mt = wide_mt(nsm), mtb = wide_bwd_mt(nsm);
        p.w_nnt = d->H / (16 * nsm);
        p.w_nmt = std::min(sm_count() / p.w_nnt, (d->B + mt - 1) / mt);
        p.w_nmt_b = std::min(sm_count() / p.w_nnt, (d->B + mtb - 1) / mtb);
        if (p.w_nmt < 1 || p.w_nmt_b < 1) return Family::WideGen;
        p.w_npass_b = (d->B + p.w_nmt_b * mtb - 1) / (p.w_nmt_b * mtb);
        return Family::WideTc;
    }
    if (!tc_cell) return Family::Simt;
    if (!d->recurrent) return Family::NonRec;
    if (d->H == kTcH && d->O <= 15 && env_switch("SNNK_MMA_RECUR", d->B >= 1024) &&
        bwd_tc_smem_bytes(d->T) <= 200 * 1024 && fwd_tc_smem_bytes(d->T) <= 200 * 1024)
        return Family::TcRec;
    return Family::Simt;
}

Plan make_plan(const SnnkDesc* d)
{
    Plan p{};
    p.wide = d->H > 128;
    p.family = pick_family(d, p);
    p.R = p.wide ? gen_rows(d->H) : (d->B > 1024 ? 2 : 1);
    // lean forward (recur_lean.cuh): recurrent LIF / ALIF, H = 128, one row per CTA, the row's input current resident
    // in shared memory; SNNK_LEAN=0 keeps the general kernel
    p.lean_fwd = p.family == Family::Simt && d->recurrent && d->layer_type != SNNK_IZHIKEVICH && d->H == 128 &&
                 p.R == 1 && d->O <= kLeanOP && lean_fwd_smem_bytes<128>(d->T, d->O) <= 110 * 1024 &&
                 env_switch("SNNK_LEAN", true);
    p.grid_rows = (d->B + p.R - 1) / p.R;
    const int BT = d->B * d->T;
    p.tileN = p.wide ? 128 : d->H;
    p.ntiles_tc = d->H / p.tileN;
    p.n_pwout = p.readout_in_sweep() ? p.grid_rows : (BT < 256 ? BT : 256);
    p.n_pdb = p.readout_in_sweep() ? p.grid_rows * p.R : p.n_pwout;
    p.BN = d->H >= 64 ? 64 : 32;
    p.ntiles = d->H / p.BN;
    p.mtiles_x = (d->N + kGemmBM - 1) / kGemmBM;
    p.mtiles_z = d->recurrent ? (d->H + kGemmBM - 1) / kGemmBM : 0;
    p.m_total = d->N + (d->recurrent ? d->H : 0);
    // TMA needs 16-byte global strides: N % 4 == 0 (H is a multiple of 32 already)
    p.tc = (d->flags & SNNK_F_TENSOR_CORE) != 0 && d->N % 4 == 0;
    p.bits = p.tc && (d->flags & SNNK_F_INPUT_BITS) != 0;
    p.check = p.tc && !p.bits && (d->flags & SNNK_F_INPUT_BINARY) == 0;
    p.kpad = (d->N + tc::kBlockK - 1) / tc::kBlockK * tc::kBlockK;
    int S;
    if (p.bits) {
        S = 148 / (((p.mtiles_x + p.mtiles_z + kBitsMT - 1) / kBitsMT) * p.ntiles_tc);   // kBitsMT feature tiles per CTA
    } else if (p.tc) {
        S = 148 / ((p.mtiles_x + p.mtiles_z) * p.ntiles_tc);   // one CTA per SM: the tcgen05 kernel owns the whole smem
    } else {
        const int tiles = (p.mtiles_x + p.mtiles_z) * p.ntiles;
        S = (4 * 148 + tiles - 1) / tiles;
    }
    if (S > d->B) S = d->B;
    if (S < 1) S = 1;
    p.samples_per_split = (d->B + S - 1) / S;
    p.S = (d->B + p.samples_per_split - 1) / p.samples_per_split;
    size_t off = 0;
    p.off_gI = off;     off = align_up(off + sizeof(float) * (size_t)BT * d->H, 256);
    p.off_gIlo = off;   off = align_up(off + (p.tc ? sizeof(float) * (size_t)BT * d->H : 0), 256);
    p.off_pwout = off;  off = align_up(off + sizeof(float) * (size_t)p.n_pwout * d->H * d->O, 256);
    p.off_pdb = off;    off = align_up(off + sizeof(float) * (size_t)p.n_pdb * d->O, 256);
    p.off_pw = off;     off = align_up(off + sizeof(float) * (size_t)p.S * p.m_total * d->H, 256);
    p.off_flag = off;   off = align_up(off + 256, 256);
    p.off_weffT = off;  off = align_up(off + sizeof(float) * (size_t)d->H * d->H, 256);
    p.off_gyscan = off; off = align_up(off + (p.readout_in_sweep() ? 0 : sizeof(float) * (size_t)BT * kOMax), 256);
    if (p.family == Family::WideTc) {
        const int nsm = wide_nsm(d->H);
        p.off_gx = off;       off = align_up(off + sizeof(float) * 2 * (size_t)p.w_nmt_b * (d->H / wide_bwd_kc(nsm)) * wide_bwd_chunk_floats(nsm), 256);
        p.off_gmask = off;    off = align_up(off + sizeof(unsigned int) * (size_t)p.w_nmt_b * p.w_npass_b * d->T, 256);
        p.off_wflags_b = off; off = align_up(off + sizeof(unsigned int) * (size_t)p.w_nmt_b * kWideFlagStride, 256);
    }
    p.runs = p.tc && !p.wide && !p.bits;
    p.dedup = p.runs && !p.check;
    if (p.runs) {
        const int cap = run_cap(BT);
        p.run_rows = (cap + 127) / 128 * 128;
        p.sps_rec = (d->B + 127) / 128;
        p.S_rec = (d->B + p.sps_rec - 1) / p.sps_rec;
        p.S_cmp = p.S < 8 ? p.S : 8;
        p.gu_plane = align_up(sizeof(float) * (size_t)p.run_rows * d->H, 256);
        p.off_xu_b = off;  off = align_up(off + sizeof(float) * (size_t)p.run_rows * d->N, 256);
        p.off_gu = off;    off = align_up(off + 2 * p.gu_plane, 256);
        p.off_pwrec = off; off = align_up(off + (d->recurrent ? sizeof(float) * (size_t)p.S_rec * d->H * d->H : 0), 256);
    }
    p.bwd_bytes = off;
    off = align_up(sizeof(float) * (size_t)BT * d->H, 256);
    p.off_wplanes = off; off = align_up(off + (p.tc ? sizeof(float) * 3 * (size_t)d->H * p.kpad : 0), 256);
    p.off_fflag = off;   off = align_up(off + 256, 256);
    p.off_weff = off;    off = align_up(off + sizeof(float) * (size_t)d->H * d->H, 256);
    if (p.family == Family::WideTc) {
        const int mt = wide_mt(wide_nsm(d->H));
        p.off_zx = off;     off = align_up(off + sizeof(uint32_t) * 2 * (size_t)p.w_nmt * (d->H / 32) * mt, 256);
        p.off_wflags = off; off = align_up(off + sizeof(unsigned int) * (size_t)p.w_nmt * kWideFlagStride, 256);
    }
    if (p.runs) {
        p.off_xu_f = off; off = align_up(off + sizeof(float) * (size_t)p.run_rows * p.kpad, 1024);   // tiled, k padded
        p.off_iu = off;   off = align_up(off + sizeof(float) * (size_t)p.run_rows * d->H, 256);
    }
    p.fwd_bytes = off;
    return p;
}

// ---- TMA tensor maps (driver entry point resolved at run time: the library does not link libcuda) ------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// fp32 tensor, innermost dimension first; strides in bytes for dims 1..rank-1; 128-byte swizzle; OOB -> 0
int make_map(CUtensorMap* m, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
             const cuuint32_t* box, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B)
{
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) { snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled unavailable"); return SNNK_ERR_CUDA; }
    const cuuint32_t ones[5] = {1, 1, 1, 1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box,
                    ones, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        snprintf(g_cuda_err, sizeof(g_cuda_err), "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
        return SNNK_ERR_CUDA;
    }
    return SNNK_OK;
}

template <int H>   // H = N extent of one CTA tile (the whole hidden width when it is <= 128)
int launch_proj_tc(const SnnkDesc* d, const Plan& pl, const float* x, float* I_in, const float* planes,
                   unsigned int* flag, cudaStream_t st, const int* run_table, int run_variant)
{
    // planes: W_in^T as split by k_split_w.  run_variant 1: x / I_in are the compact buffers of the frame-dedup path
    // (run_rows rows); 0 with a table: the dense launch, which the kernel skips when the table says ok
    constexpr int P = 2;   // planes of W_in^T fed to the tensor pipe (k_split_w writes three)
    using Cfg = tc::ProjCfg<H, P>;
    const int M = run_variant == 1 ? pl.run_rows : d->B * d->T;
    const int Hf = d->H;
    CUtensorMap mx;
    {
        const cuuint64_t dims[2] = {(cuuint64_t)d->N, (cuuint64_t)M};
        const cuuint64_t str[1] = {(cuuint64_t)d->N * 4};
        const cuuint32_t box[2] = {tc::kBlockK, tc::kBlockM};
        int rc = make_map(&mx, x, 2, dims, str, box);
        if (rc != SNNK_OK) return rc;
    }
    const float* xc = run_variant == 1 ? x : nullptr;
    return launch(SNNK_K_PROJ, tc::k_proj_tc<H, P>, dim3((M + tc::kBlockM - 1) / tc::kBlockM, Hf / H), tc::kThreads,
                  Cfg::kSmemBytes, st, mx, planes, I_in, M, pl.kpad / tc::kBlockK, Hf, flag, run_table, run_variant, xc);
}

// Geometry of one weight-gradient launch.  The dense launch contracts [x ; Z_{t-1}]^T gI over (B, T); the frame-dedup
// variant (runs.cuh) splits it into an x-only launch over compact rows (S slabs of run_Tp rows standing in for samples)
// and a Z-only launch over the dense rows with its own, finer split.
struct WgradGeom {
    const float* x; const float* Ztrace; const float* g_planes; size_t g_plane_stride;
    int T, B, N;             // extents of the (N|H, T, B) operand views
    int mtiles_x, mtiles_z, m_total, S, samples_per_split;
    float* part; unsigned int* flag; const int* run_table; int run_gate, run_clip;
};

template <int H>
int launch_wgrad_tc(const SnnkDesc* d, const WgradGeom& g, cudaStream_t st)
{
    constexpr int P = 2;
    using Cfg = tc::WgradCfg<H, P>;
    const cuuint64_t T = g.T, B = g.B, N = g.N > 0 ? g.N : 4, Hf = d->H;
    CUtensorMap mx, mz, mg;
    {
        const cuuint64_t dims[3] = {N, T, B};
        const cuuint64_t str[2] = {N * 4, T * N * 4};
        const cuuint32_t box[3] = {32, tc::kBlockK, 1};
        int rc = make_map(&mx, g.x ? g.x : g.g_planes, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
        if (rc != SNNK_OK) return rc;
    }
    {
        const cuuint64_t dims[3] = {Hf, T, B};
        const cuuint64_t str[2] = {Hf * 4, T * Hf * 4};
        const cuuint32_t box[3] = {32, tc::kBlockK, 1};
        int rc = make_map(&mz, g.Ztrace ? g.Ztrace : g.g_planes, 3, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
        if (rc != SNNK_OK) return rc;
    }
    {
        const cuuint64_t dims[4] = {Hf, T, B, (cuuint64_t)P};
        const cuuint64_t str[3] = {Hf * 4, T * Hf * 4, (cuuint64_t)g.g_plane_stride};   // planes are 256-B aligned
        const cuuint32_t box[4] = {32, tc::kBlockK, 1, 1};
        int rc = make_map(&mg, g.g_planes, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
        if (rc != SNNK_OK) return rc;
    }
    tc::WgradTcParams wp{};
    wp.N = g.N; wp.T = g.T; wp.B = g.B; wp.mtiles_x = g.mtiles_x; wp.m_total = g.m_total; wp.H_full = d->H;
    wp.samples_per_split = g.samples_per_split; wp.part = g.part; wp.inexact_flag = g.flag;
    wp.run_table = g.run_table; wp.run_gate = g.run_gate; wp.run_clip = g.run_clip;
    return launch(SNNK_K_WGRAD, tc::k_wgrad_tc<H, P>, dim3(g.mtiles_x + g.mtiles_z, g.S, d->H / H), tc::kThreads,
                  Cfg::kSmemBytes, st, mx, mz, mg, wp);
}

// ---- bit-packed input (SNNK_F_INPUT_BITS, gemm_bits.cuh) --------------------------------------------------------------
template <int H>
int launch_proj_bits(const SnnkDesc* d, const uint32_t* xbits, const float* W_in, float* I_in, void* plane_ws, cudaStream_t st)
{
    using Cfg = tc::ProjBitsCfg<H, kBitsMT>;
    const int M = d->B * d->T, Hf = d->H;
    const int kblocks = (d->N + tc::kBitsBlockK - 1) / tc::kBitsBlockK, wd = (d->N + 31) / 32;
    __half* planes = static_cast<__half*>(plane_ws);
    // the per-column scales sit behind the two planes (the region was sized for three tf32 planes: always larger)
    float* inv_scale = reinterpret_cast<float*>(planes + 2 * (size_t)kblocks * Hf * tc::kBitsBlockK);
    tc::k_split_w_h<<<Hf, 256, 0, st>>>(W_in, d->N, Hf, kblocks, planes, inv_scale);
    SNNK_CUDA(cudaGetLastError());
    return launch(SNNK_K_PROJ, tc::k_proj_bits<H, kBitsMT>,
                  dim3((M + kBitsMT * tc::kBlockM - 1) / (kBitsMT * tc::kBlockM), Hf / H), tc::bits_threads<kBitsMT>(),
                  Cfg::kSmemBytes, st, xbits, wd, planes, inv_scale, I_in, M, kblocks, Hf);
}

template <int H>
int launch_wgrad_bits(const SnnkDesc* d, const Plan& pl, const uint32_t* xbits, const uint32_t* zbits, const float* g_planes,
                      size_t g_plane_stride, float* part, cudaStream_t st)
{
    constexpr int P = 2;
    using Cfg = tc::WgradBitsCfg<H, kBitsMT>;
    const cuuint64_t T = d->T, B = d->B, Hf = d->H;
    CUtensorMap mg;
    {
        const cuuint64_t dims[4] = {Hf, T, B, (cuuint64_t)P};
        const cuuint64_t str[3] = {Hf * 4, T * Hf * 4, (cuuint64_t)g_plane_stride};
        const cuuint32_t box[4] = {32, tc::kBlockK, 1, 1};
        int rc = make_map(&mg, g_planes, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
        if (rc != SNNK_OK) return rc;
    }
    tc::WgradBitsParams wp{};
    wp.N = d->N; wp.T = d->T; wp.B = d->B; wp.mtiles_x = pl.mtiles_x; wp.mtiles_z = pl.mtiles_z; wp.m_total = pl.m_total;
    wp.H_full = d->H; wp.samples_per_split = pl.samples_per_split;
    wp.xbits = xbits; wp.wd_x = (d->N + 31) / 32; wp.zbits = zbits; wp.wd_z = d->H / 32; wp.part = part;
    return launch(SNNK_K_WGRAD, tc::k_wgrad_bits<H, kBitsMT>,
                  dim3((pl.mtiles_x + pl.mtiles_z + kBitsMT - 1) / kBitsMT, pl.S, d->H / H), tc::bits_threads<kBitsMT>(),
                  Cfg::kSmemBytes, st, mg, wp);
}

int launch_wgrad_tc_any(const SnnkDesc* d, int tileN, const WgradGeom& g, cudaStream_t st)
{
    return by_width(tileN, [&](auto tn) { return launch_wgrad_tc<decltype(tn)::value>(d, g, st); });
}

// SIMT forward recurrence (recur_fwd.cuh)
int launch_fwd_simt(const FwdParams& fp, bool rec, const Plan& pl, cudaStream_t st)
{
    return by_width(fp.H, [&](auto h) {
        return by_rows_rec(pl.R, rec, [&](auto r, auto re) {
            constexpr int H = decltype(h)::value, R = decltype(r)::value;
            constexpr bool REC = decltype(re)::value;
            const size_t smem = fwd_smem_bytes<H, R>(fp.T, fp.O);
            if (smem > 200 * 1024) return (int)SNNK_ERR_SHAPE;
            // the Izhikevich body is a compile-time variant: a run-time branch in the step loop cost the LIF/ALIF
            // kernels 6 %
            auto kern = fp.iz.on ? k_recur_fwd<H, R, REC, 2> : (fp.alif ? k_recur_fwd<H, R, REC, 1> : k_recur_fwd<H, R, REC, 0>);
            return launch(SNNK_K_RECUR_FWD, kern, pl.grid_rows, H, smem, st, fp);
        });
    });
}

// Lean forward recurrence (recur_lean.cuh; Plan::lean_fwd).  pdl: launch as a programmatic dependent of the kernel
// queued before it on the stream (the projection GEMM, which executes griddepcontrol.launch_dependents at its start):
// the recurrence kernel's prologue then overlaps the projection.
int launch_fwd_lean(FwdParams fp, cudaStream_t st, bool pdl)
{
    const size_t smem = lean_fwd_smem_bytes<128>(fp.T, fp.O);
    void (*kern)(const FwdParams) = fp.alif ? (fp.traces ? k_recur_fwd_lean<128, true, true> : k_recur_fwd_lean<128, true, false>)
                                            : (fp.traces ? k_recur_fwd_lean<128, false, true> : k_recur_fwd_lean<128, false, false>);
    SNNK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fp.pdl = pdl ? 1 : 0;
    {
        ProfScope ps(SNNK_K_RECUR_FWD, st);
        if (pdl) {
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3(fp.B); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = smem; cfg.stream = st;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            SNNK_CUDA(cudaLaunchKernelEx(&cfg, kern, (const FwdParams)fp));
        } else {
            kern<<<fp.B, 128, smem, st>>>(fp);
        }
    }
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

// Lean BPTT sweep (recur_lean.cuh): the training step of the headline geometry -- recurrent LIF / ALIF, H = 128, one row
// per CTA, sparse seeds from the fused head, no seeds on V / Z.  A refinement of the SIMT family that also depends on
// the seeds of the call; SNNK_LEAN=0 keeps the general kernel.
bool use_lean_bwd(const BwdParams& bp, bool rec, int R)
{
    if (!rec || bp.iz.on || bp.H != 128 || R != 1 || bp.g_y || bp.g_V || bp.g_Z || !bp.g_logits || !bp.tstar) return false;
    if (bwd_smem_bytes<128, 1>(bp.T, true) > 110 * 1024 || bp.T > 128) return false;   // T * 4 spike words <= 4 per thread
    return env_switch("SNNK_LEAN", true);
}

int launch_bwd_lean(const BwdParams& bp, cudaStream_t st)
{
    const size_t smem = bwd_smem_bytes<128, 1>(bp.T, true);
    const bool planes = bp.gI_lo != nullptr, runs = bp.run_table != nullptr;
    return by_cell(bp.alif ? 1 : 0, bp.surrogate, [&](auto m, auto s) -> int {
        constexpr bool A = decltype(m)::value == 1;
        constexpr int S = decltype(s)::value;
        auto pick = [&](auto op) {
            constexpr int OP = decltype(op)::value;
            return planes ? (runs ? k_recur_bwd_lean<A, S, true, true, OP> : k_recur_bwd_lean<A, S, true, false, OP>)
                          : (runs ? k_recur_bwd_lean<A, S, false, true, OP> : k_recur_bwd_lean<A, S, false, false, OP>);
        };
        return launch(SNNK_K_RECUR_BWD, bp.O <= 12 ? pick(Int<12>{}) : pick(Int<16>{}), bp.B, 128, smem, st, bp);
    });
}

// SIMT BPTT sweep (recur_bwd.cuh)
int launch_bwd_simt(const BwdParams& bp, bool rec, const Plan& pl, cudaStream_t st)
{
    const int mode = bp.iz.on ? 2 : (bp.alif ? 1 : 0);
    return by_width(bp.H, [&](auto h) -> int {
        return by_rows_rec(pl.R, rec, [&](auto r, auto re) -> int {
            constexpr int H = decltype(h)::value, R = decltype(r)::value;
            constexpr bool REC = decltype(re)::value;
            const size_t smem = bwd_smem_bytes<H, R>(bp.T, REC);
            if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
            return by_cell(mode, bp.surrogate, [&](auto m, auto s) -> int {
                return launch(SNNK_K_RECUR_BWD, k_recur_bwd<H, R, REC, decltype(m)::value, decltype(s)::value>,
                              pl.grid_rows, H, smem, st, bp);
            });
        });
    });
}

WideParams wide_params(const FwdParams& fp, const Plan& pl, char* ws)
{
    WideParams wp{};
    wp.B = fp.B; wp.T = fp.T; wp.H = fp.H; wp.O = fp.O; wp.alif = fp.alif; wp.traces = fp.traces;
    wp.alpha = fp.alpha; wp.rho = fp.rho; wp.theta = fp.theta;
    wp.I_in = fp.I_in; wp.W = fp.W_eff; wp.beta = fp.beta; wp.V0 = fp.V0; wp.a0 = fp.a0; wp.Z0 = fp.Z0;
    wp.V = fp.V; wp.a = fp.a; wp.Z = fp.Z; wp.zbits = fp.zbits;
    wp.zx = reinterpret_cast<uint32_t*>(ws + pl.off_zx);
    wp.flags = reinterpret_cast<unsigned int*>(ws + pl.off_wflags);
    wp.n_mt = pl.w_nmt; wp.n_nt = pl.w_nnt;
    return wp;
}

// Wide layers (H > 128) in tensor-core mode: weight-stationary, grid-synchronous kernels (recur_wide.cuh).  Cooperative
// launches: every CTA waits for its m-tile's peers each step, so all of them must be resident.
int launch_wide_fwd(const WideParams& wp, cudaStream_t st)
{
    return by_nsm(wide_nsm(wp.H), [&](auto nsm) -> int {
        constexpr int NSM = decltype(nsm)::value;
        const size_t smem = wide_fwd_smem_bytes(wp.H);
        void* kern = wp.alif ? (void*)k_wide_fwd<NSM, true> : (void*)k_wide_fwd<NSM, false>;
        SNNK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SNNK_CUDA(cudaMemsetAsync(wp.flags, 0, sizeof(unsigned int) * (size_t)wp.n_mt * kWideFlagStride, st));
        WideParams arg = wp;
        void* args[] = {&arg};
        ProfScope ps(SNNK_K_RECUR_FWD, st);
        SNNK_CUDA(cudaLaunchCooperativeKernel(kern, dim3(wp.n_mt * wp.n_nt), dim3(kWideThreads), args, smem, st));
        return SNNK_OK;
    });
}

int launch_wide_bwd(const WideBwdParams& wp, int n_pass, cudaStream_t st)
{
    return by_nsm(wide_nsm(wp.H), [&](auto nsm) -> int {
        return by_cell(wp.alif ? 1 : 0, wp.surrogate, [&](auto m, auto s) -> int {
            const size_t smem = wide_bwd_smem_bytes(wp.H);
            void* kern = (void*)k_wide_bwd<decltype(nsm)::value, decltype(m)::value == 1, decltype(s)::value>;
            SNNK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            SNNK_CUDA(cudaMemsetAsync(wp.flags, 0, sizeof(unsigned int) * (size_t)wp.n_mt * kWideFlagStride, st));
            SNNK_CUDA(cudaMemsetAsync(wp.gmask, 0, sizeof(unsigned int) * (size_t)wp.n_mt * n_pass * wp.T, st));
            WideBwdParams arg = wp;
            void* args[] = {&arg};
            ProfScope ps(SNNK_K_RECUR_BWD, st);
            SNNK_CUDA(cudaLaunchCooperativeKernel(kern, dim3(wp.n_mt * wp.n_nt), dim3(kWideThreads), args, smem, st));
            return SNNK_OK;
        });
    });
}

// Non-recurrent LIF / ALIF layers of width 32 / 64 / 128 in tensor-core mode: lean scan kernels (recur_nr.cuh).
int launch_nonrec_fwd(const FwdParams& fp, cudaStream_t st)
{
    return by_width(fp.H, [&](auto h) -> int {
        constexpr int H = decltype(h)::value;
        const size_t smem = nonrec_fwd_smem_bytes<H>(fp.T, fp.O);
        if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
        return launch(SNNK_K_RECUR_FWD, fp.alif ? k_nonrec_fwd<H, true> : k_nonrec_fwd<H, false>, fp.B, H, smem, st, fp);
    });
}

int launch_nonrec_bwd(const BwdParams& bp, const float* gy_scan, cudaStream_t st)
{
    return by_width(bp.H, [&](auto h) -> int {
        constexpr int H = decltype(h)::value;
        const size_t smem = nonrec_bwd_smem_bytes<H>(bp.T);
        if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
        return by_cell(bp.alif ? 1 : 0, bp.surrogate, [&](auto m, auto s) -> int {
            return launch(SNNK_K_RECUR_BWD, k_nonrec_bwd<H, decltype(m)::value == 1, decltype(s)::value>, bp.B, H, smem, st,
                          bp, gy_scan);
        });
    });
}

// 4-D view {32, B, 4, T} of a (B, T, 128) fp32 trace (H = 4 groups of 32 neurons) with the box {32, rows, 4, steps} the
// tensor-core recurrence kernels move per TMA operation (recur_tc.cuh); 128-byte swizzle
int make_trace_map(CUtensorMap* m, const float* base, int B, int T, int rows, int steps)
{
    const cuuint64_t dims[4] = {32, (cuuint64_t)B, 4, (cuuint64_t)T};
    const cuuint64_t str[3] = {(cuuint64_t)T * kTcH * 4, 128, (cuuint64_t)kTcH * 4};
    const cuuint32_t box[4] = {32, (cuuint32_t)rows, 4, (cuuint32_t)steps};
    return make_map(m, base, 4, dims, str, box);
}

// Tensor-core recurrence (recur_tc.cuh): H = 128 recurrent LIF / ALIF layers in tensor-core mode.
int launch_fwd_tc(const FwdParams& fp, cudaStream_t st)
{
    const size_t smem = fwd_tc_smem_bytes(fp.T);
    if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
    const int grid = (fp.B + kTcRows - 1) / kTcRows;
    CUtensorMap mV{}, mA{}, mZ{};
    if (fp.traces) {
        int rc = make_trace_map(&mV, fp.V, fp.B, fp.T, kTcRows, kTcK);
        if (rc == SNNK_OK) rc = make_trace_map(&mZ, fp.Z, fp.B, fp.T, kTcRows, kTcK);
        if (rc == SNNK_OK && fp.alif) rc = make_trace_map(&mA, fp.a, fp.B, fp.T, kTcRows, kTcK);
        if (rc != SNNK_OK) return rc;
    }
    return launch(SNNK_K_RECUR_FWD, fp.alif ? k_recur_fwd_tc<true> : k_recur_fwd_tc<false>, grid, kTcFwdThreads, smem, st,
                  fp, mV, fp.alif ? mA : mV, mZ);
}

int launch_bwd_tc(const BwdParams& bp, const float* gy_scan, cudaStream_t st)
{
    const size_t smem = bwd_tc_smem_bytes(bp.T);
    if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
    const int grid = (bp.B + kTcRows - 1) / kTcRows;
    CUtensorMap mV{}, mA{}, mG{}, mGlo{};
    {
        int rc = make_trace_map(&mV, bp.V, bp.B, bp.T, kTcRows, kTcK);
        if (rc == SNNK_OK && bp.alif) rc = make_trace_map(&mA, bp.a, bp.B, bp.T, kTcRows, kTcK);
        if (rc == SNNK_OK) rc = make_trace_map(&mG, bp.gI, bp.B, bp.T, kTcRows, kTcKb);
        if (rc == SNNK_OK && bp.gI_lo) rc = make_trace_map(&mGlo, bp.gI_lo, bp.B, bp.T, kTcRows, kTcKb);
        if (rc != SNNK_OK) return rc;
    }
    return by_cell(bp.alif ? 1 : 0, bp.surrogate, [&](auto m, auto s) -> int {
        return launch(SNNK_K_RECUR_BWD, k_recur_bwd_tc<decltype(m)::value == 1, decltype(s)::value>, grid, kTcThreads, smem,
                      st, bp, gy_scan, mV, bp.alif ? mA : mV, mG, bp.gI_lo ? mGlo : mG);
    });
}

// Readout-adjoint scan of the families whose sweep does not evaluate the readout (Plan::readout_in_sweep), and the
// dW_out / db partials contracted from it and the spike raster
int launch_gy_scan(const SnnkDesc* d, const BwdParams& bp, float* gy_scan, cudaStream_t st)
{
    return launch(SNNK_K_REDUCE_OUT, k_gy_scan, (d->B * kOMax + 255) / 256, 256, 0, st, d->B, d->T, d->O, d->kappa, bp.g_y,
                  bp.g_logits, bp.tstar, bp.g_scale, gy_scan);
}

int launch_wout_grad(const SnnkDesc* d, const Plan& pl, const uint32_t* zbits, const float* gy_scan, float* pwout,
                     float* pdb, cudaStream_t st)
{
    return launch(SNNK_K_REDUCE_OUT, k_wout_grad, dim3(pl.n_pwout, (d->H + 127) / 128), 128, 0, st, d->B * d->T, d->H,
                  d->O, zbits, gy_scan, pwout, pdb);
}

// ---- wide hidden layers (H > 128) on the fp32 kernels (recur_gen.cuh): generic recurrence, then the readout --------
int launch_readout_scan(const SnnkDesc* d, const FwdParams& fp, cudaStream_t st)
{
    const size_t smem = sizeof(uint32_t) * (size_t)d->T * (d->H / 32) + sizeof(float) * ((size_t)d->H * d->O + (size_t)d->T * d->O);
    if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
    return launch(SNNK_K_HEAD, k_readout_scan, d->B, 128, smem, st, d->T, d->H, d->O, d->kappa, fp.zbits, fp.W_out, fp.b_out,
                  fp.y, fp.logits, fp.tstar);
}

int launch_fwd_gen(const SnnkDesc* d, const FwdParams& fp, bool rec, const Plan& pl, cudaStream_t st)
{
    auto go = [&](auto npt, auto r) -> int {
        constexpr int NPT = decltype(npt)::value, R = decltype(r)::value;
        const size_t smem = sizeof(float) * 2 * (size_t)d->H * R;
        return launch(SNNK_K_RECUR_FWD, rec ? k_recur_fwd_gen<NPT, R, true> : k_recur_fwd_gen<NPT, R, false>, pl.grid_rows,
                      d->H / NPT, smem, st, fp);
    };
    return gen_npt(d->H) == 1 ? go(Int<1>{}, Int<4>{}) : go(Int<2>{}, Int<2>{});
}

// writes the readout-adjoint scan itself
int launch_bwd_gen(const SnnkDesc* d, const BwdParams& bp, bool rec, const Plan& pl, float* gy_scan, cudaStream_t st)
{
    auto go = [&](auto npt, auto r) -> int {
        constexpr int NPT = decltype(npt)::value, R = decltype(r)::value;
        const size_t smem = sizeof(float) * (2 * (size_t)d->H * R + (size_t)R * d->T * kOMax);
        if (smem > 200 * 1024) return SNNK_ERR_SHAPE;
        auto kern = bp.surrogate == SNNK_SURROGATE_TRACE
                        ? (rec ? k_recur_bwd_gen<NPT, R, true, true> : k_recur_bwd_gen<NPT, R, false, true>)
                        : (rec ? k_recur_bwd_gen<NPT, R, true> : k_recur_bwd_gen<NPT, R, false>);
        return launch(SNNK_K_RECUR_BWD, kern, pl.grid_rows, d->H / NPT, smem, st, bp, gy_scan);
    };
    return gen_npt(d->H) == 1 ? go(Int<1>{}, Int<4>{}) : go(Int<2>{}, Int<2>{});
}

// pass 0: raster (+ change flags when chg != null)          k_encode
// pass 1: change flags only                                  k_encode_flags   } lazy raster of snnk_encode_runs
// pass 2: the rows the consumers of run_table will read      k_encode_rows    }
template <typename TIn>
int launch_encode(const TIn* x, int64_t n_items, int64_t n_pix, int32_t n_steps, double t_max, double tau,
                  double thr, double eps, int32_t periodic, void* out, int32_t out_dtype, int64_t* periods,
                  unsigned char* chg, cudaStream_t st, int pass = 0, const int* run_table = nullptr)
{
    dim3 grid((unsigned)n_items, (unsigned)((n_pix + 255) / 256));
    long long* per = reinterpret_cast<long long*>(periods);
    if (chg && pass != 2) SNNK_CUDA(cudaMemsetAsync(chg, 0, (size_t)n_items * n_steps, st));
    ProfScope ps(SNNK_K_ENCODE, st);
    if (pass == 1) {
        k_encode_flags<TIn><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic, chg);
        SNNK_CUDA(cudaGetLastError());
        return SNNK_OK;
    }
    if (out_dtype == SNNK_BITS) {
        if (pass != 0 || chg) return SNNK_ERR_ARG;      // the packed raster has no run-table / lazy form
        k_encode_bits<TIn><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                static_cast<uint32_t*>(out));
        SNNK_CUDA(cudaGetLastError());
        return SNNK_OK;
    }
    switch (out_dtype) {
    case SNNK_F32:
        if (pass == 2) k_encode_rows<TIn, float><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                                      static_cast<float*>(out), run_table);
        else k_encode<TIn, float><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                       static_cast<float*>(out), per, chg);
        break;
    case SNNK_F64:
        if (pass == 2) k_encode_rows<TIn, double><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                                       static_cast<double*>(out), run_table);
        else k_encode<TIn, double><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                        static_cast<double*>(out), per, chg);
        break;
    case SNNK_U8:
        if (pass == 2) k_encode_rows<TIn, uint8_t><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                                        static_cast<uint8_t*>(out), run_table);
        else k_encode<TIn, uint8_t><<<grid, 256, 0, st>>>(x, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic,
                                                         static_cast<uint8_t*>(out), per, chg);
        break;
    default:
        return SNNK_ERR_ARG;
    }
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

}  // namespace

extern "C" {

int snnk_abi_version(void) { return SNNK_ABI_VERSION; }

const char* snnk_strerror(int code)
{
    switch (code) {
    case SNNK_OK: return "ok";
    case SNNK_ERR_ARG: return "invalid argument (null pointer, bad enum or flag)";
    case SNNK_ERR_SHAPE: return "geometry outside what the kernels support";
    case SNNK_ERR_DEVICE: return "current CUDA device is not sm_100 (B200); there is no fallback path";
    case SNNK_ERR_WORKSPACE: return "workspace too small";
    case SNNK_ERR_CUDA: return "CUDA runtime error (see snnk_last_cuda_error)";
    case SNNK_ERR_UNSUPPORTED: return "request not implemented by the B200 path";
    default: return "unknown snnk error code";
    }
}

const char* snnk_last_cuda_error(void) { return g_cuda_err; }

int snnk_device_supported(void) { return device_ok(); }

const char* snnk_kernel_name(int id)
{
    switch (id) {
    case SNNK_K_ENCODE: return "K5 k_encode (to_spikes)";
    case SNNK_K_PROJ: return "K1 k_proj (input projection GEMM)";
    case SNNK_K_RECUR_FWD: return "K2 k_recur_fwd (fused recurrence + readout)";
    case SNNK_K_HEAD: return "K6 k_head_nll";
    case SNNK_K_RECUR_BWD: return "K3 k_recur_bwd (fused reverse-time BPTT)";
    case SNNK_K_REDUCE_OUT: return "k_wout_grad (wide layers: dW_out, db partials)";
    case SNNK_K_WGRAD: return "K4 k_wgrad (weight-gradient GEMM)";
    case SNNK_K_PROJ_FALLBACK: return "K1f k_proj_simt (gated fallback)";
    case SNNK_K_WGRAD_FALLBACK: return "K4f k_wgrad_simt (gated fallback)";
    case SNNK_K_INPUT_GRAD: return "k_input_grad (stacked layers: dL/dx)";
    case SNNK_K_ADAM: return "k_adam_step (optimizer)";
    case SNNK_K_REDUCE_W: return "k_finalize_grads (all partial reductions)";
    default: return "?";
    }
}

int snnk_profile_begin(void)
{
    if (g_prof_on) return SNNK_ERR_ARG;
    g_prof_n = 0;
    g_prof_on = true;
    return SNNK_OK;
}

int snnk_profile_end(double* ms_total, int64_t* launches)
{
    if (!g_prof_on || !ms_total || !launches) return SNNK_ERR_ARG;
    g_prof_on = false;
    for (int k = 0; k < SNNK_K_COUNT; ++k) { ms_total[k] = 0.0; launches[k] = 0; }
    SNNK_CUDA(cudaDeviceSynchronize());
    for (int q = 0; q < g_prof_n; ++q) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, g_prof[q].a, g_prof[q].b) == cudaSuccess) {
            ms_total[g_prof[q].id] += ms;
            launches[g_prof[q].id] += 1;
        }
        cudaEventDestroy(g_prof[q].a);
        cudaEventDestroy(g_prof[q].b);
    }
    g_prof_n = 0;
    return SNNK_OK;
}

static int encode_any(const void* x, int32_t x_dtype, int64_t n_items, int64_t n_pix, int32_t n_steps, double t_max,
                      double tau, double thr, double eps, int32_t periodic, void* out, int32_t out_dtype,
                      int64_t* periods, unsigned char* chg, cudaStream_t st, int pass = 0, const int* run_table = nullptr)
{
    if (x_dtype == SNNK_F32)
        return launch_encode(static_cast<const float*>(x), n_items, n_pix, n_steps, t_max, tau, thr, eps,
                             periodic, out, out_dtype, periods, chg, st, pass, run_table);
    if (x_dtype == SNNK_F64)
        return launch_encode(static_cast<const double*>(x), n_items, n_pix, n_steps, t_max, tau, thr, eps,
                             periodic, out, out_dtype, periods, chg, st, pass, run_table);
    if (x_dtype == SNNK_I64)
        return launch_encode(static_cast<const long long*>(x), n_items, n_pix, n_steps, t_max, tau, thr, eps,
                             periodic, out, out_dtype, periods, chg, st, pass, run_table);
    return SNNK_ERR_ARG;
}

int snnk_encode(const void* x, int32_t x_dtype, int64_t n_items, int64_t n_pix, int32_t n_steps, double t_max,
                double tau, double thr, double eps, int32_t periodic, void* out, int32_t out_dtype,
                int64_t* periods, snnk_stream_t stream)
{
    if (n_items < 0 || n_pix < 0 || n_steps <= 0 || n_items > 0x7fffffffll || n_pix > 65535ll * 256) return SNNK_ERR_SHAPE;
    if (n_items == 0 || n_pix == 0) return SNNK_OK;   /* empty batch: nothing to do (pointers may be NULL) */
    if (!x || !out) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    return encode_any(x, x_dtype, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic, out, out_dtype, periods,
                      nullptr, static_cast<cudaStream_t>(stream));
}

int snnk_unpack_raster(const uint32_t* bits, int64_t n_rows, int32_t n_pix, float* out, snnk_stream_t stream)
{
    if (n_rows < 0 || n_pix <= 0) return SNNK_ERR_SHAPE;
    if (n_rows == 0) return SNNK_OK;
    if (!bits || !out) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    const long long total = n_rows * (long long)n_pix;
    const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 32ll * sm_count());
    return launch(SNNK_K_ENCODE, k_unpack_raster, grid, 256, 0, static_cast<cudaStream_t>(stream), bits, n_rows, n_pix, out);
}

size_t snnk_run_table_bytes(int64_t n_items, int32_t n_steps)
{
    if (n_items <= 0 || n_steps <= 0 || n_items * n_steps >= (1ll << 31) / 4) return 0;
    return sizeof(int32_t) * run_table_ints(n_items, n_steps);
}

// Run table followed by the compact rows, tiled for the projection kernel (k_gather_rows_tiled's output)
static size_t run_table_tiled_offset(int64_t n_items, int32_t n_steps)
{
    return align_up(sizeof(int32_t) * run_table_ints(n_items, n_steps), 1024);
}

size_t snnk_run_table_tiled_bytes(int64_t n_items, int32_t n_steps, int32_t n_pix)
{
    if (snnk_run_table_bytes(n_items, n_steps) == 0 || n_pix <= 0 || n_pix % 4 != 0) return 0;
    const size_t rows = ((size_t)run_cap(n_items * n_steps) + 127) / 128 * 128;
    const size_t kpad = ((size_t)n_pix + tc::kBlockK - 1) / tc::kBlockK * tc::kBlockK;
    return run_table_tiled_offset(n_items, n_steps) + sizeof(float) * rows * kpad;
}

int snnk_frame_runs(int64_t n_items, int32_t n_steps, const uint8_t* frame_changed, int32_t* run_table,
                    snnk_stream_t stream)
{
    if (n_items <= 0 || n_steps <= 0 || n_items * n_steps >= (1ll << 31) / 4) return SNNK_ERR_SHAPE;
    if (!frame_changed || !run_table) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_steps <= 128) {   // warp per sample, two launches spread over the chip (runs.cuh)
        int* counts = run_table + kRunHdr + n_items * n_steps + 2 * (int64_t)run_cap(n_items * n_steps);
        const unsigned grid = (unsigned)((n_items + 7) / 8);
        k_frame_counts<<<grid, 256, 0, st>>>((int)n_items, n_steps, frame_changed, counts);
        k_frame_fill<<<grid, 256, 0, st>>>((int)n_items, n_steps, frame_changed, counts, run_table);
    } else {
        k_frame_runs<<<1, 1024, 0, st>>>((int)n_items, n_steps, frame_changed, run_table);
    }
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

// The first row of every run, tiled and swizzled for the compact projection, behind the table (lazy & 2): the gather
// that snnk_forward would otherwise run at the head of every step is done once, where the raster is made.
static int tile_compact_rows(const void* out, int32_t out_dtype, int64_t n_items, int64_t n_pix, int32_t n_steps,
                             int32_t* run_table, cudaStream_t st)
{
    if (out_dtype != SNNK_F32 || snnk_run_table_tiled_bytes(n_items, n_steps, (int32_t)n_pix) == 0) return SNNK_ERR_ARG;
    const int BT = (int)(n_items * n_steps);
    const int rows = (run_cap(BT) + 127) / 128 * 128;
    const int kpad = ((int)n_pix + tc::kBlockK - 1) / tc::kBlockK * tc::kBlockK;
    float* Xu = reinterpret_cast<float*>(reinterpret_cast<char*>(run_table) + run_table_tiled_offset(n_items, n_steps));
    k_gather_rows_tiled<<<std::min(rows, 8 * sm_count()), 256, 0, st>>>(static_cast<const float*>(out), run_table, BT,
                                                                      (int)n_pix, kpad, Xu);
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

int snnk_encode_runs(const void* x, int32_t x_dtype, int64_t n_items, int64_t n_pix, int32_t n_steps, double t_max,
                     double tau, double thr, double eps, int32_t periodic, void* out, int32_t out_dtype,
                     int64_t* periods, uint8_t* frame_changed, int32_t* run_table, int32_t lazy, snnk_stream_t stream)
{
    if (n_items <= 0 || n_pix <= 0 || n_steps <= 0 || n_items > 0x7fffffffll || n_pix > 65535ll * 256) return SNNK_ERR_SHAPE;
    if (n_items * n_steps >= (1ll << 31) / 4) return SNNK_ERR_SHAPE;
    if (!x || !out || !frame_changed || !run_table) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!(lazy & 1)) {
        int rc = encode_any(x, x_dtype, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic, out, out_dtype, periods,
                            frame_changed, st);
        if (rc != SNNK_OK) return rc;
        rc = snnk_frame_runs(n_items, n_steps, frame_changed, run_table, stream);
        if (rc != SNNK_OK) return rc;
        return (lazy & 2) ? tile_compact_rows(out, out_dtype, n_items, n_pix, n_steps, run_table, st) : SNNK_OK;
    }
    // lazy raster: flags -> run table -> only the rows the consumers of the table will read (all of them if not ok)
    int rc = encode_any(x, x_dtype, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic, out, out_dtype, periods,
                        frame_changed, st, 1, nullptr);
    if (rc != SNNK_OK) return rc;
    rc = snnk_frame_runs(n_items, n_steps, frame_changed, run_table, stream);
    if (rc != SNNK_OK) return rc;
    rc = encode_any(x, x_dtype, n_items, n_pix, n_steps, t_max, tau, thr, eps, periodic, out, out_dtype, nullptr,
                    frame_changed, st, 2, run_table);
    if (rc != SNNK_OK) return rc;
    return (lazy & 2) ? tile_compact_rows(out, out_dtype, n_items, n_pix, n_steps, run_table, st) : SNNK_OK;
}

int snnk_spike_forward(const float* v, const float* thr, int64_t n, int64_t thr_n, float* out,
                       snnk_stream_t stream)
{
    if (!v || !thr || !out) return SNNK_ERR_ARG;
    if (n < 0 || (thr_n != 1 && thr_n != n)) return SNNK_ERR_SHAPE;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    if (n == 0) return SNNK_OK;
    k_spike_fwd<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(v, thr, n, thr_n, out);
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

int snnk_spike_backward(int32_t surrogate, const float* v, const float* thr, const float* gamma,
                        const float* g_out, int64_t n, int64_t thr_n, float* g_in, snnk_stream_t stream)
{
    if (!v || !thr || !gamma || !g_out || !g_in) return SNNK_ERR_ARG;
    if (surrogate != SNNK_FAST_SIGMOID && surrogate != SNNK_PHI) return SNNK_ERR_ARG;
    if (n < 0 || (thr_n != 1 && thr_n != n)) return SNNK_ERR_SHAPE;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    if (n == 0) return SNNK_OK;
    k_spike_bwd<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        surrogate, v, thr, gamma, g_out, n, thr_n, g_in);
    SNNK_CUDA(cudaGetLastError());
    return SNNK_OK;
}

size_t snnk_forward_workspace_bytes(const SnnkDesc* d)
{
    if (check_desc(d) != SNNK_OK) return 0;
    return make_plan(d).fwd_bytes;
}

size_t snnk_backward_workspace_bytes(const SnnkDesc* d)
{
    if (check_desc(d) != SNNK_OK) return 0;
    return make_plan(d).bwd_bytes;
}

// Head arguments of snnk_forward_nll (null for snnk_forward)
struct HeadArgs {
    const int64_t* labels; float* logp; float* loss; float* g_logits; void* head_ws; uint64_t* mailbox; uint32_t* counter;
};

static int forward_impl(const SnnkDesc* d, const float* x, const float* W_in, const float* W_rec, const float* rec_mask,
                 const float* beta, const float* W_out, const float* b_out, const float* V0, const float* a0,
                 const float* Z0, float* V, float* a, float* Z, uint32_t* zbits, float* y, float* logits,
                 int32_t* tstar, void* workspace, size_t workspace_bytes, const int32_t* run_table, float* W_effT_out,
                 snnk_stream_t stream, const HeadArgs* head)
{
    int rc = check_desc(d);
    if (rc != SNNK_OK) return rc;
    if (!x || !W_in || !W_out || !b_out || !zbits || !y || !logits || !tstar || !workspace) return SNNK_ERR_ARG;
    if (d->recurrent && !W_rec) return SNNK_ERR_ARG;
    if (d->layer_type == SNNK_ALIF && !beta) return SNNK_ERR_ARG;
    const bool traces = (d->flags & SNNK_F_TRACES) != 0;
    if (traces && (!V || !Z || (d->layer_type != SNNK_LIF && !a))) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    const Plan pl = make_plan(d);
    if (workspace_bytes < pl.fwd_bytes) return SNNK_ERR_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(workspace);
    float* I_in = static_cast<float*>(workspace);
    // frame-dedup variant (runs.cuh): only for inputs the caller vouches to be the encoder's {0,1} raster
    const int* runs = pl.dedup ? run_table : nullptr;

    // K1: input projection for all T steps at once.  Tensor-core path first (when asked for and addressable by
    // TMA); the fp32 SIMT kernel behind it only runs if x turned out not to be tf32-exact (device-side flag).
    const int M = d->B * d->T;
    unsigned int* flag = nullptr;
    float* compact_rows = nullptr;
    // With a run table the weight planes, the dense launch (which skips itself when the table says ok) and the
    // preparation of the recurrent matrix go onto a parallel branch beside gather + compact projection; joined before K2.
    Fork* fk = nullptr;
    cudaStream_t side = st;
    if ((d->flags & SNNK_F_INPUT_BITS) && !pl.bits) return SNNK_ERR_UNSUPPORTED;
    if (pl.bits) {
        // bit-packed raster: the words are expanded inside the GEMM's shared-memory tiles (gemm_bits.cuh)
        const uint32_t* xb = reinterpret_cast<const uint32_t*>(x);
        rc = by_width(pl.tileN, [&](auto tn) {
            return launch_proj_bits<decltype(tn)::value>(d, xb, W_in, I_in, ws + pl.off_wplanes, st);
        });
        if (rc != SNNK_OK) return rc;
    } else if (pl.tc) {
        float* planes = reinterpret_cast<float*>(ws + pl.off_wplanes);
        if (pl.check) {
            flag = reinterpret_cast<unsigned int*>(ws + pl.off_fflag);
            SNNK_CUDA(cudaMemsetAsync(flag, 0, sizeof(unsigned int), st));
        }
        if (runs) {   // side: weight planes -> [mid] -> dense launch, k_prep_rec;  main: gather -> wait mid -> compact GEMM
            rc = fork_for_device(&fk);
            if (rc != SNNK_OK) return rc;
            side = fk->side;
            SNNK_CUDA(cudaEventRecord(fk->forked, st));
            SNNK_CUDA(cudaStreamWaitEvent(side, fk->forked, 0));
        }
        const int n = d->H * pl.kpad;
        tc::k_split_w<<<(n + 255) / 256, 256, 0, side>>>(W_in, d->N, d->H, pl.kpad, planes);
        SNNK_CUDA(cudaGetLastError());
        if (fk) SNNK_CUDA(cudaEventRecord(fk->mid, side));
        rc = by_width(pl.tileN, [&](auto tn) {
            return launch_proj_tc<decltype(tn)::value>(d, pl, x, I_in, planes, flag, side, runs, 0);
        });
        if (rc != SNNK_OK) return rc;
        if (runs) {
            float* Xu = reinterpret_cast<float*>(ws + pl.off_xu_f);
            compact_rows = reinterpret_cast<float*>(ws + pl.off_iu);
            if (d->flags & SNNK_F_RUNS_TILED) {
                // the encoder left the tiled compact rows behind the table (snnk_encode_runs, lazy & 2)
                Xu = reinterpret_cast<float*>(reinterpret_cast<char*>(const_cast<int32_t*>(runs)) +
                                              run_table_tiled_offset(d->B, d->T));
            } else {
                rc = launch(SNNK_K_PROJ, k_gather_rows_tiled, std::min(pl.run_rows, 8 * sm_count()), 256, 0, st, x, runs, M,
                            d->N, pl.kpad, Xu);
                if (rc != SNNK_OK) return rc;
            }
            // few compact tiles: 32-column CTA tiles spread each over H/32 SMs (the tile time is bound by what one
            // SM can pull in, two thirds of which are weight planes)
            SNNK_CUDA(cudaStreamWaitEvent(st, fk->mid, 0));
            rc = launch_proj_tc<32>(d, pl, Xu, compact_rows, planes, nullptr, st, runs, 1);
            if (rc != SNNK_OK) return rc;
        }
    }
    if (!pl.bits && (!pl.tc || pl.check)) {
        rc = launch(pl.tc ? SNNK_K_PROJ_FALLBACK : SNNK_K_PROJ, pl.BN == 64 ? k_proj_simt<64> : k_proj_simt<32>,
                    dim3((M + kGemmBM - 1) / kGemmBM, pl.ntiles), kGemmThreads, 0, st, x, W_in, I_in, M, d->N, d->H, flag);
        if (rc != SNNK_OK) return rc;
    }
    // K2: fused recurrence + readout
    float* W_eff = nullptr;
    if (d->recurrent) {
        W_eff = reinterpret_cast<float*>(ws + pl.off_weff);
        const int n = d->H * d->H;
        k_prep_rec<<<(n + 255) / 256, 256, 0, side>>>(W_rec, rec_mask, d->H, W_eff, W_effT_out);
        SNNK_CUDA(cudaGetLastError());
    }
    if (fk) {
        SNNK_CUDA(cudaEventRecord(fk->joined, side));
        SNNK_CUDA(cudaStreamWaitEvent(st, fk->joined, 0));
    }
    FwdParams fp{};
    fp.B = d->B; fp.T = d->T; fp.H = d->H; fp.O = d->O;
    fp.alif = d->layer_type == SNNK_ALIF; fp.traces = traces;
    fp.iz = izh_consts(d);
    fp.alpha = d->alpha; fp.rho = d->rho; fp.theta = d->theta; fp.kappa = d->kappa;
    fp.I_in = I_in; fp.W_eff = W_eff; fp.beta = beta; fp.W_out = W_out; fp.b_out = b_out;
    fp.V0 = V0; fp.a0 = a0; fp.Z0 = Z0; fp.V = V; fp.a = a; fp.Z = Z; fp.zbits = zbits; fp.y = y;
    fp.logits = logits; fp.tstar = tstar;
    fp.run_table = runs; fp.I_u = compact_rows;   // k_recur_fwd / k_recur_fwd_tc fetch the compact rows themselves
    const bool rec = d->recurrent != 0;
    // the register-resident recurrence evaluates the head in its own tail; every other kernel family is followed by
    // the stand-alone head kernel (same arithmetic, same summation order)
    const bool fused_head = head && pl.readout_in_sweep();
    if (fused_head) {
        fp.labels = reinterpret_cast<const long long*>(head->labels); fp.logp = head->logp; fp.g_logits = head->g_logits;
        fp.loss = head->loss; fp.part_nll = static_cast<float*>(head->head_ws);
        fp.ticket = reinterpret_cast<unsigned int*>(static_cast<float*>(head->head_ws) + d->B);
        fp.mailbox = reinterpret_cast<unsigned long long*>(head->mailbox); fp.mail_counter = head->counter;
    }
    switch (pl.family) {
    case Family::WideTc:
        rc = launch_wide_fwd(wide_params(fp, pl, ws), st);
        if (rc == SNNK_OK) rc = launch_readout_scan(d, fp, st);
        break;
    case Family::WideGen:
        rc = launch_fwd_gen(d, fp, rec, pl, st);
        if (rc == SNNK_OK) rc = launch_readout_scan(d, fp, st);
        break;
    case Family::TcRec: rc = launch_fwd_tc(fp, st); break;
    case Family::NonRec: rc = launch_nonrec_fwd(fp, st); break;
    case Family::Simt:
        // the lean kernel is a programmatic dependent of a tensor-core projection on the same stream (not while the
        // per-kernel profiler brackets launches with events)
        rc = pl.lean_fwd ? launch_fwd_lean(fp, st, pl.tc && !g_prof_on) : launch_fwd_simt(fp, rec, pl, st);
        break;
    }
    if (rc != SNNK_OK || !head || fused_head) return rc;
    return snnk_head_nll(d->B, d->O, logits, head->labels, head->logp, head->loss, head->g_logits, head->mailbox,
                         head->counter, stream);
}

int snnk_forward(const SnnkDesc* d, const float* x, const float* W_in, const float* W_rec, const float* rec_mask,
                 const float* beta, const float* W_out, const float* b_out, const float* V0, const float* a0,
                 const float* Z0, float* V, float* a, float* Z, uint32_t* zbits, float* y, float* logits,
                 int32_t* tstar, void* workspace, size_t workspace_bytes, const int32_t* run_table, float* W_effT_out,
                 snnk_stream_t stream)
{
    return forward_impl(d, x, W_in, W_rec, rec_mask, beta, W_out, b_out, V0, a0, Z0, V, a, Z, zbits, y, logits, tstar,
                        workspace, workspace_bytes, run_table, W_effT_out, stream, nullptr);
}

int snnk_forward_nll(const SnnkDesc* d, const float* x, const float* W_in, const float* W_rec, const float* rec_mask,
                     const float* beta, const float* W_out, const float* b_out, const float* V0, const float* a0,
                     const float* Z0, float* V, float* a, float* Z, uint32_t* zbits, float* y, float* logits,
                     int32_t* tstar, void* workspace, size_t workspace_bytes, const int32_t* run_table, float* W_effT_out,
                     const int64_t* labels, float* logp, float* loss, float* g_logits, void* head_ws,
                     uint64_t* loss_mailbox, uint32_t* mailbox_counter, snnk_stream_t stream)
{
    if (!labels || !loss || !head_ws) return SNNK_ERR_ARG;
    if ((loss_mailbox != nullptr) != (mailbox_counter != nullptr)) return SNNK_ERR_ARG;
    const HeadArgs h{labels, logp, loss, g_logits, head_ws, loss_mailbox, mailbox_counter};
    return forward_impl(d, x, W_in, W_rec, rec_mask, beta, W_out, b_out, V0, a0, Z0, V, a, Z, zbits, y, logits, tstar,
                        workspace, workspace_bytes, run_table, W_effT_out, stream, &h);
}

int snnk_head_nll(int32_t B, int32_t O, const float* logits, const int64_t* labels, float* logp, float* loss,
                  float* g_logits, uint64_t* loss_mailbox, uint32_t* mailbox_counter, snnk_stream_t stream)
{
    if (!logits || !labels || !loss) return SNNK_ERR_ARG;
    if ((loss_mailbox != nullptr) != (mailbox_counter != nullptr)) return SNNK_ERR_ARG;
    if (B <= 0 || O <= 0 || O > kOMax) return SNNK_ERR_SHAPE;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    return launch(SNNK_K_HEAD, k_head_nll, 1, 256, 0, static_cast<cudaStream_t>(stream), B, O, logits,
                  reinterpret_cast<const long long*>(labels), logp, loss, g_logits,
                  reinterpret_cast<unsigned long long*>(loss_mailbox), mailbox_counter);
}

// The tensor list of both Adam entry points (1 <= count <= kAdamMaxTensors, non-null arrays), checked and packed
static int adam_tensors(int32_t count, float* const* params, const float* const* grads, float* const* exp_avg,
                        float* const* exp_avg_sq, float* const* steps, const int64_t* numel, AdamTensors* t)
{
    *t = AdamTensors{};
    t->count = count;
    long long total = 0;
    for (int k = 0; k < count; ++k) {
        if (!params[k] || !grads[k] || !exp_avg[k] || !exp_avg_sq[k] || !steps[k] || numel[k] < 0) return SNNK_ERR_ARG;
        t->p[k] = params[k]; t->g[k] = grads[k]; t->m[k] = exp_avg[k]; t->v[k] = exp_avg_sq[k]; t->step[k] = steps[k];
        t->n[k] = numel[k]; t->start[k] = total; total += numel[k];
    }
    t->start[count] = total;
    return SNNK_OK;
}

int snnk_adam_step(int32_t count, float* const* params, const float* const* grads, float* const* exp_avg,
                   float* const* exp_avg_sq, float* const* steps, const int64_t* numel, float lr, float beta1, float beta2,
                   float eps, float weight_decay, snnk_stream_t stream)
{
    if (count < 0 || count > kAdamMaxTensors) return SNNK_ERR_SHAPE;
    if (count == 0) return SNNK_OK;
    if (!params || !grads || !exp_avg || !exp_avg_sq || !steps || !numel) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    AdamTensors t;
    const int rc = adam_tensors(count, params, grads, exp_avg, exp_avg_sq, steps, numel, &t);
    if (rc != SNNK_OK) return rc;
    const long long total = t.start[count];
    return launch(SNNK_K_ADAM, k_adam_step, (unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream), t,
                  lr, beta1, beta2, eps, weight_decay);
}

int snnk_adam_dp_buffer_bytes(int32_t world, int64_t total_numel, size_t* bytes)
{
    if (!bytes) return SNNK_ERR_ARG;
    if (world < 1 || world > kDpMaxWorld || total_numel < 0) return SNNK_ERR_SHAPE;
    *bytes = (size_t)2 * world * (size_t)total_numel * sizeof(unsigned long long);
    return SNNK_OK;
}

int snnk_adam_step_dp(int32_t count, float* const* params, float* const* grads, float* const* exp_avg,
                      float* const* exp_avg_sq, float* const* steps, const int64_t* numel, float lr, float beta1, float beta2,
                      float eps, float weight_decay, int32_t rank, int32_t world, void* const* peer_buffers,
                      uint32_t* state, snnk_stream_t stream)
{
    if (count < 0 || count > kAdamMaxTensors) return SNNK_ERR_SHAPE;
    if (world < 1 || world > kDpMaxWorld || rank < 0 || rank >= world) return SNNK_ERR_SHAPE;
    if (count == 0) return SNNK_OK;
    if (!params || !grads || !exp_avg || !exp_avg_sq || !steps || !numel || !peer_buffers || !state) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    AdamTensors t;
    const int rc = adam_tensors(count, params, grads, exp_avg, exp_avg_sq, steps, numel, &t);
    if (rc != SNNK_OK) return rc;
    const long long total = t.start[count];
    AdamDp dp{};
    dp.rank = rank; dp.world = world; dp.state = state;
    {   // two-phase exchange from 4 ranks on (at 2 the all-to-all IS one hop and one word); SNNK_DP_RSAG=0/1 forces it --
        // every rank must decide alike, which an environment variable of the launcher guarantees
        const char* env = getenv("SNNK_DP_RSAG");
        dp.rsag = env ? (env[0] != '0' && world >= 2) : (world >= 4);
    }
    for (int r = 0; r < world; ++r) {
        if (!peer_buffers[r]) return SNNK_ERR_ARG;
        if (reinterpret_cast<uintptr_t>(peer_buffers[r]) & 7) return SNNK_ERR_ARG;
        dp.slots[r] = static_cast<unsigned long long*>(peer_buffers[r]);
    }
    // one gradient element per thread: every remote store of the step is in flight at once.  Threads only wait for
    // REMOTE data, never for another local CTA, so the grid need not be co-resident.
    const long long want = (total + 255) / 256;
    const unsigned grid = (unsigned)std::min<long long>(want, 8ll * sm_count());
    return launch(SNNK_K_ADAM, k_adam_step_dp, grid, 256, 0, static_cast<cudaStream_t>(stream), t, dp, lr, beta1, beta2,
                  eps, weight_decay);
}

int snnk_input_grad(const SnnkDesc* d, const float* gI, const float* W_in, float* gX, snnk_stream_t stream)
{
    int rc = check_desc(d);
    if (rc != SNNK_OK) return rc;
    if (!gI || !W_in || !gX) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    const int M = d->B * d->T;
    return launch(SNNK_K_INPUT_GRAD, k_input_grad_simt, dim3((M + kGemmBM - 1) / kGemmBM, (d->N + 63) / 64), kGemmThreads,
                  0, static_cast<cudaStream_t>(stream), gI, W_in, gX, M, d->H, d->N);
}

int snnk_backward(const SnnkDesc* d, const float* x, const float* W_rec, const float* rec_mask, const float* beta,
                  const float* W_out, const float* Z0, const float* V, const float* a, const float* Z,
                  const uint32_t* zbits, const float* g_y, const float* g_logits, const int32_t* tstar, const float* g_scale,
                  const float* g_V, const float* g_Z, float* dW_in, float* dW_rec, float* dW_out, float* db, void* workspace,
                  size_t workspace_bytes, const int32_t* run_table, const float* W_effT_in, snnk_stream_t stream)
{
    int rc = check_desc(d);
    if (rc != SNNK_OK) return rc;
    // sigma' trace: it arrives in `a` and is the only trace of V a LIF / ALIF sweep reads (Izhikevich still needs V)
    const bool trace = d->surrogate == SNNK_SURROGATE_TRACE, izh = d->layer_type == SNNK_IZHIKEVICH;
    if (!x || !W_out || !zbits || !dW_in || !dW_out || !db || !workspace) return SNNK_ERR_ARG;
    if ((!trace || izh) && !V) return SNNK_ERR_ARG;
    if (trace && !a) return SNNK_ERR_ARG;
    if (d->recurrent && (!W_rec || !dW_rec)) return SNNK_ERR_ARG;
    if (d->recurrent && (d->flags & SNNK_F_TENSOR_CORE) && !Z) return SNNK_ERR_ARG;
    if (!trace && d->layer_type == SNNK_ALIF && (!beta || !a)) return SNNK_ERR_ARG;
    const bool dense = g_y != nullptr, sparse = g_logits != nullptr && tstar != nullptr;
    if (dense == sparse) return SNNK_ERR_ARG;
    if (!device_ok()) return SNNK_ERR_DEVICE;
    const Plan pl = make_plan(d);
    if (workspace_bytes < pl.bwd_bytes) return SNNK_ERR_WORKSPACE;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(workspace);
    float* gI = reinterpret_cast<float*>(ws + pl.off_gI);
    float* pwout = reinterpret_cast<float*>(ws + pl.off_pwout);
    float* pdb = reinterpret_cast<float*>(ws + pl.off_pdb);
    float* pw = reinterpret_cast<float*>(ws + pl.off_pw);
    const bool rec = d->recurrent != 0;
    const int* runs = pl.dedup ? run_table : nullptr;
    float* gy_scan = reinterpret_cast<float*>(ws + pl.off_gyscan);

    // Parallel branches: the gather of the dedup variant, and the dW_out / db partials of the tensor-core and
    // non-recurrent sweeps
    const bool wout_beside = pl.family == Family::TcRec || pl.family == Family::NonRec;
    Fork* fk = nullptr;
    if (runs || wout_beside) {
        rc = fork_for_device(&fk);
        if (rc != SNNK_OK) return rc;
    }
    // dedup variant: the compact rows of x for the dW_in GEMM do not depend on the sweep -- gathered beside it
    if (runs) {
        SNNK_CUDA(cudaEventRecord(fk->forked, st));
        SNNK_CUDA(cudaStreamWaitEvent(fk->side, fk->forked, 0));
        k_gather_rows<<<std::min(pl.run_rows, 8 * sm_count()), 256, 0, fk->side>>>(
            x, runs, d->B * d->T, d->N, reinterpret_cast<float*>(ws + pl.off_xu_b));
        SNNK_CUDA(cudaGetLastError());
        SNNK_CUDA(cudaEventRecord(fk->mid, fk->side));
    }
    // K3: reverse-time sweep
    const float* W_effT = nullptr;
    if (rec && W_effT_in) {
        W_effT = W_effT_in;      // prepared by snnk_forward of the same weights (its W_effT_out)
    } else if (rec) {
        float* wt = reinterpret_cast<float*>(ws + pl.off_weffT);
        const int n = d->H * d->H;
        k_prep_rec<<<(n + 255) / 256, 256, 0, st>>>(W_rec, rec_mask, d->H, nullptr, wt);
        SNNK_CUDA(cudaGetLastError());
        W_effT = wt;
    }
    BwdParams bp{};
    bp.B = d->B; bp.T = d->T; bp.H = d->H; bp.O = d->O;
    bp.alif = d->layer_type == SNNK_ALIF && !trace; bp.surrogate = d->surrogate;
    bp.iz = izh_consts(d);
    bp.alpha = d->alpha; bp.theta = d->theta; bp.gamma = d->gamma; bp.kappa = d->kappa;
    bp.W_effT = W_effT; bp.beta = beta; bp.W_out = W_out; bp.Z0 = Z0;
    const bool sg_in_v = trace && !izh;     // LIF / ALIF: the LIF-mode sweep reads sigma' in the V slot
    bp.V = sg_in_v ? a : V; bp.a = sg_in_v ? nullptr : a; bp.zbits = zbits; bp.g_y = g_y;
    bp.g_logits = dense ? nullptr : g_logits;
    bp.tstar = dense ? nullptr : tstar; bp.g_scale = g_scale; bp.g_V = g_V; bp.g_Z = g_Z;
    float* gI_lo = pl.tc ? reinterpret_cast<float*>(ws + pl.off_gIlo) : nullptr;
    bp.gI = gI; bp.gI_lo = gI_lo; bp.part_wout = pwout; bp.part_db = pdb;
    if (runs) {
        bp.run_table = runs;
        bp.Gu_hi = reinterpret_cast<float*>(ws + pl.off_gu);
        bp.Gu_lo = reinterpret_cast<float*>(ws + pl.off_gu + pl.gu_plane);
    }
    switch (pl.family) {
    case Family::WideTc: {
        // weight-stationary tensor-core sweep (recur_wide.cuh): adjoint scan, sweep, then dW_out / db from the scan
        rc = launch_gy_scan(d, bp, gy_scan, st);
        if (rc != SNNK_OK) return rc;
        WideBwdParams wp{};
        wp.B = d->B; wp.T = d->T; wp.H = d->H; wp.O = d->O; wp.alif = bp.alif; wp.surrogate = bp.surrogate;
        wp.alpha = bp.alpha; wp.theta = bp.theta; wp.gamma = bp.gamma;
        wp.W = bp.W_effT; wp.beta = bp.beta; wp.W_out = bp.W_out; wp.V = bp.V; wp.a = bp.a; wp.zbits = bp.zbits; wp.Z0 = bp.Z0;
        wp.gy_scan = gy_scan; wp.g_V = bp.g_V; wp.g_Z = bp.g_Z; wp.gI = bp.gI; wp.gI_lo = bp.gI_lo;
        wp.gx = reinterpret_cast<float*>(ws + pl.off_gx);
        wp.gmask = reinterpret_cast<unsigned int*>(ws + pl.off_gmask);
        wp.flags = reinterpret_cast<unsigned int*>(ws + pl.off_wflags_b);
        wp.n_mt = pl.w_nmt_b; wp.n_nt = pl.w_nnt;
        rc = launch_wide_bwd(wp, pl.w_npass_b, st);
        if (rc == SNNK_OK) rc = launch_wout_grad(d, pl, zbits, gy_scan, pwout, pdb, st);
        break;
    }
    case Family::WideGen:
        rc = launch_bwd_gen(d, bp, rec, pl, gy_scan, st);
        if (rc == SNNK_OK) rc = launch_wout_grad(d, pl, zbits, gy_scan, pwout, pdb, st);
        break;
    case Family::TcRec:
    case Family::NonRec:
        // readout-adjoint scan first; dW_out / db (a contraction of it with the spike raster) beside the sweep
        rc = launch_gy_scan(d, bp, gy_scan, st);
        if (rc != SNNK_OK) return rc;
        SNNK_CUDA(cudaEventRecord(fk->forked3, st));
        SNNK_CUDA(cudaStreamWaitEvent(fk->side, fk->forked3, 0));
        rc = launch_wout_grad(d, pl, zbits, gy_scan, pwout, pdb, fk->side);
        if (rc != SNNK_OK) return rc;
        SNNK_CUDA(cudaEventRecord(fk->joined3, fk->side));
        rc = pl.family == Family::TcRec ? launch_bwd_tc(bp, gy_scan, st) : launch_nonrec_bwd(bp, gy_scan, st);
        break;
    case Family::Simt:
        rc = use_lean_bwd(bp, rec, pl.R) ? launch_bwd_lean(bp, st) : launch_bwd_simt(bp, rec, pl, st);
        break;
    }
    if (rc != SNNK_OK) return rc;
    // K4: weight-gradient GEMM (split-K partials over whole samples, then a fixed-order reduction)
    {
        unsigned int* flag = nullptr;
        if ((d->flags & SNNK_F_INPUT_BITS) && !pl.bits) return SNNK_ERR_UNSUPPORTED;
        if (pl.bits) {
            const uint32_t* xb = reinterpret_cast<const uint32_t*>(x);
            const size_t gstride = pl.off_gIlo - pl.off_gI;
            rc = by_width(pl.tileN, [&](auto tn) {
                return launch_wgrad_bits<decltype(tn)::value>(d, pl, xb, zbits, gI, gstride, pw, st);
            });
            if (rc != SNNK_OK) return rc;
        } else if (pl.tc) {
            if (pl.check) {
                flag = reinterpret_cast<unsigned int*>(ws + pl.off_flag);
                SNNK_CUDA(cudaMemsetAsync(flag, 0, sizeof(unsigned int), st));
            }
            WgradGeom g{};
            g.x = x; g.Ztrace = rec ? Z : nullptr; g.g_planes = gI; g.g_plane_stride = pl.off_gIlo - pl.off_gI;
            g.T = d->T; g.B = d->B; g.N = d->N; g.mtiles_x = pl.mtiles_x; g.mtiles_z = pl.mtiles_z; g.m_total = pl.m_total;
            g.S = pl.S; g.samples_per_split = pl.samples_per_split; g.part = pw; g.flag = flag;
            g.run_table = runs; g.run_gate = 0; g.run_clip = 0;
            cudaStream_t st_b = st;
            if (runs) {   // dense (self-skipping) launch + Z-only GEMM on a parallel branch beside the compact GEMM
                SNNK_CUDA(cudaEventRecord(fk->forked2, st));
                SNNK_CUDA(cudaStreamWaitEvent(fk->side, fk->forked2, 0));
                st_b = fk->side;
            }
            rc = launch_wgrad_tc_any(d, pl.tileN, g, st_b);
            if (rc != SNNK_OK) return rc;
            if (runs) {
                // dedup variant: x-only GEMM over the compact rows (run sums of gI come from the BPTT sweep) and Z-only
                // GEMM over the dense rows; the two are independent
                if (rec) {
                    WgradGeom gb = g;
                    gb.x = nullptr; gb.N = 0; gb.mtiles_x = 0; gb.m_total = d->H; gb.S = pl.S_rec;
                    gb.samples_per_split = pl.sps_rec; gb.part = reinterpret_cast<float*>(ws + pl.off_pwrec); gb.flag = nullptr;
                    gb.run_gate = 1; gb.run_clip = 0;
                    rc = launch_wgrad_tc_any(d, pl.tileN, gb, st_b);
                    if (rc != SNNK_OK) return rc;
                }
                SNNK_CUDA(cudaStreamWaitEvent(st, fk->mid, 0));   // the gather issued beside the sweep
                WgradGeom ga{};
                ga.x = reinterpret_cast<float*>(ws + pl.off_xu_b); ga.Ztrace = nullptr;
                ga.g_planes = reinterpret_cast<float*>(ws + pl.off_gu); ga.g_plane_stride = pl.gu_plane;
                ga.T = pl.run_rows; ga.B = 1; ga.N = d->N; ga.mtiles_x = pl.mtiles_x; ga.mtiles_z = 0; ga.m_total = pl.m_total;
                ga.S = pl.S_cmp; ga.samples_per_split = 1; ga.part = pw; ga.flag = nullptr;
                ga.run_table = runs; ga.run_gate = 1; ga.run_clip = 1;
                rc = launch_wgrad_tc_any(d, pl.tileN, ga, st);
                if (rc != SNNK_OK) return rc;
                SNNK_CUDA(cudaEventRecord(fk->joined, fk->side));
                SNNK_CUDA(cudaStreamWaitEvent(st, fk->joined, 0));
            }
        }
        WgradParams wp{};
        wp.BT = d->B * d->T; wp.T = d->T; wp.N = d->N; wp.H = d->H;
        wp.mtiles_x = pl.mtiles_x; wp.rows_per_split = pl.samples_per_split * d->T;
        wp.x = x; wp.zbits = zbits; wp.Z0 = Z0; wp.gI = gI; wp.gI_lo = gI_lo; wp.run_if_flag = flag;
        wp.part = pw; wp.m_total = pl.m_total;
        if (!pl.bits && (!pl.tc || pl.check)) {
            rc = launch(pl.tc ? SNNK_K_WGRAD_FALLBACK : SNNK_K_WGRAD, pl.BN == 64 ? k_wgrad_simt<64> : k_wgrad_simt<32>,
                        dim3(pl.mtiles_x + pl.mtiles_z, pl.ntiles, pl.S), kGemmThreads, 0, st, wp);
            if (rc != SNNK_OK) return rc;
        }
        if (wout_beside) SNNK_CUDA(cudaStreamWaitEvent(st, fk->joined3, 0));      // dW_out / db partials of the side branch
        // every partial buffer (dW_in, dW_rec, dW_out, db) reduced by one launch
        FinalizeParams fz{};
        fz.pw = pw; fz.S = pl.S; fz.w_stride = (size_t)pl.m_total * d->H; fz.n_in = d->N * d->H;
        fz.n_rec = rec ? d->H * d->H : 0; fz.rec_mask = rec_mask; fz.dW_in = dW_in; fz.dW_rec = dW_rec;
        fz.pwout = pwout; fz.P_out = pl.n_pwout; fz.n_out = d->H * d->O; fz.dW_out = dW_out;
        fz.pdb = pdb; fz.P_b = pl.n_pdb; fz.n_b = d->O; fz.db = db;
        if (runs) {
            fz.run_table = runs; fz.S_cmp = pl.S_cmp;
            if (rec) {
                fz.pw_rec = reinterpret_cast<float*>(ws + pl.off_pwrec); fz.S_rec = pl.S_rec;
                fz.rec_stride = (size_t)d->H * d->H;
            }
        }
        fz.blocks_a = (fz.n_in + fz.n_rec + 255) / 256;
        const int blocks_b = (fz.n_out + fz.n_b + 7) / 8;
        return launch(SNNK_K_REDUCE_W, k_finalize_grads, fz.blocks_a + blocks_b, 256, 0, st, fz);
    }
}

}  // extern "C"
