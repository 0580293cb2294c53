/*
 * snnk.h -- C ABI of the B200-native spiking hot path (libsnnk.so).
 *
 * The reference (JeremieGince/SNNImageClassification) is pure Python and has no
 * FFI layer of its own; its boundary for this path is the Python surface
 *   SNN.forward                    src/modules/snn.py:201-219
 *   LIFLayer/ALIFLayer/ReadoutLayer.forward
 *                                  src/modules/spiking_layers.py:156-171, :229-243, :402-408
 *   SpikeFunction / surrogate backward
 *                                  src/modules/spike_funcs.py:12-29, :46-62, :65-79
 *   loss.backward() over the unrolled graph
 *                                  src/modules/snn.py:413
 *   ToSpikes.__call__              src/datasets/datasets.py:42-54, :72-86, :93-97
 *   max-over-time/log_softmax/NLL  src/modules/snn.py:228, :258, :297
 * Each entry point below replaces the loop named beside it; the Python mirror
 * in snnimageclassification_b200/ binds them with ctypes (INTEGRATION.md shows
 * the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     stated otherwise; all tensors are dense, C-contiguous, fp32 unless stated
 *   - the caller owns every buffer and the workspace; the library never
 *     allocates device memory and never synchronises; all work is enqueued on
 *     the stream passed in (a cudaStream_t cast to void*)
 *   - return value: SNNK_OK (0) or a negative SNNK_ERR_* code; no exceptions
 *     cross the ABI; snnk_strerror() gives the text, snnk_last_cuda_error() the
 *     CUDA runtime message behind SNNK_ERR_CUDA
 *   - stateless and re-entrant (one host thread per rank; data-parallel ranks
 *     are separate processes)
 *   - sm_100 only: there is no fallback path; on any other device every compute
 *     entry point returns SNNK_ERR_DEVICE
 */
#ifndef SNNK_H
#define SNNK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNNK_ABI_VERSION 8   /* 8: SNNK_F_RUNS_TILED, snnk_run_table_tiled_bytes; 7: snnk_forward_nll; 6: SNNK_F_INPUT_BITS; 5: loss mailbox of snnk_head_nll; 4: W_effT_out / W_effT_in; 2: run_table argument of snnk_forward / snnk_backward, snnk_encode_runs, snnk_adam_step_dp; 3: Izhikevich fields of SnnkDesc */

typedef void* snnk_stream_t; /* cudaStream_t */

/* LayerType, src/modules/spiking_layers.py:11-14.  SNNK_IZHIKEVICH (spiking_layers.py:246-353; wider than 128: the fp32 kernels of recur_gen.cuh): the
 * `a` trace and the a0 state hold the recovery variable u; V0 == NULL starts the membrane at v_rest (:309). */
enum { SNNK_LIF = 0, SNNK_ALIF = 1, SNNK_IZHIKEVICH = 2 };
/* SpikeFuncType, src/modules/spike_funcs.py:7-9.  SNNK_SURROGATE_TRACE: a user-defined SpikeFunction subclass whose
 * derivative the caller evaluates itself and hands to snnk_backward as a trace (see there); snnk_forward and
 * snnk_forward_nll accept it and ignore it (the forward is the same Heaviside step), snnk_spike_backward refuses it. */
enum { SNNK_FAST_SIGMOID = 0, SNNK_PHI = 1, SNNK_SURROGATE_TRACE = 2 };
/* element types accepted by snnk_encode */
enum { SNNK_F32 = 0, SNNK_F64 = 1, SNNK_U8 = 2, SNNK_I64 = 3, SNNK_BITS = 4 };

enum {
    SNNK_OK = 0,
    SNNK_ERR_ARG = -1,         /* null pointer / bad enum / bad flag */
    SNNK_ERR_SHAPE = -2,       /* geometry outside what the kernels support */
    SNNK_ERR_DEVICE = -3,      /* current device is not sm_100 */
    SNNK_ERR_WORKSPACE = -4,   /* workspace too small */
    SNNK_ERR_CUDA = -5,        /* a CUDA runtime call failed: see snnk_last_cuda_error() */
    SNNK_ERR_UNSUPPORTED = -6  /* valid request the library does not implement */
};

/* SnnkDesc.flags */
#define SNNK_F_TRACES 0x1u     /* write the hidden traces V,(a),Z (snn.py:216-219) */
#define SNNK_F_TENSOR_CORE 0x2u /* allow the tcgen05 projection / weight-gradient GEMMs (exact for {0,1}
                                  inputs; the library falls back to the fp32 SIMT GEMM when x is not
                                  exactly representable) */

#define SNNK_F_INPUT_BINARY 0x4u /* the caller guarantees x is exactly {0,1} (its own encoder's output, or the
                                  spike trace of the layer below): the tensor-core kernels skip their on-device
                                  exactness check and the gated fp32 fallback launches */

#define SNNK_F_INPUT_BITS 0x8u  /* x is the BIT-PACKED raster (B*T, ceil(N/32)) uint32 -- the SNNK_BITS output of
                                  snnk_encode, bit l of word w = feature 32w+l, padding bits zero -- instead of fp32
                                  (cast the pointer).  Needs SNNK_F_TENSOR_CORE and N % 4 == 0, else
                                  SNNK_ERR_UNSUPPORTED (unpack with snnk_unpack_raster then).  The projection and
                                  the weight-gradient contraction expand the words inside shared memory
                                  (k_proj_bits / k_wgrad_bits): the fp32 raster of datasets.py:93-97 never exists.
                                  A run table is ignored with this flag (dense kernels). */

#define SNNK_F_RUNS_TILED 0x10u /* the run table passed to snnk_forward / snnk_forward_nll is followed by the compact rows
                                  tiled for the projection (snnk_run_table_tiled_bytes, snnk_encode_runs with lazy & 2):
                                  the per-step gather of those rows is skipped */

/* Geometry and constants of one hidden spiking layer + leaky readout. */
typedef struct SnnkDesc {
    int32_t B;          /* batch rows (independent)                           */
    int32_t T;          /* time steps, snn.py:58 int_time_steps               */
    int32_t N;          /* input features (784)                               */
    int32_t H;          /* hidden neurons                                     */
    int32_t O;          /* readout units (10); O <= 16                        */
    int32_t layer_type; /* SNNK_LIF | SNNK_ALIF | SNNK_IZHIKEVICH             */
    int32_t surrogate;  /* SNNK_FAST_SIGMOID | SNNK_PHI | SNNK_SURROGATE_TRACE */
    int32_t recurrent;  /* use_recurrent_connection                           */
    float alpha;        /* exp(-dt/tau_m),  spiking_layers.py:119             */
    float rho;          /* exp(-dt/tau_a),  spiking_layers.py:199 (ALIF)      */
    float theta;        /* threshold,       spiking_layers.py:120             */
    float gamma;        /* surrogate scale, spiking_layers.py:121             */
    float kappa;        /* exp(-dt/tau_out),spiking_layers.py:377             */
    uint32_t flags;     /* SNNK_F_*                                           */
    /* SNNK_IZHIKEVICH only (ignored otherwise), spiking_layers.py:275-296: next_V = (V + dt (k (V - v_rest)(V - v_th)
     * - u + I) / C)(1 - Z) + c Z;  next_u = u + dt a (b (V - v_rest) - u) + d Z;  spike at v_peak */
    float dt, iz_C, iz_v_rest, iz_v_th, iz_k, iz_a, iz_b, iz_c, iz_d, iz_v_peak;
} SnnkDesc;

/* kernel groups reported by the optional profiler below */
enum {
    SNNK_K_ENCODE = 0, SNNK_K_PROJ = 1, SNNK_K_RECUR_FWD = 2, SNNK_K_HEAD = 3, SNNK_K_RECUR_BWD = 4,
    SNNK_K_REDUCE_OUT = 5, SNNK_K_WGRAD = 6, SNNK_K_REDUCE_W = 7, SNNK_K_PROJ_FALLBACK = 8,
    SNNK_K_WGRAD_FALLBACK = 9, SNNK_K_INPUT_GRAD = 10, SNNK_K_ADAM = 11, SNNK_K_COUNT = 12
};

int snnk_abi_version(void);
const char* snnk_strerror(int code);
/* Host string describing the last CUDA runtime error seen by this thread ("" if none). */
const char* snnk_last_cuda_error(void);
/* 1 if the CURRENT CUDA device is sm_100 (B200), 0 if not, <0 on error. */
int snnk_device_supported(void);

/*
 * Optional per-kernel timing (bench.py's roofline): between snnk_profile_begin() and snnk_profile_end()
 * every kernel launch of this library is bracketed by CUDA events on its stream.  snnk_profile_end()
 * synchronises the device (the one exception to "never synchronises") and fills ms_total[SNNK_K_COUNT]
 * (summed kernel time per group, milliseconds) and launches[SNNK_K_COUNT].  Process-global debug
 * facility; not for concurrent use.
 */
const char* snnk_kernel_name(int id);
int snnk_profile_begin(void);
int snnk_profile_end(double* ms_total, int64_t* launches);

/*
 * Image -> spike-train encoder.  Replaces ToSpikes.__call__ (datasets.py:93-97) for a whole batch.
 *   x    (n_items, n_pix)            x_dtype  SNNK_F32 | SNNK_F64 (arithmetic is done in that type, as numpy does)
 *                                    or SNNK_I64: x already holds firing times / periods, i.e. the call is
 *                                    firing_times_to_spikes (datasets.py:81-86) / firing_periods_to_spikes (:72-79)
 *   out  (n_items, n_steps, n_pix)   out_dtype SNNK_F32 | SNNK_F64 | SNNK_U8, values in {0,1}; or SNNK_BITS:
 *                                    (n_items, n_steps, ceil(n_pix/32)) uint32, bit l of word w = pixel 32 w + l --
 *                                    the raster at 1/32 of its fp32 size for storage and host <-> device transport
 *                                    (SURVEY.md 8f.1); snnk_unpack_raster turns it back into fp32 {0,1}
 *   periods (n_items, n_pix) int64, optional (may be NULL): pixels_to_firing_periods (datasets.py:42-54)
 *   periodic = use_periods (datasets.py:40)
 */
int snnk_encode(const void* x, int32_t x_dtype, int64_t n_items, int64_t n_pix, int32_t n_steps,
                double t_max, double tau, double thr, double eps, int32_t periodic, void* out,
                int32_t out_dtype, int64_t* periods, snnk_stream_t stream);

/* bits (n_rows, ceil(n_pix/32)) uint32 -> out (n_rows, n_pix) fp32 {0,1}: the inverse of the SNNK_BITS raster format. */
int snnk_unpack_raster(const uint32_t* bits, int64_t n_rows, int32_t n_pix, float* out, snnk_stream_t stream);

/*
 * Frame runs of an encoded batch (SURVEY.md 8f.1, "frame-dedup fast path for production ToSpikes output").
 * ToSpikes with the production tau = 0.02 (datasets.py:21) emits at most three distinct frames per item, so
 * consecutive time steps mostly repeat the previous frame.  snnk_encode_runs is snnk_encode that also records
 *   frame_changed (n_items, n_steps) uint8: 1 where frame t differs from frame t-1 (scratch owned by the caller)
 *   run_table     int32, snnk_run_table_bytes(n_items, n_steps) bytes:
 *                 [0] number of runs in the batch  [1] ok: 1 when that number fits the table's capacity
 *                 [2] capacity = max(128, n_items*n_steps/4 rounded up to 128)  [3] 0
 *                 [4 ..) for every dense row item*n_steps+t the index of its run; then capacity first-rows; then
 *                 capacity run lengths; then n_items words of scratch.
 * lazy != 0: `out` is only written where a consumer of the table will read it -- every row when the table is not
 * ok, otherwise just the first row of every run (the rest of `out` stays uninitialised): for callers that hand
 * `out` to snnk_forward / snnk_backward together with the table and to nobody else.
 * snnk_frame_runs builds the table from change flags the caller produced itself.  snnk_forward / snnk_backward
 * take the table of THEIR input x (or NULL): with SNNK_F_TENSOR_CORE | SNNK_F_INPUT_BINARY and H <= 128 the input
 * projection is then evaluated once per run and the dW_in contraction runs over runs instead of rows.  Whether
 * that variant or the dense one executes is decided on the device from word [1]; both are always enqueued, so
 * the call stays CUDA-graph capturable and a batch with too many runs silently takes the dense kernels.
 */
size_t snnk_run_table_bytes(int64_t n_items, int32_t n_steps);
/* Table + (1 KB aligned) the first row of every run as the 128-row x 32-feature swizzled tiles the compact projection
 * reads (fp32 rasters, n_pix % 4 == 0; else 0).  snnk_encode_runs fills that tail when bit 1 of `lazy` is set (bit 0:
 * lazy raster), and a forward call given such a table sets SNNK_F_RUNS_TILED. */
size_t snnk_run_table_tiled_bytes(int64_t n_items, int32_t n_steps, int32_t n_pix);
int snnk_frame_runs(int64_t n_items, int32_t n_steps, const uint8_t* frame_changed, int32_t* run_table,
                    snnk_stream_t stream);
int snnk_encode_runs(const void* x, int32_t x_dtype, int64_t n_items, int64_t n_pix, int32_t n_steps,
                     double t_max, double tau, double thr, double eps, int32_t periodic, void* out,
                     int32_t out_dtype, int64_t* periods, uint8_t* frame_changed, int32_t* run_table,
                     int32_t lazy, snnk_stream_t stream);

/*
 * SpikeFunction.apply used stand-alone (spike_funcs.py:12-29): out = (v >= thr) ? 1 : 0, and its surrogate
 * backward (spike_funcs.py:46-62 FastSigmoid, :65-79 Phi): g_in = g_out * sigma'(v, thr, gamma).  thr has n
 * elements or 1 (broadcast); gamma is a device scalar.  The threshold and gamma get no gradient.
 */
int snnk_spike_forward(const float* v, const float* thr, int64_t n, int64_t thr_n, float* out,
                       snnk_stream_t stream);
int snnk_spike_backward(int32_t surrogate, const float* v, const float* thr, const float* gamma,
                        const float* g_out, int64_t n, int64_t thr_n, float* g_in, snnk_stream_t stream);

size_t snnk_forward_workspace_bytes(const SnnkDesc* d);
size_t snnk_backward_workspace_bytes(const SnnkDesc* d);

/*
 * Forward over all T steps.  Replaces the time loop of SNN.forward (snn.py:209-214) around
 * LIFLayer/ALIFLayer.forward and ReadoutLayer.forward, plus torch.stack (snn.py:216-218) and the
 * max over time of get_prediction_logits (snn.py:228).
 *   x        (B,T,N)  input spikes / currents
 *   W_in     (N,H)    forward_weights;  W_rec (H,H) recurrent_weights (raw), NULL iff !recurrent
 *   rec_mask (H,H)    or NULL for all-ones (spiking_layers.py:50-57)
 *   beta     device scalar (ALIF; may be an nn.Parameter), NULL for LIF
 *   W_out    (H,O), b_out (O)
 *   V0,a0,Z0 (B,H)    optional initial state, NULL = zeros (spiking_layers.py:69-83)
 * outputs
 *   V,a,Z    (B,T,H)  traces; required iff SNNK_F_TRACES (a only for ALIF)
 *   zbits    (B,T,H/32) uint32, bit l of word w = spike of neuron 32*w+l; always written
 *   y        (B,T,O)  readout trace; logits (B,O) = max_t y, tstar (B,O) int32 = first argmax_t
 *   workspace: >= snnk_forward_workspace_bytes(); on return its first B*T*H floats hold the input
 *   current I_in = x @ W_in (exposed for tests) -- unless run_table was given and its ok word is set: the
 *   projection then exists only for the first row of every run (compact rows further up in the workspace)
 *   run_table: table of x from snnk_encode_runs / snnk_frame_runs, or NULL (see there)
 *   W_effT_out: optional (H,H): receives the transpose of W_rec (.) rec_mask, which snnk_backward of the same
 *   weights accepts as W_effT_in and then need not prepare itself (one launch less on the training step)
 */
int snnk_forward(const SnnkDesc* d, const float* x, const float* W_in, const float* W_rec,
                 const float* rec_mask, const float* beta, const float* W_out, const float* b_out,
                 const float* V0, const float* a0, const float* Z0, float* V, float* a, float* Z,
                 uint32_t* zbits, float* y, float* logits, int32_t* tstar, void* workspace,
                 size_t workspace_bytes, const int32_t* run_table, float* W_effT_out,
                 snnk_stream_t stream);

/*
 * Fused head: log_softmax over the max-over-time logits (snn.py:258) + NLLLoss mean (snn.py:297)
 * and the gradient of that loss w.r.t. the logits.
 *   logits (B,O), labels (B) int64 -> logp (B,O), loss (1), g_logits (B,O) = (softmax - onehot)/B
 *   labels follow torch.nn.NLLLoss defaults: rows labelled -100 (ignore_index) are excluded from the mean (B becomes
 *   the number of valid rows) and get a zero gradient; any other label outside [0, O) makes the loss and that row's
 *   gradient NaN (torch raises a device-side assert there)
 *   loss_mailbox / mailbox_counter: both NULL, or: loss_mailbox is one 8-byte word of PINNED HOST memory (device-
 *   accessible under unified addressing) and mailbox_counter a zero-initialised device word.  Every launch then also
 *   stores ((++counter) << 32 | bits of loss) into the mailbox with a single store, so that the host can read the
 *   step's loss (SNN._exec_batch returns it as a Python float, snn.py:415) by polling for the launch number it
 *   expects -- no stream synchronisation, the backward pass may still be running.
 */
int snnk_head_nll(int32_t B, int32_t O, const float* logits, const int64_t* labels, float* logp,
                  float* loss, float* g_logits, uint64_t* loss_mailbox, uint32_t* mailbox_counter,
                  snnk_stream_t stream);

/*
 * snnk_forward followed by snnk_head_nll as ONE call (what SNN._exec_batch does for its default criterion,
 * snn.py:384-412: forward, max over time :228, log_softmax :258, NLLLoss :297).  Same arguments and results as the two
 * calls.  For layers on the register-resident recurrence kernel (H <= 128, batch below the tensor-core recurrence's
 * threshold) the head is evaluated in that kernel's tail -- the CTA that owns a row computes its log-probabilities, NLL
 * term and dL/dlogits, the last CTA to finish reduces the loss in the stand-alone kernel's order (bit-identical,
 * deterministic) -- so no launch sits between the forward pass and the BPTT sweep; other geometries launch
 * k_head_nll behind the forward kernels.
 *   head_ws  (B + 1) * 4 bytes of device memory, ZERO before the first call that uses it (the library leaves its last
 *            word, a ticket counter, zero again after every launch); must not be shared by launches that may overlap
 */
int snnk_forward_nll(const SnnkDesc* d, const float* x, const float* W_in, const float* W_rec,
                     const float* rec_mask, const float* beta, const float* W_out, const float* b_out,
                     const float* V0, const float* a0, const float* Z0, float* V, float* a, float* Z,
                     uint32_t* zbits, float* y, float* logits, int32_t* tstar, void* workspace,
                     size_t workspace_bytes, const int32_t* run_table, float* W_effT_out, const int64_t* labels,
                     float* logp, float* loss, float* g_logits, void* head_ws, uint64_t* loss_mailbox,
                     uint32_t* mailbox_counter, snnk_stream_t stream);

/*
 * Reverse-time BPTT.  Replaces autograd's sweep for batch_loss.backward() (snn.py:413) over the graph
 * built by the forward loop, with the surrogate derivatives of spike_funcs.py:59-62 / :75-79.
 * Gradient seeds: either g_y (B,T,O) dense w.r.t. the output trace, or -- the fused-head form --
 * g_logits (B,O) with tstar (B,O) (the gradient lands on y[b,tstar[b,o],o]), optionally multiplied by
 * the device scalar g_scale (dL/dloss handed in by autograd; NULL = 1).  Exactly one of the two forms
 * must be given.  g_V, g_Z (B,T,H) are optional extra seeds on the hidden traces.
 * V, a (ALIF), Z (B,T,H) and zbits are the traces the forward wrote (Z, the fp32 spike trace, is read by the
 * tensor-core weight-gradient GEMM only and may be NULL without SNNK_F_TENSOR_CORE).
 * With surrogate SNNK_SURROGATE_TRACE, `a` instead holds sigma'_t = dZ_t/dV_t (B,T,H), the surrogate derivative the
 * caller evaluated on the saved traces (threshold theta for LIF, theta + beta a_t for ALIF, v_peak for Izhikevich);
 * the sweep streams it where it would evaluate the built-in formula.  V may then be NULL for LIF / ALIF (the
 * derivative was its only use) and is required for Izhikevich (its membrane Jacobian reads V); beta is unused; a NULL
 * `a` is SNNK_ERR_ARG.
 * Outputs: dW_in (N,H), dW_rec (H,H, masked; NULL iff !recurrent), dW_out (H,O), db (O); they are
 * OVERWRITTEN.  beta receives no gradient (the threshold input of the spike function has none,
 * spike_funcs.py:62).  workspace: on return its first B*T*H floats hold gI, the gradient w.r.t. the
 * input current (exposed for tests); with SNNK_F_TENSOR_CORE gI is stored as two tf32 planes, high plane
 * first and the exact remainder in the next B*T*H floats (256-byte aligned), whose sum is gI.
 */
int snnk_backward(const SnnkDesc* d, const float* x, const float* W_rec, const float* rec_mask,
                  const float* beta, const float* W_out, const float* Z0, const float* V,
                  const float* a, const float* Z, const uint32_t* zbits, const float* g_y, const float* g_logits,
                  const int32_t* tstar, const float* g_scale, const float* g_V, const float* g_Z, float* dW_in,
                  float* dW_rec, float* dW_out, float* db, void* workspace, size_t workspace_bytes,
                  const int32_t* run_table, const float* W_effT_in,
                  snnk_stream_t stream);

/*
 * Optimizer step of SNN._exec_batch (snn.py:414) for the reference's default optimizer, Adam with L2 weight decay
 * (snn.py:299): torch.optim.Adam semantics (no amsgrad) over `count` <= 16 tensors in one launch.  params, grads,
 * exp_avg, exp_avg_sq, steps are HOST arrays of device pointers; steps[k] is the float32 device scalar torch keeps
 * per parameter when the optimizer is capturable (incremented here).  Graph-capturable.
 */
int snnk_adam_step(int32_t count, float* const* params, const float* const* grads, float* const* exp_avg,
                   float* const* exp_avg_sq, float* const* steps, const int64_t* numel, float lr, float beta1,
                   float beta2, float eps, float weight_decay, snnk_stream_t stream);

/*
 * Data-parallel form of snnk_adam_step (one process per GPU, batch rows sharded, weights replicated): the mean of
 * the weight gradients over the ranks -- the single exchange step of SNN._exec_batch's path (SURVEY.md 8e) -- and
 * the Adam update in ONE kernel over NVLink peer memory.  The thread owning a gradient element stores it, tagged
 * with the launch epoch in the same 8-byte word, into its rank's slot of every peer's exchange buffer, polls the
 * peers' slots of its own buffer until the tags match and sums the values in rank order, so all ranks compute
 * bit-identical means; grads[k] is overwritten with the mean (as after an all-reduce).
 *   peer_buffers: HOST array of `world` device pointers; entry r is rank r's exchange buffer as mapped into this
 *                 process (entry `rank` is the local one).  Each buffer holds snnk_adam_dp_buffer_bytes(world,
 *                 sum(numel)) bytes of peer-accessible memory, zero-filled on every rank before the first call.
 *   state:        16 zero-initialised uint32 in LOCAL device memory: [0] epoch and [2] grid counter (never reset
 *                 them), [3] timeout marker, [4..11] four uint64 %globaltimer stamps of the last launch as seen by
 *                 the first thread (start, stores issued, all peers seen, done) for measuring the exchange.
 * From 4 ranks on the exchange is two-phase over the same words and buffers: a value goes to the element's OWNER rank
 * only (contiguous slices of the flat gradient), the owner sums in rank order and stores the tagged mean into the slot
 * its own value would have had in every peer's buffer -- 1/world of the bytes, one more one-way trip, identical bits
 * on all ranks.  The environment variable SNNK_DP_RSAG = 0 / 1 (read at every call; it must be the same on all
 * ranks) forces the one-phase / two-phase form.
 * All ranks must issue the same sequence of calls.  Graph-capturable; a peer that never arrives traps the kernel
 * after 20 s (a sticky CUDA error) instead of hanging.
 */
int snnk_adam_dp_buffer_bytes(int32_t world, int64_t total_numel, size_t* bytes);
int snnk_adam_step_dp(int32_t count, float* const* params, float* const* grads, float* const* exp_avg,
                      float* const* exp_avg_sq, float* const* steps, const int64_t* numel, float lr, float beta1,
                      float beta2, float eps, float weight_decay, int32_t rank, int32_t world,
                      void* const* peer_buffers, uint32_t* state, snnk_stream_t stream);

/*
 * Gradient w.r.t. the layer input, for stacked hidden layers (snn.py:116-128): gX (B,T,N) = gI (B,T,H) @ W_in^T.
 * MmBackward of spiking_layers.py:163/233 w.r.t. `inputs`; layer l+1 hands gX down as the g_Z seed of layer l.
 * gI is the gradient w.r.t. the input current that snnk_backward leaves in its workspace (sum of the two tf32
 * planes in tensor-core mode).
 */
int snnk_input_grad(const SnnkDesc* d, const float* gI, const float* W_in, float* gX, snnk_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SNNK_H */
