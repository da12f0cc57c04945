/*
 * ntm_b200.h -- C ABI of the B200-native engine for the recurrent forward pass of
 * 01tot10/neural-tape-modeling (GRU-HS[64] + Linear head, optional time-varying delay line).
 *
 * The reference has no FFI of its own for this path: its boundary is the Python torch.nn.Module API in
 * code/model.py.  Each entry point below names the reference method whose arithmetic it replaces; the
 * Python classes in neural-tape-modeling_b200/model.py (same names/signatures as code/model.py) call
 * exactly these symbols through ctypes (see INTEGRATION.md for the binding a reference maintainer adds).
 *
 * Conventions
 *   - Plain pointers and sizes only.  Unless a name ends in _host, data pointers are DEVICE pointers on the
 *     handle's device and `stream` is a cudaStream_t (NULL = legacy default stream).  Launches are
 *     asynchronous; nothing here synchronises unless stated.
 *   - Audio tensors are the reference's (B, 1, T) float32 layout: row b starts at ptr + b*ld, ld >= T.
 *   - Return value: 0 (NTM_OK) or a negative NTM_E* code; never throws, never aborts.  After NTM_ECUDA,
 *     ntm_last_cuda_error() returns the cudaError_t of the calling thread's last failure.
 *   - Caller owns every buffer passed in; the engine owns only the handle (prepare/destroy) and the
 *     staging buffers of the *_host entry points (allocated on first use, freed by ntm_destroy).
 */
#ifndef NTM_B200_H
#define NTM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define NTM_API_VERSION 2

/* error codes */
#define NTM_OK            0
#define NTM_EINVAL       (-1)   /* bad argument (null pointer, negative size, ld < T, ...) */
#define NTM_EUNSUPPORTED (-2)   /* hidden size / mode not built into this library */
#define NTM_ENOMEM       (-3)
#define NTM_ECUDA        (-4)   /* a CUDA runtime call failed: see ntm_last_cuda_error() */
#define NTM_EDELAY       (-5)   /* a delay value exceeds the history length D (the reference's assert,
                                   code/model.py:283) -- only returned by ntm_delay_check */
#define NTM_ENODEVICE    (-6)   /* no CUDA device / not an sm_100 device */
#define NTM_ECLOSED      (-7)   /* real-time stream: the resident kernel has left (closed or idle timeout) */

/* arithmetic modes of the hidden-to-hidden contraction (gates, state and head are always fp32) */
#define NTM_MODE_FP32     0     /* fp32 FFMA on CUDA cores, libm-grade activations: the parity anchor */
#define NTM_MODE_TF32     1     /* tensor cores, tf32 operands, fp32 accumulate */
#define NTM_MODE_BF16     2     /* tensor cores, bf16 operands, fp32 accumulate (opt-in, lower accuracy) */
#define NTM_MODE_F16X3    3     /* STRICT tensor-core mode, fp32-grade result (max-abs <= 1e-5 vs the reference, like
                                   NTM_MODE_FP32): every operand is an f16 pair hi + lo'/2^11, three MMAs per product
                                   (W_hi h_hi + W_hi h_lo + W_lo h_hi), fp32 accumulate -- the 3xTF32 scheme at half
                                   the MMA count */
#define NTM_MODE_TF32X3   NTM_MODE_F16X3   /* the name SURVEY.md section 8b reserved for the strict mode */
#define NTM_MODE_F16      4     /* tensor cores, f16 operands (11-bit significand like tf32, half the MMAs), fp32 acc. */

/* ntm_query selectors */
#define NTM_Q_VERSION        0
#define NTM_Q_DEVICE_COUNT   1
#define NTM_Q_SM_COUNT       2   /* of the current device */
#define NTM_Q_MODE_MASK      3   /* bit m set <=> mode m is implemented */
#define NTM_Q_KERNEL_LAUNCHES 4  /* number of engine kernels launched by this process so far */
#define NTM_Q_LAST_KERNEL    5   /* recurrent kernel of the process's last launch: 0 fp32 CUDA-core, 1 warp-level
                                    mma.sync (general form), 3 stream-major tcgen05, 4 warp-level mma.sync, lean 4-stream
                                    form (gru_mma4_kernel) (per handle: ntm_handle_last_kernel) */

int         ntm_query(int what);
const char* ntm_strerror(int code);
int         ntm_last_cuda_error(void);

/*
 * Pack one model's parameters (HOST pointers, PyTorch layouts, gate row order r,z,n) into an engine-owned
 * device blob on `device`.   Replaces: RNN.__init__/load_state_dict parameter ownership, code/model.py:44-45
 * (b_out != NULL) and DiffDelRNN, code/model.py:364-365 (b_out == NULL).
 *   w_ih (3H,1)  w_hh (3H,H)  b_ih (3H)  b_hh (3H)  w_out (1,H)  b_out (1) or NULL.   1 <= H <= 64 (NTM_EUNSUPPORTED beyond).
 * The engine's state is 64 units wide whatever H is: every `h` / `h_in` / `h_out` of this header is B x 64 floats.  A model
 * with H < 64 (code/train.py:50 defaults to 16, scripts/sbatch-train.sh:15 trains 32) is embedded with zero weights for the
 * units H .. 63; their state stays 0 and never reaches a real unit or the output, so the result is the H-unit GRU's exactly.
 * Callers keep columns H .. 63 of the state zero (the Python classes pad / cut `self.hidden`).
 */
int  ntm_gru_prepare(const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh,
                     const float* w_out, const float* b_out, int H, int device, void** handle);
/* Handles are reference counted: ntm_gru_prepare returns one reference, ntm_retain adds one, ntm_release (alias
 * ntm_destroy) drops one and frees the device blob with the last.  An open real-time stream holds a reference, so
 * releasing the model's handle under a live stream is safe. */
int  ntm_retain(void* handle);
void ntm_release(void* handle);
void ntm_destroy(void* handle);

/*
 * y = head(GRU(x, h_in)); h_out receives the final state.
 * Replaces: RNN.forward, code/model.py:67-88  (`self.GRU(x, self.hidden)` + `self.output(x)` [+ skip]).
 *   x (B rows, ld ldx)  y (B rows, ld ldy)  h_in (B x 64 contiguous, NULL = zero state, the reference's
 *   `hidden = None`, code/model.py:50-52)  h_out (B x 64; may alias h_in).  T == 0 copies h_in to h_out.
 */
int ntm_gru_forward(void* handle, int mode, const float* x, int64_t ldx, float* y, int64_t ldy,
                    const float* h_in, float* h_out, int64_t B, int64_t T, int skip, void* stream);

/*
 * pre_d = head(GRU(x, h));  y = delay(pre_d, d)  in ONE kernel (delay read fused after the GRU output).
 * Replaces: DiffDelRNN.forward, code/model.py:393-424 (GRU + Linear(bias=False) + self.diffdel).
 *   d: delay in samples per output sample.  hist_in / hist_out: (B x D) carried delay history
 *   (TimeVaryingDelayLine.buffer, code/model.py:267,314-315); hist_out must not alias hist_in.
 *   warmup != 0: y = pre_d, history still rolled (code/model.py:288-292).
 */
int ntm_diffdel_forward(void* handle, int mode, const float* x, int64_t ldx, const float* d, int64_t ldd,
                        float* y, int64_t ldy, float* pre_d, int64_t ldp, const float* h_in, float* h_out,
                        const float* hist_in, float* hist_out,
                        int64_t B, int64_t T, int64_t D, int warmup, int skip, void* stream);

/*
 * Stand-alone time-varying fractional delay line.
 * Replaces: TimeVaryingDelayLine.forward, code/model.py:269-320 (used alone by apply_delay,
 * code/test-model.py:259-290).  Same argument meaning as above; x may not alias y.
 */
int ntm_delay_forward(const float* x, int64_t ldx, const float* d, int64_t ldd, float* y, int64_t ldy,
                      const float* hist_in, float* hist_out, int64_t B, int64_t T, int64_t D,
                      int warmup, int device, void* stream);

/* The reference's `assert self.max_delay >= torch.max(dt)` (code/model.py:283).  SYNCHRONISES the stream.
 * Returns NTM_EDELAY if any d[b][t] > D. */
int ntm_delay_check(const float* d, int64_t ldd, int64_t B, int64_t T, int64_t D, int device, void* stream);

/*
 * Real-time block mode with a RESIDENT kernel (BASELINE cfg 5: consecutive RNN.forward calls on short blocks with the
 * state carried, code/model.py:67-88 with self.hidden kept).  ntm_rt_open launches one persistent CTA that keeps the
 * weights, the hidden state and its staging on chip and waits on a page-locked mailbox; ntm_rt_process hands it one block
 * (x_host: B x block_len contiguous HOST floats) and returns when y_host is filled -- two PCIe round trips per block
 * instead of a kernel launch, a prologue and a stream synchronisation.  ntm_rt_close stops the kernel and returns the
 * final state.  B <= 4 streams, block_len <= 256, tensor-core modes only (NTM_EUNSUPPORTED for NTM_MODE_FP32).
 * h_host: B x 64 initial state or NULL (zeros).  The kernel leaves by itself after idle_timeout_ms without a block
 * (ntm_rt_process then returns NTM_ECLOSED).  While a stream is open, do NOT synchronise the whole device
 * (cudaDeviceSynchronize, cudaFree): the resident kernel only ends at close / idle timeout.  One thread per stream.
 */
int ntm_rt_open(void* handle, int mode, const float* h_host, int64_t B, int64_t block_len, int skip,
                int idle_timeout_ms, void** rt);
int ntm_rt_process(void* rt, const float* x_host, float* y_host);
int ntm_rt_close(void* rt, float* h_host_out);

/*
 * Evaluation losses on the device (the step right after the recurrent path, code/test-model.py:250-253,386-388).
 * Replaces: ESRLoss, code/Automated_GuitarAmpModelling/CoreAudioML/training.py:5-16 (dc_pre == 0) and
 * ESRLoss(dc_pre=True) = DC_PreEmph + ESR, code/GreyBoxDRC/loss_funcs.py:6-52 (dc_pre != 0: 2000-tap truncation of
 * (1 - z^-1)/(1 - 0.995 z^-1) applied to both signals, zero-padded in front).
 *   out, target: B rows of T samples (row strides ldo, ldt), the reference's (B,1,T) tensors.
 *   sums (DEVICE, 2 doubles, written asynchronously): sum (f(t)-f(o))^2 and sum f(t)^2 over all B*T samples;
 *   loss = (sums[0]/(B*T)) / (sums[1]/(B*T) + 1e-5).
 */
int ntm_esr_sums(const float* out, int64_t ldo, const float* target, int64_t ldt, int64_t B, int64_t T,
                 int dc_pre, double* sums, int device, void* stream);

/*
 * Whole-signal prediction from HOST buffers (page-locked for full speed): time-chunked H2D copy, kernel and
 * D2H copy pipelined on the engine's own streams.  Replaces the loop of RNN.predict, code/model.py:218-246
 * (host->device at code/test-model.py:427-433, device->host at :525).  SYNCHRONOUS.
 *   x_host, y_host: B x T contiguous.  h_host: B x 64 in-out (initial state in, final state out).
 *   chunk_T: samples per pipelined chunk (0 = engine default).
 */
int ntm_gru_predict_host(void* handle, int mode, const float* x_host, float* y_host, float* h_host,
                         int64_t B, int64_t T, int skip, int64_t chunk_T);

/*
 * The same with a 16-BIT HOST TRANSPORT (opt-in; no counterpart in the reference, whose audio is float32 end to end):
 * x_host_f16 / y_host_f16 hold IEEE binary16 samples (B x T contiguous), cross the host link as such -- half the bytes per
 * sample, which is what bounds the end-to-end rate once several GPUs share one host (DESIGN.md section 5) -- and are widened
 * / narrowed on the device around the same fp32 kernels.  State in / out stays float32.  Cost in accuracy: the quantisation
 * of the input and of the output to 11 significant bits (ESR ~1e-7 against the float32 transport, tests/test_host_f16_gpu.py).
 */
int ntm_gru_predict_host_f16(void* handle, int mode, const void* x_host_f16, void* y_host_f16, float* h_host,
                             int64_t B, int64_t T, int skip, int64_t chunk_T);

/* DiffDelRNN.predict (code/model.py:618-653) from HOST buffers; hist_host: B x D in-out. */
int ntm_diffdel_predict_host(void* handle, int mode, const float* x_host, const float* d_host,
                             float* y_host, float* pre_d_host, float* h_host, float* hist_host,
                             int64_t B, int64_t T, int64_t D, int skip, int64_t chunk_T);

/* Per-row variant: sums is DEVICE memory for B x 2 doubles; row b is evaluated over its own window of samples
 * [first[b], first[b] + count[b]) (DEVICE int64 arrays of B values; NULL = 0 / T), clipped to the row -- ragged batches and
 * the reference's INIT_LEN cut (code/test-model.py:323-325,367-370: the DC filter starts from zero state at the cut) in
 * ONE launch.  loss_b = (sums[b][0]/n_b) / (sums[b][1]/n_b + 1e-5). */
int ntm_esr_sums_rows(const float* out, int64_t ldo, const float* target, int64_t ldt, int64_t B, int64_t T,
                      const int64_t* first, const int64_t* count, int dc_pre, double* sums, int device, void* stream);

/* Kernel-selection knob for tests and benchmarks.  The pair (streams_per_cta, ksplit) means, by mode:
 *   mode          pair                        runs
 *   any           (0, 0)                      automatic dispatch
 *   fp32          (s, ks), s in {0,1,2,4,8},  CUDA-core kernel, s streams per CTA, ks k-slices per hidden unit
 *                 ks in {0,2,4}; ks = 2 only  (0 = automatic)
 *                 with s = 1 or 2
 *   tensor-core   (4, 3), (8, 3)              general warp-level mma.sync kernel, 4 or 8 streams per CTA
 *   tensor-core   (4, 6)                      lean 4-stream mma.sync kernel (tf32 has no lean form: the general kernel with
 *                                             automatic streams per CTA)
 *   tensor-core   (t, 4), t in {1, 2}         stream-major tcgen05 kernel, t 128-stream tiles per CTA
 *   tensor-core   (t + 4, 4)                  the same with the static schedule (one CTA per tile group, no job queue)
 * Any other pair makes the launch return NTM_EINVAL.  ntm_set_tuning sets the process-wide default (one atomic word, safe
 * to call concurrently with launches); ntm_handle_set_tuning overrides it for one handle (streams_per_cta = -1: follow the
 * default again).  ntm_handle_last_kernel: NTM_Q_LAST_KERNEL of that handle's last launch. */
int ntm_set_tuning(int streams_per_cta, int ksplit);
int ntm_handle_set_tuning(void* handle, int streams_per_cta, int ksplit);
int ntm_handle_last_kernel(void* handle);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* NTM_B200_H */
