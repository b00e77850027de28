/*
 * dsx -- C ABI of the B200-native DiffSinger reverse-diffusion sampler.
 *
 * The reference (MoonInTheRiver/DiffSinger) has no native boundary: the hot path is a Python
 * class surface (SURVEY.md section 8b).  This header is the boundary a binding would target;
 * each entry point names the reference interface it replaces (paths relative to the
 * reference tree).  Conventions:
 *   - plain pointers and sizes only; device pointers unless a parameter says "host";
 *   - every call returns 0 on success or a negative DSX_E_* code; dsx_last_error() gives a
 *     thread-local message; nothing throws across the ABI;
 *   - all GPU work is enqueued on the caller's stream (a cudaStream_t passed as void*);
 *     no internal threads; a handle belongs to one device and is not thread-safe;
 *   - the library owns only packed weights, step tables and workspace (freed by
 *     dsx_destroy); inputs are never modified except the documented in/out state.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with DSX_E_CUDA.
 */
#ifndef DSX_H_
#define DSX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSX_VERSION 100

enum {
  DSX_OK = 0,
  DSX_E_INVALID = -1,   /* bad argument / unsupported shape                      */
  DSX_E_CUDA = -2,      /* CUDA runtime / driver error (message has the string)  */
  DSX_E_STATE = -3,     /* call order: weights or schedule not loaded            */
  DSX_E_KERNEL = -4,    /* in-kernel watchdog or self-check tripped              */
  DSX_E_NOMEM = -5
};

/* Arithmetic of the contractions of each residual layer (usr/diff/net.py:66-78).  In the tcgen05 modes the conditioner
 * projection -- it does not depend on the diffusion step -- is computed once per call with hi+lo operands and kept in
 * fp32; the modes differ in the dilated conv and the output projection. */
enum {
  DSX_PREC_FP32_SIMT = 0, /* fp32 CUDA-core path, any channel count                          */
  DSX_PREC_FP16 = 1,      /* tcgen05 kind::f16, fp16 operands, fp32 accumulate (fast mode)   */
  DSX_PREC_FP16X2 = 2,    /* tcgen05, weights as hi+lo fp16 pairs, running activations fp16: 2 MMA passes;
                             max |d| ~2e-4 after 100 steps (default parity mode)                               */
  DSX_PREC_FP16X3 = 3,    /* tcgen05, hi+lo fp16 split of both operands, 3 MMAs (fp32-equivalent)*/
  DSX_PREC_FP16S = 4      /* tcgen05, ONE MMA pass; the weights are rounded to fp16 stochastically into R sets
                             (DSX_OPT_SR_SETS, default 64) and evaluation j of a sampling loop uses set j % R, so the weight
                             rounding error is unbiased and decorrelated across diffusion steps instead of accumulating:
                             max |d| ~3e-4 after 100 steps at half the MMA work of FP16X2 */
};

typedef struct dsx_handle dsx_handle;

/* Element strides of a logically [B, C, T] fp32 tensor (the reference hands the sampler
 * x[:,0] with strides (80T,1... or (80T,80,1,80)) and cond as a transposed view with strides
 * (256T,1,256); usr/diff/shallow_diffusion_tts.py:238,253-259). */
typedef struct {
  int64_t b, c, t;
} dsx_strides;

/* DiffNet parameters, fp32 device pointers, each tensor contiguous in the reference's own
 * state-dict layout (usr/diff/net.py:58-64, 91-104).  Per-layer arrays are HOST arrays of L
 * device pointers. */
typedef struct {
  const float* in_w;   /* input_projection.weight            [C, M, 1]  */
  const float* in_b;   /* input_projection.bias              [C]        */
  const float* mlp0_w; /* mlp.0.weight                       [4C, C]    */
  const float* mlp0_b; /* mlp.0.bias                         [4C]       */
  const float* mlp2_w; /* mlp.2.weight                       [C, 4C]    */
  const float* mlp2_b; /* mlp.2.bias                         [C]        */
  const float* const* dil_w;  /* residual_layers.l.dilated_conv.weight           [2C, C, 3] */
  const float* const* dil_b;  /* residual_layers.l.dilated_conv.bias             [2C]       */
  const float* const* dif_w;  /* residual_layers.l.diffusion_projection.weight   [C, C]     */
  const float* const* dif_b;  /* residual_layers.l.diffusion_projection.bias     [C]        */
  const float* const* cond_w; /* residual_layers.l.conditioner_projection.weight [2C, H, 1] */
  const float* const* cond_b; /* residual_layers.l.conditioner_projection.bias   [2C]       */
  const float* const* out_w;  /* residual_layers.l.output_projection.weight      [2C, C, 1] */
  const float* const* out_b;  /* residual_layers.l.output_projection.bias        [2C]       */
  const float* skip_w; /* skip_projection.weight             [C, C, 1]  */
  const float* skip_b; /* skip_projection.bias               [C]        */
  const float* fin_w;  /* output_projection.weight           [M, C, 1]  */
  const float* fin_b;  /* output_projection.bias             [M]        */
} dsx_diffnet_params;

/* Order of the schedule buffers for dsx_set_schedule == the registered buffers of
 * GaussianDiffusion.__init__ (usr/diff/shallow_diffusion_tts.py:101-123). */
enum {
  DSX_SCH_BETAS = 0,
  DSX_SCH_ALPHAS_CUMPROD,
  DSX_SCH_ALPHAS_CUMPROD_PREV,
  DSX_SCH_SQRT_ALPHAS_CUMPROD,
  DSX_SCH_SQRT_ONE_MINUS_ALPHAS_CUMPROD,
  DSX_SCH_LOG_ONE_MINUS_ALPHAS_CUMPROD,
  DSX_SCH_SQRT_RECIP_ALPHAS_CUMPROD,
  DSX_SCH_SQRT_RECIPM1_ALPHAS_CUMPROD,
  DSX_SCH_POSTERIOR_VARIANCE,
  DSX_SCH_POSTERIOR_LOG_VARIANCE_CLIPPED,
  DSX_SCH_POSTERIOR_MEAN_COEF1,
  DSX_SCH_POSTERIOR_MEAN_COEF2,
  DSX_SCH_COUNT
};

int dsx_version(void);
const char* dsx_last_error(void);

/* Handle: owns packed weights + workspace on `device`. */
int dsx_create(int device, dsx_handle** out);
void dsx_destroy(dsx_handle* h);

/* Replaces: DiffNet.__init__ / load_state_dict (usr/diff/net.py:82-105; checkpoint keys
 * model.denoise_fn.*, utils/__init__.py:178-203).  (Re)packs the weights for the selected
 * precision; call again after every load_state_dict / .to().  M mel bins, C residual
 * channels, H conditioner channels, L layers, dilation 2^(l % cycle). */
int dsx_load_diffnet(dsx_handle* h, const dsx_diffnet_params* p, int M, int C, int H, int L,
                     int dilation_cycle, int precision, void* stream);

/* Replaces: the schedule buffers registered in GaussianDiffusion.__init__
 * (usr/diff/shallow_diffusion_tts.py:90-123).  bufs: HOST array of DSX_SCH_COUNT HOST
 * pointers to fp32[T] -- the module's buffers verbatim, never recomputed from hparams. */
int dsx_set_schedule(dsx_handle* h, const float* const* bufs, int T);

/* Replaces: DiffNet.forward(spec, diffusion_step, cond) (usr/diff/net.py:107-130).
 * x: [B,1,M,T] addressed through xs (b, c=mel bin, t); t: device int64[B];
 * cond: [B,H,T] through cs; eps out: contiguous [B,1,M,T]. */
int dsx_diffnet_forward(dsx_handle* h, const float* x, dsx_strides xs, const int64_t* t,
                        const float* cond, dsx_strides cs, float* eps, int B, int T, void* stream);

/* Conditioner of the following calls: packs cond [B,H,T] (any strides) and computes the step-independent
 * conditioner_projection of every residual layer (usr/diff/net.py:56,70) once.  Every entry point below that takes `cond`
 * does the same when the pointer is non-NULL and accepts cond == NULL to re-use the conditioner already set for the same
 * (B, T) -- for callers that drive the sampling loop themselves, one p_sample / p_sample_plms / DiffNet.forward per call
 * (usr/diff/shallow_diffusion_tts.py:159-204), so that the pack + projection are paid once per batch, not once per step. */
int dsx_set_cond(dsx_handle* h, const float* cond, dsx_strides cs, int B, int T, void* stream);

/* Replaces: the linear-multistep combination + get_x_pred of ONE p_sample_plms step
 * (usr/diff/shallow_diffusion_tts.py:174-199), fp32 in the reference's operation order, for callers that keep the eps
 * history themselves (self.noise_list).  eps: HOST array of device pointers, most recent first; all tensors contiguous
 * [B,1,M,T].  mode 0: x_out = phi(x_in, eps[0], t) (the warm-up prediction); 1: eps' = (eps[0] + eps[1]) / 2;
 * 2: (3 e0 - e1) / 2; 3: (23 e0 - 16 e1 + 5 e2) / 12; 4: (55 e0 - 59 e1 + 37 e2 - 9 e3) / 24; then x_out = phi(x_in, eps', t). */
int dsx_plms_update(dsx_handle* h, float* x_out, const float* x_in, const float* const* eps, int mode, int t,
                    int interval, int B, int T, void* stream);

/* Replaces: the DDPM loop `for i in reversed(range(0, t)): x = p_sample(x, i, cond)`
 * (usr/diff/shallow_diffusion_tts.py:159-166, 269-270): n_steps steps t_start-1 ... t_start-n_steps.
 * x_inout: contiguous [B,1,M,T], overwritten with the result.  noise: contiguous
 * [n_steps,B,1,M,T] consumed in execution order (noise[j] at t = t_start-1-j), or NULL
 * for the in-kernel Philox4x32-10 generator seeded by `seed`. */
int dsx_sample_ddpm(dsx_handle* h, float* x_inout, const float* cond, dsx_strides cs, int B, int T,
                    int t_start, int n_steps, const float* noise, uint64_t seed, void* stream);

/* Replaces: the PNDM loop `for i in reversed(range(0, t, interval)): x = p_sample_plms(...)`
 * (usr/diff/shallow_diffusion_tts.py:168-204, 261-267), history owned by the call. */
int dsx_sample_plms(dsx_handle* h, float* x_inout, const float* cond, dsx_strides cs, int B, int T,
                    int t_start, int interval, void* stream);

/* Replaces: the infer branch of GaussianDiffusion.forward after self.fs2
 * (usr/diff/shallow_diffusion_tts.py:248-275): norm_spec + q_sample(K_step-1) prologue (or a
 * gaussian start when fs2_mel == NULL and x_start != NULL), the sampling loop, and the
 * transpose + denorm_spec + (mel2ph > 0) mask epilogue.
 *   fs2_mel [B,T,M] contiguous (or NULL), start_noise [B,1,M,T] (or NULL -> Philox),
 *   x_start [B,1,M,T] (gaussian start; may be NULL), step_noise as in dsx_sample_ddpm,
 *   mel2ph device int64 [B,T] or NULL, spec_min/spec_max device fp32 [M],
 *   pndm_interval 0 = DDPM.  mel_out [B,T,M] contiguous. */
int dsx_infer(dsx_handle* h, const float* cond, dsx_strides cs, const float* fs2_mel,
              const float* start_noise, const float* x_start, const float* step_noise, uint64_t seed,
              const int64_t* mel2ph, const float* spec_min, const float* spec_max, int B, int T,
              int K_step, int pndm_interval, float* mel_out, void* stream);

/* Same as dsx_infer but every tensor pointer is a HOST pointer (pinned or pageable); the
 * copies to and from the device are issued on `stream` inside the call and the call returns
 * after mel_out_host is complete (it synchronises the stream). */
int dsx_infer_host(dsx_handle* h, const float* cond_host, dsx_strides cs, const float* fs2_mel_host,
                   const float* x_start_host, uint64_t seed, const int64_t* mel2ph_host,
                   const float* spec_min_host, const float* spec_max_host, int B, int T, int K_step,
                   int pndm_interval, float* mel_out_host, void* stream);

/* Introspection for tests / bench. */
int dsx_get_info(dsx_handle* h, int what, int64_t* out);
enum {
  DSX_INFO_PRECISION = 0,
  DSX_INFO_KERNEL_LAUNCHES = 1, /* kernels launched by this handle so far               */
  DSX_INFO_WORKSPACE_BYTES = 2,
  DSX_INFO_SM_COUNT = 3,
  DSX_INFO_TC_CTA_GROUP = 4,    /* 1 or 2: cta_group of the tcgen05 path in use          */
  DSX_INFO_LAYER_KERNEL_NS = 5, /* DSX_OPT_PROFILE: summed device time of the residual-layer kernels since the
                                   option was set (CUDA events on the launching stream; synchronises)     */
  DSX_INFO_LAYER_KERNEL_LAUNCHES = 6, /* number of (start, stop) brackets = evaluations profiled */
  DSX_INFO_STACK_MODE = 7,
  DSX_INFO_CLUSTER_OCCUPANCY = 8, /* co-resident CTA pairs of the layer kernel reported by the driver */
  DSX_INFO_STACK_KERNEL_LAUNCHES = 9, /* launches of the register-resident stack kernel (dsx_stack.cu) so far */
  DSX_INFO_STACK_ROWS = 10 /* frames per CTA of the last stack-kernel launch: 128, or 64 for small batches */
};
/* Tuning knobs (tests exercise every variant): */
int dsx_set_option(dsx_handle* h, int what, int64_t value);
enum {
  DSX_OPT_TC_CTA_GROUP = 0, /* 2 (the layer kernel pairs CTAs; kept for forward compatibility) */
  DSX_OPT_CP_PREFETCH = 1,  /* tuning knob, results do not depend on it: 1 = the layer kernel's activation producer streams the
                               hoisted conditioner projection HBM -> L2 half a layer ahead of the gate epilogue */
  DSX_OPT_PROFILE = 2,      /* 1: bracket the residual-layer kernel(s) of every evaluation with CUDA events; 2: bracket the
                               head / update kernel(s) of every evaluation instead (the head then runs as a launch of its
                               own); 0: off.  Setting it resets the sums */
  DSX_OPT_STACK_MODE = 3,   /* 1 (default): all residual layers of an evaluation in ONE persistent launch whenever every
                               128-frame tile can own an SM at once (tiles <= co-resident CTAs); 0: one launch per layer */
  DSX_OPT_STACK_KERNEL = 4, /* 1 (default): the register-resident stack kernel (residual stream in registers, conv input in
                               shared memory, skip sum in tensor memory) for FP16 / FP16X2 / FP16S; 0: the round-1 layer kernel */
  DSX_OPT_SR_SETS = 5,      /* number of stochastically rounded weight sets of DSX_PREC_FP16S; set before dsx_load_diffnet */
  DSX_OPT_GATE_APPROX = 7,  /* stack kernel: gate sigmoid(g) * tanh(f) with tanh.approx.f32 (1) or with ex2 / rcp to ~2e-7 (0);
                               -1 (default) = 1: its 2^-11 relative error is below the fp16 rounding of the gate output that
                               follows (K = 100 golden loop: 3.3e-4 either way in FP16S, 1.5e-4 / 1.6e-4 in FP16X2) */
  DSX_OPT_FUSED_HEAD = 9,   /* 1 (default): the skip / output projections, the sampler update and the next input projection run
                               inside the stack kernel's launch (one kernel per diffusion step); 0: separate head kernel */
  DSX_OPT_STACK_ROWS = 8,   /* stack kernel: frames per CTA.  0 (default) = 64 whenever the whole batch then fits the machine at once
                               (small batches: twice the CTAs, about half the time per layer), else 128; 64 / 128 force it */
  DSX_OPT_BATCH_OFFSET = 6  /* global index of this call's utterance 0: the in-kernel Philox noise of utterance b is drawn for
                               index (offset + b), so a batch sharded over ranks (one seed) reproduces the unsharded noise */
};

/* Debug taps for layer-by-layer parity (tests only): copies internal fp32 frames-major
 * buffers after a dsx_diffnet_forward.  which: 0 = residual stream after the last layer
 * executed, 1 = skip sum.  out: [B, T, C] contiguous. */
int dsx_debug_read(dsx_handle* h, int which, float* out, int B, int T, void* stream);
/* Debug timeline of the residual-layer kernel: enable != 0 makes CTAs 0 and 1 of every following layer
 * launch record clock64 stamps ([2][3 roles: producer, MMA issuer, epilogue][256] int64); out_host (may be
 * NULL) receives the current buffer contents (6*256 int64) after synchronising the device.  enable == 2: out_host
 * receives 10*256 int64, the extra [256][4] being per-CTA {globaltimer ns, clock64} at kernel entry and exit. */
int dsx_debug_trace(dsx_handle* h, int enable, int64_t* out_host);
/* Run only layers [0, n_layers) in the next dsx_diffnet_forward calls (<0: all). */
int dsx_debug_set_layer_limit(dsx_handle* h, int n_layers);

/* Hardware self-tests of the tcgen05 / TMA encodings this library relies on (one small
 * launch each, results checked on the host).  which = -1 runs all; returns 0 when every
 * selected test passes, otherwise DSX_E_KERNEL with the failing names in dsx_last_error().
 * which = 0 / 1: UMMA + TMA round trip with cta_group::1 / ::2; 2 = row-shifted SWIZZLE_128B operand descriptors (the
 * dilated taps rely on them); 3 = TMA ingest micro-benchmark (informational, only in -DDSX_EXPERIMENTS builds, not part of -1).
 * report (may be NULL): host buffer receiving a text report. */
int dsx_selftest(int device, int which, char* report, int report_bytes);

#ifdef __cplusplus
}
#endif
#endif /* DSX_H_ */
