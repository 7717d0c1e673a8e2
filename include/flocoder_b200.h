/*
 * flocoder_b200 -- C ABI of the B200 (sm_100a) latent flow-matching sampling path.
 *
 * This is the drop-in boundary for ONE hot path of drscotthawley/flocoder:
 *   - the velocity field  Unet.forward(x, time, cond)          flocoder/unet.py:289-377
 *   - the fixed-step ODE loop rk4_step / v_func_cfg /
 *     generate_latents_rk4 / generate_latents                   flocoder/sampling.py:36-146
 *   - the legacy Euler sampler                                   legacy/train_sd_flowers.py:50-67
 *
 * The reference has no FFI of its own (it is pure Python/PyTorch); these entry points are
 * what a ctypes/cffi binding for that path binds (see INTEGRATION.md).  Plain pointers and
 * sizes only -- no torch types.  Unless stated otherwise pointers are DEVICE pointers on the
 * handle's device, calls are asynchronous on `stream` (a cudaStream_t passed as void*), do no
 * host synchronisation, and return FLO_OK (0) or a negative flo_status; the message for the
 * last failure on the calling thread is flo_last_error().  There is no CPU fallback.
 *
 * A handle is bound to one device and is not re-entrant: its stage table, control block and per-batch
 * workspaces are shared by all calls, so it serves ONE stream and ONE host thread at a time.  A call on a
 * different stream than the previous call first waits (cudaStreamSynchronize) for the previous stream, so
 * switching streams is safe but serialises; concurrent calls from two host threads are not supported --
 * create one handle per stream / thread (weights are ~5 MB).  At most 8 per-batch-size plans (workspace +
 * CUDA graphs) are cached per handle; the least recently used one is released when a ninth size arrives.
 * class_ids must lie in [0, n_classes): the kernels clamp out-of-range ids instead of faulting, and the
 * Python boundary raises IndexError for them as nn.Embedding does (unet.py:207).
 */
#ifndef FLOCODER_B200_H
#define FLOCODER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FLO_VERSION 100 /* 0.1.0 */

#if defined(__GNUC__)
#define FLO_API __attribute__((visibility("default")))
#else
#define FLO_API
#endif

typedef enum flo_status {
    FLO_OK = 0,
    FLO_ERR_INVALID = -1,     /* bad argument (ValueError in Python) */
    FLO_ERR_UNSUPPORTED = -2, /* feature outside the built path, e.g. mask_cond with FLO_F16, or with FLO_BF16 without
                                 FLO_FLAG_LAYERWISE (NotImplementedError) */
    FLO_ERR_CUDA = -3,        /* CUDA runtime / driver failure (RuntimeError) */
    FLO_ERR_NOMEM = -4,
    FLO_ERR_STEP = -5         /* adaptive integrator: step size below the minimum step, or max_steps used up (RuntimeError) */
} flo_status;

typedef enum flo_dtype { FLO_F32 = 0, FLO_BF16 = 1, FLO_F16 = 2 } flo_dtype;

/* Integrators.  Stage times are formed in fp32 exactly as the reference forms them on 0-d
 * tensors (sampling.py:44-47,117): dt = ts[i+1]-ts[i];  t, t+dt/2, t+dt;  time fed to the
 * U-Net is fl32(t)*t_scale (sampling.py:63).  The grid of FLO_RK4 / FLO_EULER_GRID need not be ascending: over a
 * descending grid every dt is negative and the call integrates backwards in time (e.g. from data at t = 1 back to
 * noise at t = 0, the inversion of a sampled trajectory). */
typedef enum flo_method {
    FLO_RK4 = 0,          /* ts = time grid with n_ts points -> n_ts-1 classic RK4 intervals (sampling.py:37-48) */
    FLO_EULER_LEGACY = 1, /* ts = the n_ts evaluation times t_i, fixed dt: x += v(x, t_i*t_scale)*dt
                             (legacy/train_sd_flowers.py:58-64) */
    FLO_EULER_GRID = 2    /* ts = time grid with n_ts points; forward Euler with dt_i = ts[i+1]-ts[i] */
} flo_method;

enum {
    FLO_FLAG_NO_BUFFER_REUSE = 1, /* debug: every op output keeps its own buffer (flo_unet_read_activation) */
    FLO_FLAG_NO_GRAPH = 2,        /* debug: launch kernels directly instead of replaying a CUDA graph */
    FLO_FLAG_LAYERWISE = 4        /* 16-bit paths: one kernel per layer (139 launches/forward) instead of the fused
                                     stage kernels; the reference point the fused path is validated against */
};

/* Constructor arguments of flocoder.unet.Unet (unet.py:165-175) + latent size + compute type. */
typedef struct flo_unet_cfg {
    int32_t dim;           /* Unet(dim=...)                         */
    int32_t channels;      /* latent channels C                     */
    int32_t n_mults;       /* len(dim_mults), 1..8                  */
    int32_t mults[8];      /* dim_mults                             */
    int32_t groups;        /* resnet_block_groups                   */
    int32_t n_classes;     /* 0 = no class_cond_mlp                 */
    int32_t height, width; /* latent H, W                           */
    int32_t compute_dtype; /* flo_dtype: FLO_F32 = fp32 CUDA-core path (<=1e-5 parity),
                              FLO_BF16 / FLO_F16 = 16-bit tcgen05 operands, fp32 accumulate */
    int32_t mask_cond;     /* Unet(mask_cond=...): 1 builds the inpainting U-Net with its mask-fusion branches
                              (unet.py:214-235); FLO_F32, or FLO_BF16 with FLO_FLAG_LAYERWISE and dim % 16 == 0
                              (the fused stage kernels have no mask branches) */
    int32_t flags;         /* FLO_FLAG_*                            */
    int32_t device;        /* CUDA device ordinal                   */
} flo_unet_cfg;

typedef struct flo_unet flo_unet_t;

FLO_API int flo_version(void);
FLO_API const char* flo_last_error(void);

/* Parameter manifest: the tensors of the reference state_dict, in state_dict order
 * (SURVEY.md section 8a; e.g. "downs.0.2.fn.fn.to_qkv.weight").  Shapes are the reference's
 * (OIHW conv weights, [out,in] linear weights). */
FLO_API int flo_param_count(const flo_unet_cfg* cfg);
FLO_API int flo_param_info(const flo_unet_cfg* cfg, int index, char* name, int name_cap, int64_t shape[4], int* ndim);

/* Build a handle from fp32 device tensors given in manifest order; packs them into the
 * kernels' layouts (replaces Unet.__init__ + load_state_dict, unet.py:165-286). */
FLO_API int flo_unet_create(flo_unet_t** out, const flo_unet_cfg* cfg, const void* const* params, int n_params,
                    void* stream);
FLO_API int flo_unet_destroy(flo_unet_t* h);

/* Optional: overwrite the dim/2 sinusoidal-embedding frequencies exp(-j*ln(1e4)/(dim/2-1))
 * (unet.py:26-27) with host values computed by the caller's own exp(), so the table is bit-identical
 * to the reference's torch.exp; the built-in default is the correctly rounded value. */
FLO_API int flo_unet_set_time_freqs(flo_unet_t* h, const float* freqs_host, int n);

/* Bytes of activation workspace the handle holds for batch size B. */
FLO_API size_t flo_workspace_bytes(flo_unet_t* h, int B);

/* v = Unet.forward(x, time, cond)  (unet.py:374-377).
 * x, v: [B,C,H,W] fp32 NCHW;  time: [B] fp32, already multiplied by t_scale;
 * class_ids: [B] int64 or NULL (cond['class_cond'], unet.py:315-316). */
FLO_API int flo_unet_forward(flo_unet_t* h, const float* x, const float* time, const int64_t* class_ids, float* v,
                     int B, void* stream);

/* cond['mask_cond'] for every following flo_unet_forward / flo_integrate call at batch size B (unet.py:298-305,
 * 336-340,360-364).  mask: [B,C,H,W] fp32 NCHW (latent-shaped, as MaskEncoder produces it, inpainting.py:180-245) or
 * NULL = no mask (every mask branch is skipped, as when key_usable(cond,'mask_cond') is false).  The call resizes the
 * mask to every resolution level (F.interpolate bilinear) and evaluates the reference's all-ones bypass
 * (torch.allclose(mask, 1), unet.py:301) on the device; no host synchronisation.  The state is per batch size and
 * persists until the next call.  Handles built with mask_cond=0 accept only NULL. */
FLO_API int flo_unet_set_mask(flo_unet_t* h, const float* mask, int B, void* stream);

/* Whole trajectory on the device, no host synchronisation (replaces the loop of
 * generate_latents_rk4, sampling.py:116-117, with v_func_cfg, sampling.py:51-76, inside).
 * y: [B,C,H,W] fp32, in = start point, out = final latents.
 * ts: HOST array of n_ts fp32 times (see flo_method).  dt: step for FLO_EULER_LEGACY, else ignored.
 * class_ids: [B] int64 device or NULL.  cfg_strength: classifier-free guidance; if class_ids
 *   != NULL and cfg_strength != 0 every evaluation is v_nc + cfg*(v_c - v_nc) (sampling.py:69-74).
 * v_trace: optional [n_eval,B,C,H,W] fp32 device buffer receiving every stage velocity, or NULL. */
FLO_API int flo_integrate(flo_unet_t* h, float* y, const float* ts, int n_ts, int method, float dt, float t_scale,
                  const int64_t* class_ids, float cfg_strength, float* v_trace, int B, void* stream);

/* Same with HOST buffers: copies x0 (host, ideally pinned) to the device, integrates, copies the
 * final latents back into x1 (host) and waits for completion.  class_ids is a HOST array here. */
FLO_API int flo_integrate_host(flo_unet_t* h, const float* x0, float* x1, const float* ts, int n_ts, int method,
                       float dt, float t_scale, const int64_t* class_ids, float cfg_strength, int B,
                       void* stream);

/* v = Unet.forward(x, time, cond) and dv[p] = J_x v · dx[p] for P tangents: exact forward mode, fp32 handles only.
 * x, v: [B,C,H,W]; dx, dv: [P,B,C,H,W] fp32 device; time, class_ids as flo_unet_forward.  Asynchronous.
 * FLO_ERR_INVALID for P outside 1..65534, B < 1 or a NULL pointer (checked first, no device needed);
 * FLO_ERR_UNSUPPORTED, before anything is allocated, for 16-bit handles, mask_cond handles and linear attention over
 * more than 256 pixels. */
FLO_API int flo_unet_jvp(flo_unet_t* h, const float* x, const float* time, const int64_t* class_ids,
                         const float* dx, int P, float* v, float* dv, int B, void* stream);

/* FLO_RK4 over ts (either direction, stage times exactly as flo_integrate forms them) with, at every stage input, the
 * Hutchinson divergence of the fixed probes [P,B,C,H,W]; div: [B] fp64 device, out = Σ_intervals dt/6·(d1+2d2+2d3+d4)
 * with d = (1/P) Σ_p probe_p · (J_x v · probe_p), summed in fp64 in an order that depends on C*H*W and P only.
 * y as flo_integrate.  Whole trajectory on the device, no host synchronisation, one graph replay per evaluation.
 * FLO_ERR_INVALID for P outside 1..65534, n_ts < 2, B < 1 or a NULL y / ts / probes / div (checked first, no device
 * needed); FLO_ERR_UNSUPPORTED as flo_unet_jvp. */
FLO_API int flo_integrate_divergence(flo_unet_t* h, float* y, const float* ts, int n_ts, float t_scale,
                         const int64_t* class_ids, const float* probes, int P, double* div, int B, void* stream);

/* Adaptive Dormand-Prince 5(4) from t0 to t1 with scipy.integrate.solve_ivp(method='RK45')'s step-size control
 * (scipy/integrate/_ivp/rk.py, common.py): select_initial_step, SAFETY 0.9, factors in [0.2, 10], exponent -1/5,
 * min_step = 10*|nextafter(t, inf) - t|, the last step clipped to land on t1, max_step = inf.
 * ONE ODE system for the whole batch: the flattened [B,C,H,W] state has one step size and the error norm is the RMS over
 * all B*C*H*W elements of err/(atol + rtol*max(|y|,|y_new|)), so a sample's trajectory depends on the rest of its batch.
 * y: [B,C,H,W] fp32 device, in = state at t0, out = state at t1.  The U-Net sees fl32(fl32(t)*t_scale) at stage time t;
 * class_ids / cfg_strength as flo_integrate; the flo_unet_set_mask state applies.  Stage times, stage inputs, the error
 * norm (fp64, bit-reproducible) and the controller run on the device; the host waits once per attempt (6 evaluations) for
 * a small status record, so the call is HOST-SYNCHRONISING like flo_integrate_host and returns when y holds the result.
 * counts (HOST, may not be NULL): nfev = 2 + 6*attempts (scipy's nfev), accepted steps, rejected attempts.
 * FLO_ERR_INVALID for rtol <= 0, atol < 0, t1 <= t0 or max_steps < 1 (checked before anything else, no device needed);
 * FLO_ERR_STEP when the step falls below min_step or more than max_steps attempts would be needed (message gives t). */
FLO_API int flo_integrate_rk45(flo_unet_t* h, float* y, double t0, double t1, double rtol, double atol, float t_scale,
                       const int64_t* class_ids, float cfg_strength, int max_steps, int counts[3], int B, void* stream);

/* flo_integrate_rk45 backwards in time: from t0 down to t1 < t0, with scipy's direction = -1 (signed steps h = -h_abs,
 * the last step clipped to land on t1, min_step = 10*|nextafter(t, -inf) - t|, the trial point of select_initial_step at
 * t0 - h0), as solve_ivp(fun, (t0, t1), ...) with t1 < t0 does.  Arguments, routes, counts and error codes are those of
 * flo_integrate_rk45, except that it requires finite t1 < t0 (FLO_ERR_INVALID otherwise, no device needed). */
FLO_API int flo_integrate_rk45_reverse(flo_unet_t* h, float* y, double t0, double t1, double rtol, double atol,
                       float t_scale, const int64_t* class_ids, float cfg_strength, int max_steps, int counts[3], int B,
                       void* stream);

/* Per-sample adaptive Dormand-Prince 5(4): every sample is its own solve_ivp(fun_i, (t0, t1), y0[i].ravel(), 'RK45') with
 * its own t, step size, accept / reject decisions and nfev; the error norm of sample i is the RMS over its C*H*W elements,
 * so a sample's result does not depend on the rest of its batch.  The batch still shares every U-Net evaluation: a sample
 * that reached t1 stays frozen (evaluated at t1, state unchanged) until the last one is done.  Arguments, routes, the
 * host-synchronising wait per attempt and the error codes are those of flo_integrate_rk45; at B = 1 the result and counts
 * equal it bit for bit.  max_steps counts attempts per sample.
 * counts (HOST, may not be NULL): [B][3] = nfev (2 + 6*attempts_i), accepted steps, rejected attempts per sample.
 * FLO_ERR_STEP when a sample's step falls below its min_step or it needs more than max_steps attempts: the message names
 * the lowest failing sample index and its t, and y is left unchanged. */
FLO_API int flo_integrate_rk45_per_sample(flo_unet_t* h, float* y, double t0, double t1, double rtol, double atol,
                       float t_scale, const int64_t* class_ids, float cfg_strength, int max_steps, int32_t* counts, int B,
                       void* stream);

/* flo_integrate_rk45_per_sample backwards in time, from t0 down to t1 < t0 (direction -1 as flo_integrate_rk45_reverse);
 * a sample that reached t1 stays frozen there.  Requires finite t1 < t0; everything else as the forward call. */
FLO_API int flo_integrate_rk45_per_sample_reverse(flo_unet_t* h, float* y, double t0, double t1, double rtol,
                       double atol, float t_scale, const int64_t* class_ids, float cfg_strength, int max_steps,
                       int32_t* counts, int B, void* stream);

/* Number of function evaluations flo_integrate performs for (method, n_ts) -- the honest count,
 * not the reference's n_steps*4 over-count (sampling.py:121). */
FLO_API int flo_integrate_nfe(int method, int n_ts);

/* ---- introspection (tests, bench) ---- */
/* Host-only (no GPU needed): text description of the op program, activation buffers with their live
 * ranges / arena offsets, and the tcgen05 tiling chosen for every convolution at batch B.
 * Returns the length of the full text (which may exceed cap), or a negative flo_status. */
FLO_API int flo_describe_plan(const flo_unet_cfg* cfg, int B, char* out, int cap);
FLO_API int flo_unet_num_ops(flo_unet_t* h);
FLO_API int flo_unet_op_name(flo_unet_t* h, int index, char* name, int name_cap);
/* Per-op metadata: kind (0 init conv, 1 conv, 2 GroupNorm pass, 3 linear attention, 4 mid attention,
 * 5 final conv + integrator epilogue, 6 fused conv-chain stage, 7 fused attention stage), ALGORITHMIC conv
 * flops (2*M*N*K over real pixels / channels, all output channels of an N-split stage; the sum over the
 * ops of one forward is SURVEY.md 8d's 66,846,720 for the BASELINE U-Net) and bytes per sample. */
FLO_API int flo_unet_op_info(flo_unet_t* h, int index, int* kind, double* flops_per_sample, double* bytes_per_sample);
/* Runs one forward at batch B op by op (no graph) `reps` times with a CUDA event around every kernel on
 * `stream` and returns the best duration of each op in milliseconds (ms_per_op: HOST array, one per op). */
FLO_API int flo_unet_profile_ops(flo_unet_t* h, int B, int reps, float* ms_per_op, void* stream);
/* Debug: SM-clock timeline (clock64) of CTA 0 of fused stage `stage` from the last forward at batch B; needs the
 * environment variable FLO_TIMELINE=1 when the batch plan is created.  out128: HOST array of 128 int64. */
FLO_API int flo_unet_read_timeline(flo_unet_t* h, int B, int stage, long long* out128);
/* Last flo_integrate_rk45, flo_integrate_rk45_per_sample or _reverse call: out = {attempts (per-sample: of the whole batch),
 * host wall ms over the attempts, device ms of the attempt graphs (CUDA events)}; wall - device is the host round trip the
 * per-attempt wait costs. */
FLO_API int flo_integrate_rk45_timing(flo_unet_t* h, double out[3]);
/* Kernel launches issued per forward pass (graph nodes) and total since creation. */
FLO_API int flo_unet_launches_per_forward(flo_unet_t* h, int B);
FLO_API int64_t flo_unet_launch_count(flo_unet_t* h);
/* Copy a named intermediate of the LAST forward at batch B to a HOST fp32 NCHW buffer (needs
 * FLO_FLAG_NO_BUFFER_REUSE).  shape receives [B,C,H,W]. */
FLO_API int flo_unet_read_activation(flo_unet_t* h, const char* name, int B, float* out, int64_t cap,
                             int64_t shape[4], void* stream);

/* ---- self tests of the sm_100a building blocks (GPU required) ---- */
/* Runs tcgen05/TMEM/TMA micro-GEMMs with the exact descriptor forms the conv kernel uses and
 * compares with a CPU result.  Returns the number of failing cases (0 = all good, <0 = error);
 * a human-readable report is written to `report` (may be NULL). */
FLO_API int flo_selftest_umma(char* report, int report_cap, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FLOCODER_B200_H */
