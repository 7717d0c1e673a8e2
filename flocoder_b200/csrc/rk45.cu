// Adaptive Dormand-Prince 5(4) on the device, step for step what scipy.integrate.solve_ivp(method='RK45') does
// (scipy/integrate/_ivp/rk.py: RK45, rk_step, RungeKutta._step_impl; common.py: select_initial_step, norm).
//
//   k_rk45_stage  before evaluation s of an attempt: xs = y + h*sum_{j<s} A[s][j] K[j]  (s = 1..5), and before the last
//                 one y_new = y + h*sum_j B[j] K[j], xs = y_new  (fp32, fixed summation order)
//   k_rk45_end    error norm of the attempt (or the norms of select_initial_step) as fp64 per-CTA partials; the last CTA
//                 adds them in a fixed order and runs the step-size controller, swaps y <- y_new and K[0] <- K[6] by index
//                 on accept, and writes the next attempt's stage table
//
// One ODE system for the whole batch: the flattened [B,C,H,W] state has one step size and the RMS norm runs over all
// B*C*H*W elements, so a sample's trajectory depends on the rest of its batch (as solve_ivp on y0.ravel()).
//
// Both directions: Rk45Ctl::direction = sign(t1 - t0) enters where scipy's OdeSolver.direction does (the signed step, the
// clip to t1, min_step, the end test, the trial point of select_initial_step).  It is an int, +1 or -1: converted to double
// it multiplies exactly, so the forward solve is bit-identical to a controller without it.
#include <math.h>

#include "umma_common.cuh"

namespace flo {

// ---- scipy's RK45 tableau and controller constants (rk.py) ----------------------------------------------------------
__constant__ float RK_A[6][5] = {
    {0.f, 0.f, 0.f, 0.f, 0.f},
    {(float)(1.0 / 5), 0.f, 0.f, 0.f, 0.f},
    {(float)(3.0 / 40), (float)(9.0 / 40), 0.f, 0.f, 0.f},
    {(float)(44.0 / 45), (float)(-56.0 / 15), (float)(32.0 / 9), 0.f, 0.f},
    {(float)(19372.0 / 6561), (float)(-25360.0 / 2187), (float)(64448.0 / 6561), (float)(-212.0 / 729), 0.f},
    {(float)(9017.0 / 3168), (float)(-355.0 / 33), (float)(46732.0 / 5247), (float)(49.0 / 176), (float)(-5103.0 / 18656)}};
__constant__ float RK_B[6] = {(float)(35.0 / 384), 0.f, (float)(500.0 / 1113), (float)(125.0 / 192), (float)(-2187.0 / 6784),
                              (float)(11.0 / 84)};
__constant__ double RK_E[7] = {-71.0 / 57600, 0.0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
__constant__ double RK_C[6] = {0.0, 1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9, 1.0};
constexpr double RK_SAFETY = 0.9, RK_MIN_FACTOR = 0.2, RK_MAX_FACTOR = 10.0;
constexpr double RK_ERR_EXP = -1.0 / (4 + 1);        // error_exponent = -1 / (error_estimator_order + 1)

// The step-size controller: one call per k_rk45_end (mode), with the RMS norms it measured.  Copies select_initial_step
// (NORM0 / NORM1) and _step_impl (STEP) line by line; the attempt it leaves prepared is (c.t, c.h) -> c.t_new.
__host__ __device__ inline void rk45_begin_attempt(Rk45Ctl& c) {
    if (c.h_abs < c.min_step) { c.status.state = RK_TOO_SMALL; return; }
    if (c.attempts >= c.max_steps) { c.status.state = RK_TOO_MANY; return; }
    double t_new = c.t + c.h_abs * c.direction;     // h = h_abs * direction; exact for direction = +-1
    if (c.direction * (t_new - c.t1) > 0) t_new = c.t1;
    c.h = t_new - c.t;
    c.h_abs = fabs(c.h);
    c.t_new = t_new;
}
__host__ __device__ inline void rk45_begin_step(Rk45Ctl& c) {
    c.min_step = 10 * fabs(nextafter(c.t, c.direction * INFINITY) - c.t);
    if (c.h_abs > c.max_step) c.h_abs = c.max_step;
    else if (c.h_abs < c.min_step) c.h_abs = c.min_step;
    c.step_rejected = 0;
    rk45_begin_attempt(c);
}
__host__ __device__ inline void rk45_control(Rk45Ctl& c, int mode, double norm0, double norm1) {
    if (mode == RK_END_NORM0) {                     // d0 = norm(y0/scale), d1 = norm(f0/scale)
        const double d0 = norm0, d1 = norm1;
        double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        c.h0 = fmin(h0, c.interval);
        c.d1 = d1;
        c.status.nfev = 1;
    } else if (mode == RK_END_NORM1) {              // d2 = norm((f1 - f0)/scale) / h0
        const double d1 = c.d1, d2 = norm0 / c.h0;
        double h1;
        if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, c.h0 * 1e-3);
        else h1 = pow(0.01 / fmax(d1, d2), 1.0 / (4 + 1));
        c.h_abs = fmin(fmin(100 * c.h0, h1), fmin(c.interval, c.max_step));
        c.status.nfev = 2;
        rk45_begin_step(c);
    } else {
        const double error_norm = norm0;
        c.attempts += 1;
        c.status.nfev += 6;
        if (error_norm < 1) {
            double factor = error_norm == 0 ? RK_MAX_FACTOR : fmin(RK_MAX_FACTOR, RK_SAFETY * pow(error_norm, RK_ERR_EXP));
            if (c.step_rejected) factor = fmin(1.0, factor);
            c.h_abs *= factor;
            c.t = c.t_new;
            c.status.y_idx ^= 1;                    // y <- y_new
            c.k0 = 6 - c.k0;                        // K[0] <- K[6] (FSAL)
            c.status.accepted += 1;
            if (c.direction * (c.t - c.t1) >= 0) c.status.state = RK_DONE;
            else rk45_begin_step(c);
        } else {
            // python's max(MIN_FACTOR, nan) is MIN_FACTOR, as fmax
            c.h_abs *= fmax(RK_MIN_FACTOR, RK_SAFETY * pow(error_norm, RK_ERR_EXP));
            c.step_rejected = 1;
            c.status.rejected += 1;
            rk45_begin_attempt(c);
        }
    }
    c.status.t = c.t;
    c.status.h_abs = c.h_abs;
}

// physical slot of K[j]: K[0] and K[6] trade places on every accepted step
__device__ __forceinline__ int rk_slot(int k0, int j) { return j == 0 ? k0 : (j == 6 ? 6 - k0 : j); }

// stage-table entries of evaluation e (0-based) at ODE time t, velocity to K slot `slot`
__device__ void rk45_write_eval(Stage* stages, const Rk45Ctl& c, int e, double t, int slot) {
    Stage s{};
    s.t_scaled = __fmul_rn((float)t, c.t_scale);    // fl32(fl32(t) * 999): torch.ones(B) * t * 999 in fp32
    s.film_row = 0;
    if (c.two_pass) {
        Stage a = s;
        a.kind = ST_CFG_COND; a.flags = 0; a.eval_idx = -1;
        stages[2 * e] = a;
        s.kind = ST_STORE; s.flags = SF_CFG_COMBINE; s.eval_idx = slot;
        stages[2 * e + 1] = s;
    } else {
        s.kind = ST_STORE; s.flags = c.flags; s.eval_idx = slot;
        stages[e] = s;
    }
}
__device__ void rk45_write_attempt(Stage* stages, const Rk45Ctl& c) {
    if (c.status.state != RK_RUNNING) return;
    for (int e = 1; e <= 5; ++e) rk45_write_eval(stages, c, e - 1, c.t + RK_C[e] * c.h, rk_slot(c.k0, e));
    rk45_write_eval(stages, c, 5, c.t + c.h, rk_slot(c.k0, 6));
}

__global__ void k_rk45_setup(Rk45Ctl* dst, Rk45Ctl value, Ctrl* ctrl) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        *dst = value;
        rk45_write_eval(const_cast<Stage*>(ctrl->stages), value, 0, value.t, value.k0);     // f0 = fun(t0, y0)
        ctrl->step = 0;
    }
}
cudaError_t launch_rk45_setup(Rk45Ctl* dst, const Rk45Ctl& value, Ctrl* ctrl, cudaStream_t s) {
    k_rk45_setup<<<1, 32, 0, s>>>(dst, value, ctrl);
    return cudaGetLastError();
}

// ---- stage inputs ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_rk45_stage(Rk45Params p, int stage) {
    griddep_wait();
    const Rk45Ctl& c = *p.rc;
    const int yi = c.status.y_idx, k0 = c.k0;
    const float* y = p.ybuf + (size_t)yi * p.n;
    float* ynew = p.ybuf + (size_t)(yi ^ 1) * p.n;
    const float h = stage < 0 ? (float)(c.h0 * c.direction) : (float)c.h;       // c.h is signed already
    const float* ks[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) ks[j] = p.k + (size_t)rk_slot(k0, j) * p.n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += gridDim.x * blockDim.x) {
        const float yv = y[i];
        float x;
        if (stage == 0) {
            x = yv;
        } else if (stage < 0) {                       // select_initial_step: y1 = y0 + h0 * direction * f0
            x = __fadd_rn(yv, __fmul_rn(h, ks[0][i]));
        } else {
            const float* a = stage < 6 ? RK_A[stage] : RK_B;
            float acc = __fmul_rn(a[0], ks[0][i]);
            for (int j = 1; j < stage; ++j) acc = __fadd_rn(acc, __fmul_rn(a[j], ks[j][i]));
            x = __fadd_rn(yv, __fmul_rn(acc, h));   // y + dot(K[:s].T, a) * h
            if (stage == 6) ynew[i] = x;
        }
        p.xs[i] = x;
        if (p.xs2) p.xs2[i] = x;
    }
}
cudaError_t launch_rk45_stage(const Rk45Params& p, int stage, cudaStream_t s) {
    const int grid = std::min((p.n + 255) / 256, 148 * 8);
    k_rk45_stage<<<grid, 256, 0, s>>>(p, stage);
    return cudaGetLastError();
}

// ---- norms + controller ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double block_sum_f64(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    return t;                                          // valid in thread 0
}

__global__ void __launch_bounds__(256) k_rk45_end(Rk45Params p, int mode) {
    __shared__ double red[8];
    __shared__ int last;
    griddep_wait();
    Rk45Ctl* rc = p.rc;
    const int yi = rc->status.y_idx, k0 = rc->k0;
    const double rtol = rc->rtol, atol = rc->atol, h = rc->h;
    const float* y = p.ybuf + (size_t)yi * p.n;
    const float* yn = p.ybuf + (size_t)(yi ^ 1) * p.n;
    double s0 = 0.0, s1 = 0.0;
    const int per = (p.n + gridDim.x - 1) / gridDim.x;
    const int i0 = blockIdx.x * per, i1 = min(p.n, i0 + per);
    if (mode == RK_END_STEP) {
        const float* ks[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) ks[j] = p.k + (size_t)rk_slot(k0, j) * p.n;
        for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
            double e = 0.0;
#pragma unroll
            for (int j = 0; j < 7; ++j) e = fma((double)ks[j][i], RK_E[j], e);
            const double err = e * h;                                      // dot(K.T, E) * h
            const double scale = atol + fmax(fabs((double)y[i]), fabs((double)yn[i])) * rtol;
            const double q = err / scale;
            s0 = fma(q, q, s0);
        }
    } else {
        const float* f0 = p.k + (size_t)k0 * p.n;
        const float* f1 = p.k + (size_t)1 * p.n;                         // the trial evaluation's slot
        for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
            const double yv = (double)y[i];
            const double scale = atol + fabs(yv) * rtol;
            if (mode == RK_END_NORM0) {
                const double a = yv / scale, b = (double)f0[i] / scale;
                s0 = fma(a, a, s0); s1 = fma(b, b, s1);
            } else {
                const double d = ((double)f1[i] - (double)f0[i]) / scale;
                s0 = fma(d, d, s0);
            }
        }
    }
    s0 = block_sum_f64(s0, red);
    s1 = block_sum_f64(s1, red);
    if (threadIdx.x == 0) {
        p.part[2 * blockIdx.x] = s0;
        p.part[2 * blockIdx.x + 1] = s1;
        __threadfence();
        last = atomicAdd(&rc->arrive, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    // the last CTA to arrive: add the partials in CTA order (bit-reproducible), then the controller
    __threadfence();
    double a0 = 0.0, a1 = 0.0;
    if (threadIdx.x == 0) {
        for (int b = 0; b < (int)gridDim.x; ++b) { a0 += __ldcg(p.part + 2 * b); a1 += __ldcg(p.part + 2 * b + 1); }
        Rk45Ctl c = *rc;
        const double rn = sqrt((double)p.n);
        rk45_control(c, mode, sqrt(a0) / rn, sqrt(a1) / rn);           // norm(x) = ||x||_2 / sqrt(x.size)
        c.arrive = 0;
        Stage* stages = const_cast<Stage*>(p.ctrl->stages);   // the stage table is written by this kernel and setup only
        if (mode == RK_END_NORM0) {
            if (c.status.state == RK_RUNNING)             // f1 = fun(t0 + h0 * direction, y1)
                rk45_write_eval(stages, c, 0, c.t + c.h0 * c.direction, 1);
        } else {
            rk45_write_attempt(stages, c);
        }
        *rc = c;
        p.ctrl->step = 0;
        __threadfence();
    }
}
cudaError_t launch_rk45_end(const Rk45Params& p, int mode, cudaStream_t s) {
    k_rk45_end<<<rk45_end_grid(p.n), 256, 0, s>>>(p, mode);
    return cudaGetLastError();
}

// ---- per-sample RK45: B controllers, each sample its own solve_ivp ------------------------------------------------------
//
//   k_rk45ps_setup  every controller <- the initial state; the stage entry of f0 (slot 0)
//   k_rk45ps_stage  k_rk45_stage's arithmetic with the sample's own h (and h0), plus the sample's stage time
//                   fl32(fl32(t + c_s*h) * t_scale) into tbuf for k_temb; a finished sample is frozen: xs = y at t1
//                   (in either direction)
//   k_rk45ps_end    one CTA per sample: k_rk45_end's norm over that sample's C*H*W elements, summed in the batched kernel's
//                   partition (so B = 1 is bit-identical to the batched mode), the controller, and on accept the copies
//                   K[6] -> K[0] and y_new -> y; the last CTA to arrive counts running / done / failed samples
//
// The stage table is the same for every attempt (only times and step sizes are per sample): evaluation e writes K slot e.
__device__ void rk45ps_write_table(const Rk45PsParams& p, int mode) {
    Stage* stages = const_cast<Stage*>(p.ctrl->stages);
    Rk45Ctl c{};
    c.two_pass = p.two_pass; c.flags = p.flags;                                       // t_scaled is unused: k_temb reads tbuf
    if (mode == RK_END_NORM0) rk45_write_eval(stages, c, 0, 0.0, 1);                   // f1 = fun(t0 + h0 * direction, y1)
    else for (int e = 1; e <= 6; ++e) rk45_write_eval(stages, c, e - 1, 0.0, e);
}

__global__ void k_rk45ps_setup(Rk45PsParams p, Rk45Ctl value) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < p.B) p.rc[b] = value;
    if (b == 0) {
        Rk45Ctl c{};
        c.two_pass = p.two_pass; c.flags = p.flags;
        rk45_write_eval(const_cast<Stage*>(p.ctrl->stages), c, 0, 0.0, 0);          // f0 = fun(t0, y0)
        p.ctrl->step = 0;
        Rk45PsStatus s{};
        s.running = p.B; s.first_failed = -1;
        *p.st = s;
    }
}
cudaError_t launch_rk45ps_setup(const Rk45PsParams& p, const Rk45Ctl& value, cudaStream_t s) {
    k_rk45ps_setup<<<(p.B + 255) / 256, 256, 0, s>>>(p, value);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_rk45ps_stage(Rk45PsParams p, int stage) {
    griddep_wait();
    const int gi = blockIdx.x * blockDim.x + threadIdx.x;
    if (gi < p.B) {                                   // the sample's stage time, as rk45_write_eval forms it
        const Rk45Ctl& c = p.rc[gi];
        double t;
        if (c.status.state != RK_RUNNING) t = c.t1;
        else if (stage == 0) t = c.t;
        else if (stage < 0) t = c.t + c.h0 * c.direction;
        else if (stage < 6) t = c.t + RK_C[stage] * c.h;
        else t = c.t + c.h;
        const float ts = __fmul_rn((float)t, c.t_scale);
        p.tbuf[gi] = ts;
        if (p.xs2) p.tbuf[p.B + gi] = ts;             // the unconditional half of the 2B route
    }
    const float* y = p.ybuf;
    float* ynew = p.ybuf + p.n;
    const float* ks[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) ks[j] = p.k + (size_t)j * p.n;
    for (int i = gi; i < p.n; i += gridDim.x * blockDim.x) {
        const Rk45Ctl& c = p.rc[i / p.per];
        const float yv = y[i];
        float x;
        if (stage == 0 || c.status.state != RK_RUNNING) {
            x = yv;
        } else if (stage < 0) {                       // select_initial_step: y1 = y0 + h0 * direction * f0
            x = __fadd_rn(yv, __fmul_rn((float)(c.h0 * c.direction), ks[0][i]));
        } else {
            const float h = (float)c.h;
            const float* a = stage < 6 ? RK_A[stage] : RK_B;
            float acc = __fmul_rn(a[0], ks[0][i]);
            for (int j = 1; j < stage; ++j) acc = __fadd_rn(acc, __fmul_rn(a[j], ks[j][i]));
            x = __fadd_rn(yv, __fmul_rn(acc, h));   // y + dot(K[:s].T, a) * h
            if (stage == 6) ynew[i] = x;
        }
        p.xs[i] = x;
        if (p.xs2) p.xs2[i] = x;
    }
}
cudaError_t launch_rk45ps_stage(const Rk45PsParams& p, int stage, cudaStream_t s) {
    const int grid = std::max(std::min((p.n + 255) / 256, 148 * 8), (p.B + 255) / 256);
    k_rk45ps_stage<<<grid, 256, 0, s>>>(p, stage);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) k_rk45ps_end(Rk45PsParams p, int mode) {
    __shared__ double red[8];
    __shared__ int last, accepted, cnt[3], first;
    griddep_wait();
    const int b = blockIdx.x;
    Rk45Ctl* rc = p.rc + b;
    const size_t off = (size_t)b * p.per;
    if (rc->status.state == RK_RUNNING) {
        const double rtol = rc->rtol, atol = rc->atol, h = rc->h;
        const float* y = p.ybuf + off;
        const float* yn = p.ybuf + p.n + off;
        const float* ks[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) ks[j] = p.k + (size_t)j * p.n + off;
        // k_rk45_end's loops over the chunks its grid would give a lone sample, partials added in chunk order
        const int G = rk45_end_grid(p.per), per = (p.per + G - 1) / G;
        double a0 = 0.0, a1 = 0.0;
        for (int g = 0; g < G; ++g) {
            double s0 = 0.0, s1 = 0.0;
            const int i0 = g * per, i1 = min(p.per, i0 + per);
            if (mode == RK_END_STEP) {
                for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
                    double e = 0.0;
#pragma unroll
                    for (int j = 0; j < 7; ++j) e = fma((double)ks[j][i], RK_E[j], e);
                    const double err = e * h;                                      // dot(K.T, E) * h
                    const double scale = atol + fmax(fabs((double)y[i]), fabs((double)yn[i])) * rtol;
                    const double q = err / scale;
                    s0 = fma(q, q, s0);
                }
            } else {
                for (int i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
                    const double yv = (double)y[i];
                    const double scale = atol + fabs(yv) * rtol;
                    if (mode == RK_END_NORM0) {
                        const double a = yv / scale, f = (double)ks[0][i] / scale;
                        s0 = fma(a, a, s0); s1 = fma(f, f, s1);
                    } else {
                        const double d = ((double)ks[1][i] - (double)ks[0][i]) / scale;
                        s0 = fma(d, d, s0);
                    }
                }
            }
            s0 = block_sum_f64(s0, red);
            s1 = block_sum_f64(s1, red);
            if (threadIdx.x == 0) { a0 += s0; a1 += s1; }
        }
        if (threadIdx.x == 0) {
            // the controller works on the record in place: a register copy of all of it spills under the 64-register cap
            Rk45Ctl& c = *rc;
            const int acc0 = c.status.accepted;
            const double rn = sqrt((double)p.per);
            rk45_control(c, mode, sqrt(a0) / rn, sqrt(a1) / rn);           // norm(x) = ||x||_2 / sqrt(x.size)
            accepted = c.status.accepted != acc0;
            c.status.y_idx = 0; c.k0 = 0;             // fixed layout: the accepted step is copied below
        }
        __syncthreads();
        if (accepted) {
            float* yw = p.ybuf + off;
            float* k0 = p.k + off;
            const float* k6 = p.k + (size_t)6 * p.n + off;
            for (int i = threadIdx.x; i < p.per; i += blockDim.x) { yw[i] = yn[i]; k0[i] = k6[i]; }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(&p.st->arrive, 1u) == gridDim.x - 1;
        cnt[0] = cnt[1] = cnt[2] = 0;
        first = p.B;
    }
    __syncthreads();
    if (!last) return;
    // the last CTA to arrive: count the samples' states, publish the status record, reset the stage table position
    __threadfence();
    for (int i = threadIdx.x; i < p.B; i += blockDim.x) {
        const int s = __ldcg(&p.rc[i].status.state);
        if (s == RK_RUNNING) atomicAdd(&cnt[0], 1);
        else if (s == RK_DONE) atomicAdd(&cnt[1], 1);
        else { atomicAdd(&cnt[2], 1); atomicMin(&first, i); }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        Rk45PsStatus s{};
        s.running = cnt[0]; s.done = cnt[1]; s.failed = cnt[2]; s.first_failed = cnt[2] ? first : -1; s.arrive = 0;
        *p.st = s;
        if (mode != RK_END_STEP) rk45ps_write_table(p, mode);
        p.ctrl->step = 0;
        __threadfence();
    }
}
cudaError_t launch_rk45ps_end(const Rk45PsParams& p, int mode, cudaStream_t s) {
    k_rk45ps_end<<<p.B, 256, 0, s>>>(p, mode);
    return cudaGetLastError();
}

}  // namespace flo
